"""ctypes binding of libmimeo_b200.so (C ABI declared in include/mimeo_b200.h).

The product path must fail loudly when the CUDA extension is missing: `lib()` raises if the shared
library is not built, and `init()` raises if no B200-class device is present. Nothing here falls
back to a CPU implementation.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libmimeo_b200.so')

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_u32p = C.POINTER(C.c_uint32)
c_u64p = C.POINTER(C.c_uint64)


class AlignParams(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ('hspthresh', 'xdrop', 'ydrop', 'gap_open', 'gap_extend', 'gappedthresh',
                                         'entropy', 'chain', 'gapped', 'transition')]


class Hsps(C.Structure):
    _fields_ = [('tile', c_u32p), ('s1', c_i32p), ('s2', c_i32p), ('len', c_i32p), ('score', c_i32p), ('n', C.c_uint64)]


class SeedSurvivors(C.Structure):
    _fields_ = [('t_pos', c_u32p), ('q_pos', c_u32p), ('n', C.c_uint64), ('t_off', c_u32p), ('q_off', c_u32p),
                ('t_nscaf', C.c_int32), ('q_nscaf', C.c_int32), ('counters', C.c_uint64 * 4)]


class Hits(C.Structure):
    _fields_ = [(n, c_i32p) for n in ('t_id', 'q_id', 'strand', 'start1', 'end1', 'start2', 'end2', 'score', 'nmatch', 'ncols')] + \
               [('n', C.c_uint64), ('stats', C.c_uint64 * 16)]


class TabHits(C.Structure):
    _fields_ = [('chrom', c_i32p), ('start', c_i64p), ('end', c_i64p), ('n', C.c_uint64), ('names', C.POINTER(C.c_char_p)),
                ('nnames', C.c_int32)]


class Fasta(C.Structure):
    _fields_ = [('n', C.c_int32), ('ids', C.POINTER(C.c_char_p)), ('headers', C.POINTER(C.c_char_p)), ('off', c_u64p),
                ('seq', C.POINTER(C.c_uint8))]


class TabText(C.Structure):
    _fields_ = [('text', C.POINTER(C.c_char)), ('nbytes', C.c_uint64), ('t_id', c_i32p), ('q_id', c_i32p), ('off', c_u64p),
                ('nrows', c_u32p), ('nblocks', C.c_uint64)]


class Text(C.Structure):
    _fields_ = [('text', C.POINTER(C.c_char)), ('nbytes', C.c_uint64), ('nrows', C.c_uint64)]


class TandemParams(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ('match', 'mismatch', 'delta', 'minscore', 'maxperiod')]


class TandemRuns(C.Structure):
    _fields_ = [('off', c_u64p), ('start', c_i64p), ('end', c_i64p), ('n', C.c_uint64)]


class TandemRepeats(C.Structure):
    _fields_ = [('period', c_i32p), ('score', c_i64p), ('matches', c_u64p), ('count', c_u64p), ('cons_off', c_u64p),
                ('consensus', C.c_void_p), ('n', C.c_uint64)]


class Segments(C.Structure):
    _fields_ = [('chrom', c_i32p), ('start', c_i32p), ('end', c_i32p), ('n', C.c_uint64), ('on_device', C.c_int)]


# every symbol include/mimeo_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    'mb2_init': (C.c_int, [C.c_int]),
    'mb2_shutdown': (None, []),
    'mb2_last_error': (C.c_char_p, []),
    'mb2_stream': (C.c_void_p, []),
    'mb2_launch_count': (C.c_ulonglong, []),
    'mb2_sm_count': (C.c_int, []),
    'mb2_sync': (C.c_int, []),
    'mb2_prof_enable': (C.c_int, [C.c_int]),
    'mb2_prof_get': (C.c_int, [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_ulonglong)]),
    'mb2_prof_reset': (C.c_int, []),
    'mb2_coverage_segments': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, C.c_int,
                                        C.c_int, C.POINTER(Segments)]),
    'mb2_coverage_segments_dev': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int,
                                            C.c_int, C.c_int, C.POINTER(Segments)]),
    'mb2_coverage_segments_into': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    'mb2_free_segments': (None, [C.POINTER(Segments)]),
    'mb2_genome_create': (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    'mb2_genome_revcomp': (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    'mb2_genome_both_strands': (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    'mb2_genome_free': (None, [C.c_void_p]),
    'mb2_genome_decode': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    'mb2_test_genome_nibbles': (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    'mb2_default_align_params': (None, [C.POINTER(AlignParams)]),
    'mb2_free_hsps': (None, [C.POINTER(Hsps)]),
    'mb2_test_hsps': (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(AlignParams), C.POINTER(Hsps), C.c_void_p]),
    'mb2_test_seed_scan': (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(AlignParams), C.c_uint64, C.POINTER(SeedSurvivors)]),
    'mb2_free_seed_survivors': (None, [C.POINTER(SeedSurvivors)]),
    'mb2_align': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(AlignParams), C.c_int, C.c_void_p, C.POINTER(Hits)]),
    'mb2_free_hits': (None, [C.POINTER(Hits)]),
    'mb2_align_dev': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(AlignParams), C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    'mb2_hits_dev_free': (None, [C.c_void_p]),
    'mb2_hits_dev_count': (C.c_uint64, [C.c_void_p]),
    'mb2_filter_sort': (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_int, C.POINTER(C.c_uint64)]),
    'mb2_hits_dev_coverage': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(Segments)]),
    'mb2_hits_dev_upload': (C.c_int, [C.POINTER(Hits), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    'mb2_hits_dev_download': (C.c_int, [C.c_void_p, C.POINTER(Hits)]),
    'mb2_tab_project': (C.c_int, [C.c_char_p, C.c_int, C.POINTER(TabHits)]),
    'mb2_free_tab_hits': (None, [C.POINTER(TabHits)]),
    'mb2_fasta_read': (C.c_int, [C.c_char_p, C.c_int, C.POINTER(Fasta)]),
    'mb2_free_fasta': (None, [C.POINTER(Fasta)]),
    'mb2_fasta_split': (C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint64)]),
    'mb2_format_tab': (C.c_int, [C.c_void_p] * 10 + [C.c_uint64, C.POINTER(C.c_char_p), C.c_int, C.POINTER(C.c_char_p), C.c_int,
                                 C.c_double, C.c_double, C.POINTER(TabText)]),
    'mb2_free_tab_text': (None, [C.POINTER(TabText)]),
    'mb2_map_gff': (C.c_int, [C.c_char_p, C.c_char_p, C.c_double, C.c_double, C.c_char_p, C.c_int, C.POINTER(Text)]),
    'mb2_format_gff': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_char_p), C.c_int, C.c_char_p, C.c_char_p,
                                 C.c_char_p, C.c_uint64, C.c_int, C.POINTER(Text)]),
    'mb2_free_text': (None, [C.POINTER(Text)]),
    'mb2_default_tandem_params': (None, [C.POINTER(TandemParams)]),
    'mb2_tandem_mask': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(TandemParams), C.c_void_p]),
    'mb2_tandem_mask_runs': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(TandemParams), C.c_void_p,
                                       C.POINTER(TandemRuns)]),
    'mb2_test_tandem_mask': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(TandemParams), C.c_uint64,
                                       C.c_void_p, C.POINTER(TandemRuns)]),
    'mb2_free_tandem_runs': (None, [C.POINTER(TandemRuns)]),
    'mb2_tandem_report': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(TandemParams), C.c_void_p,
                                    C.POINTER(TandemRuns), C.POINTER(TandemRepeats)]),
    'mb2_free_tandem_report': (None, [C.POINTER(TandemRepeats)]),
    'mb2_test_sort_u32': (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int]),
    'mb2_test_sort_u64': (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int]),
    'mb2_test_sort_u32_pair': (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int]),
    'mb2_test_scan_u32': (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p]),
}

_lib = None
_inited_device = None


class Mb2Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f'libmimeo_b200 error {code}: {msg}')
        self.code = code


def lib():
    """Load the shared library (no GPU needed for loading)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f'{LIB_PATH} is not built; run `python -m mimeo_b200.build` (there is no CPU fallback)')
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


ERR_CAPACITY = -6
ERR_DUPLICATE_ID = -7


def check(rc):
    if rc != 0:
        raise Mb2Error(rc, lib().mb2_last_error().decode('utf-8', 'replace'))


def init(device=None):
    """Bind this process to one GPU (LOCAL_RANK under torchrun, else 0). Raises without a device."""
    global _inited_device
    if device is None:
        device = int(os.environ.get('LOCAL_RANK', '0'))
    if _inited_device != device:
        check(lib().mb2_init(device))
        _inited_device = device
    return device


def launch_count():
    return int(lib().mb2_launch_count())


def stream_handle():
    return lib().mb2_stream()


def sync():
    check(lib().mb2_sync())


def prof_enable(on=True):
    check(lib().mb2_prof_enable(1 if on else 0))


def prof_reset():
    check(lib().mb2_prof_reset())


def prof_get(tag):
    """(total milliseconds, number of timed regions) accumulated for a kernel tag since the last reset."""
    ms, cnt = C.c_double(0), C.c_ulonglong(0)
    check(lib().mb2_prof_get(tag.encode(), C.byref(ms), C.byref(cnt)))
    return ms.value, int(cnt.value)
