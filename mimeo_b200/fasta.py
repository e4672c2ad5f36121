"""Minimal FASTA I/O for the hot path (the reference uses Biopython's SeqIO, utils.py:301-309, 530-546)."""
from __future__ import annotations

import os
from typing import Iterator, List, Tuple

import numpy as np


class _FastaBlock:
    """Owns one mb2_fasta result; the numpy views handed out keep it alive and it frees the library memory when the last
    of them is gone (no copy of the sequence block)."""

    def __init__(self, f):
        self.f = f

    def __del__(self):
        import ctypes as C
        from . import _lib
        try:
            _lib.lib().mb2_free_fasta(C.byref(self.f))
        except Exception:
            pass


def read_fasta(path: str, nthreads: int = 0) -> List[Tuple[str, str, np.ndarray]]:
    """[(id, full header text without '>', sequence as uint8 ASCII array)] for every record of a FASTA file.
    Parsed natively (libmimeo_b200 `mb2_fasta_read`: mmap, parallel count + compact passes): a record starts at a '>' in
    column one, its id is the first word of that line, its sequence is the body without line breaks and blanks."""
    import ctypes as C
    from . import _lib
    f = _lib.Fasta()
    _lib.check(_lib.lib().mb2_fasta_read(os.fsencode(path), int(nthreads), C.byref(f)))
    owner = _FastaBlock(f)
    out: List[Tuple[str, str, np.ndarray]] = []
    n = int(f.n)
    if n:
        off = np.ctypeslib.as_array(f.off, shape=(n + 1,)).astype(np.int64)
        total = int(off[n])
        carr = (C.c_uint8 * max(total, 1)).from_address(C.addressof(f.seq.contents))
        carr._owner = owner                                  # the views' base chain ends here
        block = np.frombuffer(carr, dtype=np.uint8, count=total)
        for r in range(n):
            out.append((f.ids[r].decode('utf-8', 'replace'), f.headers[r].decode('utf-8', 'replace'),
                        block[int(off[r]):int(off[r + 1])]))
    return out


def write_fasta_record(path, header: str, seq: np.ndarray, width: int = 60) -> None:
    """One record, sequence wrapped at `width` columns (SeqIO.write's layout). `path` is a file name, which then holds
    this record alone, or a binary file open for writing, to which the record is appended (many records, one file)."""
    if not hasattr(path, 'write'):
        with open(path, 'wb') as f:
            write_fasta_record(f, header, seq, width)
        return
    f = path
    n = len(seq)
    f.write(b'>' + header.encode() + b'\n')
    if n:
        full = n // width
        if full:
            block = np.empty((full, width + 1), dtype=np.uint8)
            block[:, :width] = seq[:full * width].reshape(full, width)
            block[:, width] = 10
            f.write(block.tobytes())
        if n % width:
            f.write(seq[full * width:].tobytes() + b'\n')


def dir_records(seqdir: str) -> Iterator[Tuple[str, str, np.ndarray, str]]:
    """Every record of every file in a directory, files in sorted order: (id, header, seq, path)."""
    for fn in sorted(os.listdir(seqdir)):
        p = os.path.join(seqdir, fn)
        if os.path.isfile(p):
            for rid, header, seq in read_fasta(p):
                yield rid, header, seq, p
