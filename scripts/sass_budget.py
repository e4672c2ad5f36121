"""Instruction budget of the seed scan, read from the compiler's output (CPU only, no GPU needed).

Compiles mimeo_b200/csrc/seed.cu for sm_100a with the library's flags, and prints one JSON document:
  - ptxas registers, spill bytes and shared memory of every seed_scan_kernel instance;
  - the opcode histogram of seed_scan_kernel<4, 0x148> (the instance the scan launches), split into ALU-class, FMA-class, LSU
    and other instructions;
  - instructions per first-stage x-drop chunk and per batch set-up, measured between landmarks of the batch path: the set-up
    runs from the first of the span loads (LDG.E.64) to the first table lookup (LDS with the table base in a uniform register);
    the longest run of lookups with no global load in between is right window 0 and left window 0 of a batch, and the chunk
    count divides the instructions from its first lookup to the next global load (the loads of left window 1, so the ends of
    both windows are included) by the number of lookups in the run.
The counts are static: each instruction of the unrolled code is counted once.

  python scripts/sass_budget.py [--src path/to/seed.cu] [--out FILE]
"""
import argparse
import collections
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mimeo_b200.build import FLAGS, NVCC  # noqa: E402

KERNEL = '_ZN3mb216seed_scan_kernelILi4ELj328EEEvNS_10GenomeViewES1_PKjS3_jjiiijPmjPy'   # seed_scan_kernel<4, 0x148>
CUOBJDUMP = os.path.join(os.path.dirname(NVCC), 'cuobjdump')
# integer/logic ops of the ALU pipe, multiply-adds of the FMA pipe, memory and shuffle ops of the LSU
ALU = {'LOP3', 'SHF', 'ISETP', 'SEL', 'VIMNMX', 'IMNMX', 'IADD3', 'PRMT', 'LEA', 'FLO', 'POPC', 'BREV', 'PLOP3', 'P2R', 'R2P',
       'MOV', 'IABS', 'BMSK', 'SGXT', 'LOP', 'SHL', 'SHR', 'IADD', 'ICMP', 'FSEL', 'FSETP', 'FMNMX'}
FMA = {'IMAD', 'IMUL', 'FFMA', 'FADD', 'FMUL', 'IDP', 'IDP4A'}
LSU = {'LDS', 'STS', 'LDG', 'STG', 'LD', 'ST', 'LDL', 'STL', 'ATOM', 'ATOMS', 'ATOMG', 'RED', 'REDG', 'SHFL', 'LDSM', 'LDC'}
INSN = re.compile(r'/\*[0-9a-f]{4,}\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)([^;]*);')


def compile_seed(src, tmp):
    obj = os.path.join(tmp, 'seed.o')
    flags = [f for f in FLAGS]
    flags += ['-I', os.path.dirname(os.path.abspath(src))]
    out = subprocess.run([NVCC] + flags + ['-Xptxas', '-v', '-c', src, '-o', obj], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         text=True, check=True).stdout
    return obj, out


def ptxas_info(log):
    info, name = {}, None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            name = m.group(1)
            continue
        if name is None or 'seed_scan_kernel' not in name:
            continue
        m = re.search(r'(\d+) bytes spill stores, (\d+) bytes spill loads', line)
        if m:
            info.setdefault(name, {}).update(spill_stores=int(m.group(1)), spill_loads=int(m.group(2)))
        m = re.search(r'Used (\d+) registers.*?(\d+) bytes smem', line)
        if m:
            info.setdefault(name, {}).update(registers=int(m.group(1)), smem_bytes=int(m.group(2)))
    return info


def sass(obj):
    out = subprocess.run([CUOBJDUMP, '-sass', '-fun', KERNEL, obj], stdout=subprocess.PIPE, text=True, check=True).stdout
    return [(m.group(2), m.group(3).strip()) for m in INSN.finditer(out)]


def klass(op):
    base = op.split('.')[0]
    if base in FMA:
        return 'fma'
    if base in ALU:
        return 'alu'
    if base in LSU:
        return 'lsu'
    return 'other'


def landmarks(ins):
    is_lookup = [op == 'LDS' and '+UR' in args for op, args in ins]
    is_span = [op == 'LDG.E.64' for op, _ in ins]
    # runs of table lookups with no global load between them
    runs, cur = [], []
    for i, (op, _) in enumerate(ins):
        if op.startswith('LDG'):
            if cur:
                runs.append(cur)
            cur = []
        elif is_lookup[i]:
            cur.append(i)
    if cur:
        runs.append(cur)
    run = max(runs, key=len)
    first, last = run[0], run[-1]
    # the span loads of the batch: the LDG.E.64 between the previous table lookup and the run
    prev = max([i for i in range(first) if is_lookup[i]], default=-1)
    s0 = min(i for i in range(prev + 1, first) if is_span[i])
    end = next(i for i in range(last, len(ins)) if ins[i][0].startswith('LDG'))
    hist = collections.Counter(klass(op) for op, _ in ins[first:end])
    return {
        'lookups_in_run': len(run),
        'instructions_per_chunk': round((end - first) / len(run), 2),
        'per_chunk_by_class': {k: round(v / len(run), 2) for k, v in sorted(hist.items())},
        'batch_setup_instructions': first - s0,
        'batch_setup_by_class': dict(sorted(collections.Counter(klass(op) for op, _ in ins[s0:first]).items())),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--src', default=os.path.join(ROOT, 'mimeo_b200', 'csrc', 'seed.cu'))
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        obj, log = compile_seed(a.src, tmp)
        ins = sass(obj)
    ops = collections.Counter(op.split('.')[0] for op, _ in ins)
    by_class = collections.Counter()
    for op, n in ops.items():
        by_class[klass(op)] += n
    doc = {
        'kernel': 'seed_scan_kernel<4, 0x148> (sm_100a)',
        'ptxas': {('seed_scan_kernel<4, 0x148>' if n == KERNEL else 'seed_scan_kernel<3, 0x148>' if 'ILi3E' in n else n): v
                  for n, v in ptxas_info(log).items()},
        'instructions': len(ins),
        'by_class': dict(sorted(by_class.items())),
        'opcodes': dict(sorted(ops.items(), key=lambda kv: -kv[1])),
        'batch_path': landmarks(ins),
        'classes': {'alu': sorted(ALU), 'fma': sorted(FMA), 'lsu': sorted(LSU)},
    }
    text = json.dumps(doc, indent=1)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(text + '\n')
    print(text)


if __name__ == '__main__':
    main()
