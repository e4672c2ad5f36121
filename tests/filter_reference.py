"""The reference statement of `mimeo filter` (DESIGN §2) that the tests compare the product against: its own FASTA parser and
60-column writer, written independently of mimeo_b200.fasta, and the mask of the C oracle (oracle/tandem_oracle.c)."""
from __future__ import annotations

from typing import Dict, List, Tuple

from oracle import tandem_oracle as to


def fasta_records(text: str) -> List[Tuple[str, str]]:
    """(header, sequence) of every record: a record starts at a '>' that begins a line; its header is the rest of that line
    without trailing '\\r'; its sequence is every following line up to the next record, without '\\n', '\\r' and ' '."""
    recs: List[Tuple[str, List[str]]] = []
    for line in text.split('\n'):
        if line.startswith('>'):
            recs.append((line[1:].rstrip('\r'), []))
        elif recs:
            recs[-1][1].append(line.replace('\r', '').replace(' ', ''))
    return [(h, ''.join(body)) for h, body in recs]


def fasta_text(header: str, seq: str) -> str:
    return '>' + header + '\n' + ''.join(seq[i:i + 60] + '\n' for i in range(0, len(seq), 60))


def fasta_filter(text: str, maxtandem: float, params: Dict[str, int] = None) -> Tuple[str, str]:
    """`mimeo filter` on a FASTA text: returns (the records kept, i.e. every record unless 100*m/L > maxtandem, with L = 0
    kept; every record with its masked positions replaced by N), both as FASTA text wrapped at 60 columns in input order."""
    p = dict(to.DEFAULTS, **(params or {}))
    kept, masked = [], []
    for header, seq in fasta_records(text):
        m, runs = to.mask(seq, **p) if seq else (0, [])
        if not seq or not (100.0 * m / len(seq) > maxtandem):
            kept.append(fasta_text(header, seq))
        s = list(seq)
        for a, e in runs:
            s[a:e + 1] = 'N' * (e + 1 - a)
        masked.append(fasta_text(header, ''.join(s)))
    return ''.join(kept), ''.join(masked)
