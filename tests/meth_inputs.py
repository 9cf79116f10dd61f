"""SAM / BSP alignment text as bsx_meth_add takes it (host arrays), for the M-bias tests and tests/mbias_bench.py."""
from __future__ import annotations

import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import methratio_oracle as MO  # noqa: E402


def api_arrays(files, names):
    """-> columns seqs, chr index, pos, strand bits, insert, mate_pos, BSX_METH_* flags, read2 (FLAG 0x80) of the
    alignments methratio_oracle.parse_alignments keeps, in file order"""
    idx = {n: k for k, n in enumerate(names)}
    rows = []
    for path in files:
        sam = path.upper().endswith(".SAM")
        raw = []
        for line in open(path):
            col = line.rstrip("\n").split("\t")
            if sam:
                if line.startswith("@") or int(col[1]) & 4 or col[2] not in idx:
                    continue
                f = int(col[1])
                raw.append(((1 if f & 0x100 else 0) | (2 if f & 0x2 else 0) | 4, bool(f & 0x80)))
            else:
                if col[3][:2] in ("NM", "QC") or col[4] not in idx:
                    continue
                raw.append(((0 if col[3][:2] == "UM" else 1) | (0 if col[7] == "0" else 2), False))
        alns = MO.parse_alignments(path, set(names))
        assert len(alns) == len(raw)
        for (seq, st, cr, p, insert, mate_pos, s), (fl, r2) in zip(alns, raw):
            rows.append((seq.encode(), idx[cr], p, (1 if st[0] == "-" else 0) | (2 if st[1] == "-" else 0), insert, mate_pos if s else 0, fl, r2))
    return [list(c) for c in zip(*rows)]
