"""The methratio fuzz generator (tests/meth_fuzz.py) without a GPU: it is deterministic per seed, every record it writes
parses through the oracle's own parser, and on its files the composed oracle it compares the device with
(conversion_oracle at threshold 0, no exclusion) prints the same table as methratio_oracle, the restatement pinned
against the reference script."""
import os
import sys

import numpy as np
import pytest

import meth_fuzz as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import conversion_oracle as CV  # noqa: E402
import methratio_oracle as MO  # noqa: E402


def generate(seed, n=400):
    rng = np.random.default_rng(seed)
    names, seqs = F.make_reference(rng, big=(10_000, 40_000))
    sam = rng.random() < 0.7
    o = F.draw_options(rng, names, seqs, sam)
    recs = F.make_records(rng, names, seqs, n, rm_dup=o["rm_dup"])
    return names, seqs, o, recs


def test_generator_is_deterministic_per_seed():
    for seed in (1, 2):
        a, b = generate(seed), generate(seed)
        assert a[0] == b[0] and a[1] == b[1] and a[3] == b[3]
        assert F.sam_text(a[3], a[0], a[1]) == F.sam_text(b[3], b[0], b[1])
    assert generate(1)[3] != generate(2)[3]


@pytest.mark.parametrize("seed", range(6))
def test_records_parse_and_cover_the_edges(tmp_path, seed):
    names, seqs, o, recs = generate(seed)
    sam, bsp = tmp_path / "a.sam", tmp_path / "a.bsp"
    sam.write_text(F.sam_text(recs, names, seqs))
    bsp.write_text(F.bsp_text(recs))
    known = set(names)
    for path in (sam, bsp):
        alns = MO.parse_alignments(str(path), known)
        n = sum(1 for r in recs if r["chrom"] in known and not r["flag"] & 0x4)
        assert len(alns) == n
    strands = {r["strand"] for r in recs}
    assert strands == set(F.STRANDS)
    size = dict(zip(names, (len(s) for s in seqs)))
    ends = [r["pos"] + max(len(r["seq"]), 1) - size[r["chrom"]] for r in recs if r["chrom"] in size and r["seq"] != "*"]
    assert {-1, 0}.issubset(ends) or o["rm_dup"]                        # alignments ending one before and at the end
    assert any(r["seq"] == "*" for r in recs) or len(recs) < 100
    assert any(0 < abs(r["insert"]) < len(r["seq"]) for r in recs)
    assert any(0 < r["pnext"] < r["pos"] + 1 for r in recs) and any(r["pnext"] > r["pos"] + len(r["seq"]) for r in recs)


def test_letter_flags_mean_the_numeric_bits():
    rng = np.random.default_rng(3)
    names, seqs = ["c"], [b"ACGT" * 50]
    recs = F.make_records(rng, names, seqs, 200)
    num = F.sam_text(recs, names, seqs).splitlines()
    let = F.sam_text(recs, names, seqs, letters=[True] * len(recs)).splitlines()
    for a, b in zip(num, let):
        if a.startswith("@"):
            continue
        f, s = int(a.split("\t")[1]), b.split("\t")[1]
        assert int(s) == f if s.isdigit() else sum(1 << F.FLAG_LETTERS.index(ch) for ch in s) == f


@pytest.mark.parametrize("seed", range(8))
def test_composed_oracle_equals_the_pinned_one(tmp_path, seed):
    """conversion_oracle (threshold 0, no exclusion) + its table == methratio_oracle.methratio on the generated files,
    with the round's -u -p -z -r -t -g -m -c"""
    names, seqs, o, recs = generate(seed)
    sam = seed % 3 != 2
    path = str(tmp_path / ("a.sam" if sam else "a.bsp"))
    open(path, "w").write(F.sam_text(recs, names, seqs) if sam else F.bsp_text(recs))
    kw = dict(chroms=o["chroms"], unique=o["unique"], pair=o["pair"], trim_fillin=o["trim_fillin"], combine_cpg=o["combine_cpg"], rm_dup=o["rm_dup"])
    res = CV.conversion(names, seqs, [path], **kw)
    got, (nc, nd) = CV.table(res, meth0=o["meth0"], min_depth=o["min_depth"])
    exp, (nmap, enc, end) = MO.methratio(names, seqs, [path], meth0=o["meth0"], min_depth=o["min_depth"], **kw)
    assert got == exp
    assert (res["valid"], nc, nd) == (nmap, enc, end)
    assert len(exp.splitlines()) > 1
