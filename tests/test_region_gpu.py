"""The region report on the device (meth_region_kernel of bsx_meth.cu, `methratio --region-report`, `bsmap --methratio
--meth-region-report`) against the numpy restatement (oracle/region_oracle.py) and the lines of the -z table of the same
run, and a spike-in's conversion rate recovered end to end."""
from __future__ import annotations

import os
import subprocess
import sys

import numpy as np
import pytest

import cases as CS
from meth_inputs import api_arrays
from test_methratio_cpu import MANIFEST, alignment_files, opts_kwargs
from test_mbias_cpu import oracle_files
from test_region_cpu import random_regions

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import conversion_oracle as CV  # noqa: E402
import region_oracle as RO  # noqa: E402

import bsmap_b200 as B
from bsmap_b200 import lib as BL
from bsmap_b200 import synth

pytestmark = pytest.mark.gpu
BIN = os.path.dirname(BL.LIB_PATH)
METHRATIO, BSMAP = os.path.join(BIN, "methratio"), os.path.join(BIN, "bsmap")
IGNORE = (2, 1, 3, 2)

# name -> (option overrides, C/T SNP mode, conversion threshold with M-bias and exclusion, or None)
VARIANTS = {
    "plain": ({}, None, None),
    "g": ({"combine_cpg": True}, None, None),
    "m3": ({"min_depth": 3}, None, None),
    "skip": ({}, "skip", None),
    "correct": ({}, "correct", None),
    "g_correct": ({"combine_cpg": True}, "correct", None),
    "conv_mbias": ({}, None, 2),
}
API_KEYS = ["pe_sam.r", "se_cfg2_bsp.r_u", "pe_readthrough.p_g", "se_cfg1.u"]


def to_idx(regs, names):
    k = {n: i for i, n in enumerate(names)}
    return [k[c] for c, _, _ in regs], [s for _, s, _ in regs], [e for _, _, e in regs]


@pytest.mark.parametrize("key", API_KEYS)
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_regions_equal_the_oracle(tmp_path, key, variant):
    """Meth.regions after bsx_meth_add in one and in three batches == oracle on random regions: single positions, empty,
    across many chunks, straddling chunk edges, clipped; without -g also asked between the batches, which must leave the
    counters as they were"""
    over, ct_snp, threshold = VARIANTS[variant]
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    bsp = not files[0].upper().endswith(".SAM")
    if threshold is not None and bsp:
        pytest.skip("BSP records carry no read number (M-bias)")
    kw = dict(opts_kwargs(ent["opts"]), **over)
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth")}
    ignore = IGNORE if threshold is not None else (0, 0, 0, 0)
    res = CV.conversion(d["gnames"], d["gseqs"], files, threshold=threshold or 0, ignore=ignore, **ckw)
    if threshold:
        assert res["dropped"] > 0
    ref = {n: (s.decode() if isinstance(s, bytes) else s) for n, s in zip(d["gnames"], d["gseqs"])}
    regs = random_regions({n: len(s) for n, s in ref.items()}, 400, seed=len(key) * 31 + len(variant))
    exp = RO.regions(res["counters"], ref, regs, combine_cpg=kw.get("combine_cpg", False), min_depth=kw.get("min_depth", 1), ct_snp=ct_snp)
    assert exp[:, :, 1].sum() > 0
    cols = api_arrays(files, d["gnames"])
    ix = B.Index.packed(d["gnames"], d["gseqs"])
    ci, st, en = to_idx(regs, d["gnames"])
    for batches in (1, 3):
        mh = B.Meth(ix, B.meth_opts(**kw))
        if threshold is not None:
            mh.enable_conversion_filter(threshold)
            mh.enable_mbias()
            mh.set_ignore(*IGNORE)
        if ct_snp:
            mh.enable_ct_snp(ct_snp)
        n = len(cols[0])
        cut = [n * k // batches for k in range(batches + 1)]
        for b, e in zip(cut, cut[1:]):
            mh.add(*[c[b:e] for c in cols[:7]], read2=cols[7][b:e])
            if not kw.get("combine_cpg") and e < n:
                mh.regions(ci, st, en)                     # a look in between changes nothing
        got = mh.regions(ci, st, en)
        assert got.dtype == np.uint64 and got.shape == (len(regs), 3, 4)
        assert np.array_equal(got.astype(np.int64), exp), (batches, np.argwhere(got.astype(np.int64) != exp)[:5])
        mh.close()
    ix.close()


def test_write_regions_and_misuse(tmp_path):
    ix = B.Index.packed(["a", "b"], [b"ACGTTCAGCA" * 50, b"CCGG" * 10])
    mh = B.Meth(ix, B.meth_opts())
    mh.add([b"ACGTTCAGCA", b"CTGG"], [0, 1], [0, 4], [0, 0], [0, 0], [0, 0], [4, 4])
    regs = [("b", 0, 100), ("a", 3, 3), ("a", 0, 10)]
    path = tmp_path / "r.txt"
    fd = os.open(path, os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    mh.write_regions(fd, *to_idx(regs, ["a", "b"]))
    os.close(fd)
    ma, da = mh.counters(0)
    mb, db = mh.counters(1)
    cnt = {"a": (ma, da), "b": (mb, db)}
    ref = {"a": "ACGTTCAGCA" * 50, "b": "CCGG" * 10}
    assert path.read_text() == RO.report_text(regs, RO.regions(cnt, ref, regs))
    assert mh.regions([], [], []).shape == (0, 3, 4)
    with pytest.raises(B.BsxError, match="start 5 > end 4"):
        mh.regions([0], [5], [4])
    with pytest.raises(B.BsxError, match="sequence 2 of 2"):
        mh.regions([2], [0], [4])
    mh.close(); ix.close()


# ---- command lines ---------------------------------------------------------------------------------------------------
BED = ("# promoters\r\ntrack name=test\r\nbrowser position chr1:1-1000\n\n"
       "chr1\t1000\t9000\tp1\t0\t+\r\n"
       "chrUn\t0\t100\n"
       "chr2\t4095\t4097\n"
       "chr3\t250000\t400000\tclipped\n"
       "chr1\t5000\t5000\n"
       "chr1\t0\t300000\n"
       "chr1\t1000\t9000\n")


def check_report(report, table, ref, regs, res, kw, ct_snp=None):
    """the report == the oracle, and its covered / C / CT == the lines of the -z table of the same run"""
    exp = RO.regions(res["counters"], ref, regs, combine_cpg=kw.get("combine_cpg", False), min_depth=kw.get("min_depth", 1), ct_snp=ct_snp)
    assert report == RO.report_text(regs, exp)
    assert np.array_equal(exp[:, :, 1:], RO.table_line_sums(table, ref, regs))
    assert exp[:, :, 1].sum() > 0


CLI_KEYS = ["pe_sam.default", "se_cfg2_r0_uR.bam.default", "se_cfg2_bsp.default", "se_cfg1.g_z"]


@pytest.mark.parametrize("key", CLI_KEYS)
def test_methratio_cli(tmp_path, key):
    """methratio -z --region-report F with --tiles W and with --regions BED (comments, CRLF, an unknown and an unselected
    sequence, a clipped end), on SAM, BAM and BSP; the skip line; the table and summary as without the report"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    fa, _, _ = CS.write_inputs(case, str(tmp_path))
    files = alignment_files(case, str(tmp_path), bam=ent.get("bam", False))
    ofiles = oracle_files(ent, case, str(tmp_path))
    opts = [o for o in ent["opts"] if o != "-z"] + ["-z"]
    kw = opts_kwargs(opts)
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth")}
    bed = tmp_path / "r.bed"
    bed.write_bytes(BED.encode())
    out, out0, rep = str(tmp_path / "m.txt"), str(tmp_path / "m0.txt"), str(tmp_path / "rep.txt")
    r0 = subprocess.run([METHRATIO, "-o", out0, "-d", fa, "-q"] + opts + files, capture_output=True, text=True)
    assert r0.returncode == 0, r0.stderr
    for sel, args in ((None, ["--tiles", "1000"]), (None, ["--regions=" + str(bed)]), (["chr1", "chr3"], ["--regions", str(bed)]),
                      (None, ["--tiles=7777", "--ct-snp", "skip"])):
        ct_snp = "skip" if "--ct-snp" in args else None
        copt = ["-c", ",".join(sel)] if sel else []
        r = subprocess.run([METHRATIO, "-o", out, "-d", fa, "-q", "--region-report", rep] + copt + args + opts + files, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        res = CV.conversion(d["gnames"], d["gseqs"], ofiles, chroms=sel, **ckw)
        ref = {n: s.decode() for n, s in zip(d["gnames"], d["gseqs"]) if not sel or n in sel}
        if "--tiles" in args[0]:
            regs = RO.tiles({n: len(s) for n, s in ref.items()}, int(args[0].split("=")[-1]) if "=" in args[0] else int(args[1]))
        else:
            regs, skipped = RO.parse_bed(BED, set(ref))
            assert RO.skip_line(skipped, skipped + len(regs)) in r.stderr.splitlines()
        table = open(out).read()
        check_report(open(rep).read(), table, ref, regs, res, kw, ct_snp)
        if not sel and not ct_snp:
            assert table == open(out0).read() and r.stdout == r0.stdout


def test_methratio_usage_errors(tmp_path):
    case = CS.BY_NAME["se_n1"]
    fa, _, _ = CS.write_inputs(case, str(tmp_path))
    sam = alignment_files(case, str(tmp_path))[0]
    bed = tmp_path / "r.bed"
    bed.write_text("chr1\t0\t10\n")
    base = [METHRATIO, "-o", str(tmp_path / "t"), "-d", fa, "-q"]
    for args in (["--regions", str(bed)], ["--tiles", "10"], ["--region-report", "x"], ["--region-report", "x", "--tiles", "5", "--regions", str(bed)],
                 ["--region-report", "x", "--tiles", "0"], ["--region-report", "x", "--tiles", "-3"], ["--region-report", "x", "--tiles", "2.5"]):
        r = subprocess.run(base + args + [sam], capture_output=True, text=True)
        assert r.returncode == 2 and "methratio: error:" in r.stderr, args
    for text, msg in (("#\nchr1\t5\n", ":2: fewer than 3 columns"), ("chr1\t0\t10\nchr1\tx\t5\n", ":2: start and end"),
                      ("\nchr1\t9\t5\n", ":2: start 9 > end 5")):
        bed.write_text(text)
        r = subprocess.run(base + ["--region-report", str(tmp_path / "rep"), "--regions", str(bed), sam], capture_output=True, text=True)
        assert r.returncode == 1 and msg in r.stderr, (text, r.stderr)


@pytest.mark.parametrize("name,ext", [("se_cfg2_r0_uR", "sam"), ("pe_sam", "sam"), ("se_cfg2_bsp", "bsp")])
def test_bsmap_cli(tmp_path, name, ext):
    """bsmap --methratio T --meth-zero --meth-region-report F (in-process pile-up) == methratio on the alignment file
    the same run wrote, == the oracle and the lines of its table; the table and summary as without the report"""
    case = CS.BY_NAME[name]
    d = case.data()
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / ("out." + ext))
    t0, t, rep, rep2 = (str(tmp_path / x) for x in ("t0", "t", "rep", "rep2"))
    bed = tmp_path / "r.bed"
    bed.write_bytes(BED.encode())
    r0 = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t0, "--meth-zero"], capture_output=True, text=True)
    assert r0.returncode == 0, r0.stdout + r0.stderr
    ref = {n: s.decode() for n, s in zip(d["gnames"], d["gseqs"])}
    for args, margs in ((["--meth-tiles", "1000"], ["--tiles", "1000"]), (["--meth-regions", str(bed)], ["--regions", str(bed)])):
        r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t, "--meth-zero", "--meth-region-report", rep] + args,
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        assert open(t).read() == open(t0).read()
        summary = lambda out: [x for x in out.splitlines() if "valid mappings" in x]
        assert summary(r.stdout) == summary(r0.stdout)
        res = CV.conversion(d["gnames"], d["gseqs"], [o])
        if "--meth-tiles" in args:
            regs = RO.tiles({n: len(s) for n, s in ref.items()}, 1000)
        else:
            regs, skipped = RO.parse_bed(BED, set(ref))
            assert RO.skip_line(skipped, skipped + len(regs)) in r.stderr.splitlines()
        check_report(open(rep).read(), open(t).read(), ref, regs, res, {})
        m = subprocess.run([METHRATIO, "-o", str(tmp_path / "mt"), "-d", fa, "-q", "-z", "--region-report", rep2] + margs + [o], capture_output=True, text=True)
        assert m.returncode == 0, m.stderr
        assert open(rep).read() == open(rep2).read()


def test_bsmap_usage_errors(tmp_path):
    case = CS.BY_NAME["se_n1"]
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / "o.sam")
    bed = tmp_path / "r.bed"
    bed.write_text("chr1\t0\t10\n")
    for opt in (["--meth-region-report", "x", "--meth-tiles", "5"], ["--meth-regions", str(bed)], ["--meth-tiles", "5"]):
        r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + opt, capture_output=True, text=True)
        assert r.returncode != 0 and "need --methratio" in r.stderr, opt
    t = ["--methratio", str(tmp_path / "t")]
    for opt, msg in ((["--meth-regions", str(bed)], "need --meth-region-report"), (["--meth-tiles", "5"], "need --meth-region-report"),
                     (["--meth-region-report", "x"], "needs --meth-regions"),
                     (["--meth-region-report", "x", "--meth-tiles", "5", "--meth-regions", str(bed)], "exclude each other")):
        r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + t + opt, capture_output=True, text=True)
        assert r.returncode != 0 and msg in r.stderr, (opt, r.stderr)
    for bad in ("0", "-1", "x", "1.5"):
        r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + t + ["--meth-region-report", "x", "--meth-tiles", bad], capture_output=True, text=True)
        assert r.returncode != 0 and ("unknown option: " + bad) in r.stdout, bad
    bed.write_text("chr1\t10\t5\n")
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + t + ["--meth-region-report", "x", "--meth-regions", str(bed)], capture_output=True, text=True)
    assert r.returncode == 1 and ":1: start 10 > end 5" in r.stderr


# ---- a spike-in's conversion rate end to end --------------------------------------------------------------------------
def test_spike_in_level_end_to_end(tmp_path):
    """a 150 kb genome converted at 70 % plus a 48.5 kb lambda-like spike-in converted at 99 %: the spike-in's whole-
    sequence region reports 1 - 0.99 in every context within a binomial tolerance (the genome 0.3), and 1 kb tiles over
    the same counters sum to the same four integers"""
    import torch
    g = synth.make_genome(21, [150_000, 48_502])
    sims = [synth.simulate_reads([g[0]], 30_000, 100, seed=31, subs="none", conv=0.70),
            synth.simulate_reads([g[1]], 12_000, 100, seed=32, subs="none", conv=0.99)]
    seqs = torch.cat([s["seq"] for s in sims]).numpy()
    fa, fq, sam = str(tmp_path / "g.fa"), str(tmp_path / "r.fq"), str(tmp_path / "o.sam")
    names = ["chr1", "lambda"]
    synth.write_fasta(fa, g, names=names)
    synth.write_fastq(fq, seqs, ["r%d" % i for i in range(len(seqs))])
    bed = tmp_path / "w.bed"
    bed.write_text("chr1\t0\t150000\nlambda\t0\t48502\n")
    t, rep = str(tmp_path / "t"), str(tmp_path / "rep")
    r = subprocess.run([BSMAP, "-a", fq, "-d", fa, "-o", sam, "-v", "5", "--methratio", t, "--meth-region-report", rep, "--meth-regions", str(bed)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    rows = [x.split("\t") for x in open(rep).read().splitlines()[1:]]
    assert len(rows) == 6
    for row, conv in zip(rows, [0.70] * 3 + [0.99] * 3):
        c, ct = int(row[6]), int(row[7])
        p = 1 - conv
        assert ct > 2000 and abs(c / ct - p) < 5 * (p * (1 - p) / ct) ** 0.5 + 0.002, row
        assert row[8] == "%.4f" % (c / ct)
    # the same counters through bsx_meth_add: whole sequences == the report, and 1 kb tiles sum to them
    ix = B.Index.packed(names, [x.numpy().tobytes() for x in g])
    mh = B.Meth(ix, B.meth_opts())
    cols = api_arrays([sam], names)
    mh.add(*cols[:7], read2=cols[7])
    whole = mh.regions([0, 1], [0, 0], [150_000, 48_502]).astype(np.int64)
    assert [[int(x) for x in r[4:8]] for r in rows] == whole.reshape(6, 4).tolist()
    tiles = RO.tiles({"chr1": 150_000, "lambda": 48_502}, 1000)
    per = mh.regions(*to_idx(tiles, names)).astype(np.int64)
    assert np.array_equal(per[:150].sum(axis=0), whole[0]) and np.array_equal(per[150:].sum(axis=0), whole[1])
    mh.close(); ix.close()
