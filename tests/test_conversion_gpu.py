"""The conversion filter on the device (the Conv pile-up kernels of bsx_meth.cu, `methratio --conversion-filter`,
`bsmap --methratio --meth-conversion-filter`) against the numpy restatement (oracle/conversion_oracle.py), and
unconverted reads mapped end to end."""
from __future__ import annotations

import os
import subprocess
import sys

import numpy as np
import pytest

import cases as CS
import runners as R
from meth_inputs import api_arrays
from test_methratio_cpu import MANIFEST, alignment_files, opts_kwargs
from test_mbias_cpu import NAMES, SEQS, oracle_files
from test_conversion_cpu import KATS, kat_file

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import conversion_oracle as CV  # noqa: E402

import bsmap_b200 as B
from bsmap_b200 import lib as BL
from bsmap_b200 import synth

pytestmark = pytest.mark.gpu
BIN = os.path.dirname(BL.LIB_PATH)
METHRATIO, BSMAP = os.path.join(BIN, "methratio"), os.path.join(BIN, "bsmap")
IGNORE = (2, 1, 3, 2)
# (M-bias + exclusion, C/T SNP mode)
VARIANTS = [(False, None), (True, None), (False, "correct"), (True, "correct")]


def add_all(mh, cols, batches=1):
    n = len(cols[0])
    cut = [n * k // batches for k in range(batches + 1)]
    for b, e in zip(cut, cut[1:]):
        if e > b:
            mh.add(*[c[b:e] for c in cols[:7]], read2=cols[7][b:e])


def make_meth(ix, opts, threshold, mbias=False, ct_snp=None, ignore=None):
    mh = B.Meth(ix, opts)
    mh.enable_conversion_filter(threshold)
    if mbias:
        mh.enable_mbias()
    if ignore:
        mh.set_ignore(*ignore)
    if ct_snp:
        mh.enable_ct_snp(ct_snp)
    return mh


def same_as_oracle(mh, names, res, mbias=False, ct_snp=None):
    assert mh.valid() == res["valid"]
    bins, dropped = mh.conversion()
    assert np.array_equal(bins.astype(np.int64), res["bins"]) and dropped == res["dropped"]
    for k, n in enumerate(names):
        m, dp = mh.counters(k)
        exp = res["counters"][n]
        assert np.array_equal(m, exp[0]) and np.array_equal(dp, exp[1]), n
        if ct_snp:
            c, s = mh.ct_snp_counters(k)
            assert np.array_equal(c, exp[2]) and np.array_equal(s, exp[3]), n
    if mbias:
        hist, over = mh.mbias()
        assert np.array_equal(hist.astype(np.int64), res["mbias"]) and over == res["mbias_overflow"]


# SE / PE SAM, BSP, BAM, RRBS, -r, -g, -u / -p, -t
API_KEYS = ["pe_sam.p_u", "pe_sam.r", "pe_readthrough.p_g", "se_n1.r_t_0", "se_n1.t_5_g", "rrbs_pe.t_0", "pe_sam_v5_R.r_p",
            "se_cfg1.u", "se_cfg2_bsp.r_u", "pe_sam.bam.r", "rrbs_se_A.bam.r_u"]


@pytest.mark.parametrize("key", API_KEYS)
def test_meth_add_equals_the_oracle(tmp_path, key):
    """bsx_meth_add over three batches, thresholds 0 / 1 / 3, alone, with M-bias + exclusion, with C/T SNP evidence and
    with both: counters, evidence, M-bias, score histogram and dropped == oracle"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = opts_kwargs(ent["opts"])
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth")}
    bsp = not files[0].upper().endswith(".SAM")
    cols = api_arrays(files, d["gnames"])
    ix = B.Index.packed(d["gnames"], d["gseqs"])
    dropped = 0
    for threshold in (0, 1, 3):
        for mbias, ct_snp in VARIANTS:
            if mbias and bsp:
                continue                                          # BSP records carry no read number
            ignore = IGNORE if mbias else None
            res = CV.conversion(d["gnames"], d["gseqs"], files, threshold=threshold, ignore=ignore or (0, 0, 0, 0), **ckw)
            mh = make_meth(ix, B.meth_opts(**kw), threshold, mbias, ct_snp, ignore)
            add_all(mh, cols, batches=3)
            same_as_oracle(mh, d["gnames"], res, mbias, ct_snp)
            mh.close()
            dropped += res["dropped"]
    assert dropped > 0
    ix.close()


@pytest.mark.parametrize("name", sorted(k for k in KATS if KATS[k][1].get("sam_rules") is not False))   # SAM text takes SAM rules
def test_known_scores_on_the_device(tmp_path, name):
    """the hand-computed cases through bsx_meth_add, one batch per record, with M-bias; upper- and lower-case reference"""
    lines, kw, exp = KATS[name]
    sam = kat_file(tmp_path, lines)
    for seqs in (SEQS, [s.lower() for s in SEQS]):               # a lower-case reference reads as upper case
        res = CV.conversion(NAMES, seqs, [sam], **kw)
        assert res["scores"] == [exp]
        ix = B.Index.packed(NAMES, seqs)
        opts = B.meth_opts(trim_fillin=kw.get("trim_fillin", 2), rm_dup=kw.get("rm_dup", False), combine_cpg=kw.get("combine_cpg", False))
        mh = make_meth(ix, opts, kw.get("threshold", 0), mbias=True, ignore=kw.get("ignore"))
        add_all(mh, api_arrays([sam], NAMES), batches=len(lines))
        same_as_oracle(mh, NAMES, res, mbias=True)
        mh.close(); ix.close()


def test_last_bin_on_the_device(tmp_path):
    names, seqs = ["c"], [b"C" * 300 + b"A" * 20]
    from test_mbias_cpu import sam_line
    sam = kat_file(tmp_path, [sam_line(0, "c", 1, "C" * 300, "++"), sam_line(0, "c", 1, "C" * 255, "++"), sam_line(0, "c", 1, "C" * 254 + "T", "++")])
    res = CV.conversion(names, seqs, [sam], threshold=255)
    ix = B.Index.packed(names, seqs)
    mh = make_meth(ix, B.meth_opts(), 255)
    add_all(mh, api_arrays([sam], names))
    same_as_oracle(mh, names, res)
    rep = tmp_path / "rep.txt"
    fd = os.open(rep, os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    mh.write_conversion(fd)
    os.close(fd)
    assert rep.read_text() == CV.report_text(res["bins"], 255) == CV.HEADER + "254\t1\t0\n255+\t2\t1\n"
    mh.close(); ix.close()


CLI_KEYS = ["pe_sam.default", "pe_sam.r", "se_cfg2_bsp.default", "pe_bsp_r0.r", "se_cfg2_r0_uR.bam.default", "se_n1.t_5_g", "rrbs_se_A.z"]


@pytest.mark.parametrize("key", CLI_KEYS)
def test_methratio_cli(tmp_path, key):
    """methratio --conversion-filter N --conversion-report F (SAM, BAM and BSP): table and report == oracle, the stderr
    line, and the summary line's valid mappings unchanged; --conversion-report alone is N = 0"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    fa, _, _ = CS.write_inputs(case, str(tmp_path))
    files = alignment_files(case, str(tmp_path), bam=ent.get("bam", False))
    kw = opts_kwargs(ent["opts"])
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth")}
    ofiles = oracle_files(ent, case, str(tmp_path))
    out, rep = str(tmp_path / "meth.txt"), str(tmp_path / "rep.txt")
    for threshold, args in ((3, ["--conversion-filter", "3", "--conversion-report", rep]), (0, ["--conversion-report=" + rep]),
                            (1, ["--conversion-filter=1", "--conversion-report", rep, "--ct-snp", "correct"])):
        res = CV.conversion(d["gnames"], d["gseqs"], ofiles, threshold=threshold, **ckw)
        r = subprocess.run([METHRATIO, "-o", out, "-d", fa, "-q"] + args + ent["opts"] + files, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        assert r.stdout.split(",")[0] == ent["stdout"].split(",")[0]        # "total N valid mappings"
        txt, _ = CV.table(res, meth0=kw.get("meth0", False), min_depth=kw.get("min_depth", 1), ct_snp="correct" if "--ct-snp" in args else None)
        assert open(out).read() == txt, (threshold, R.first_diff(open(out, "rb").read(), txt.encode()))
        assert open(rep).read() == CV.report_text(res["bins"], threshold)
        assert CV.stderr_line(res, threshold) in r.stderr.splitlines()


@pytest.mark.parametrize("name,ext", [("se_cfg2_r0_uR", "sam"), ("pe_sam", "sam"), ("se_cfg2_bsp", "bsp")])
def test_bsmap_cli(tmp_path, name, ext):
    """bsmap --methratio T --meth-conversion-filter 3 --meth-conversion-report F (in-process pile-up): table and report
    == oracle on the alignment file the same run wrote, the stderr line, and the same summary as without the filter"""
    case = CS.BY_NAME[name]
    d = case.data()
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / ("out." + ext))
    t, rep = str(tmp_path / "t"), str(tmp_path / "rep")
    r0 = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t, "--meth-zero"], capture_output=True, text=True)
    assert r0.returncode == 0, r0.stdout + r0.stderr
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t, "--meth-zero", "--meth-conversion-filter", "3", "--meth-conversion-report", rep],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    summary = [x for x in r.stdout.splitlines() if "valid mappings" in x]
    assert summary[0].split(",")[0] == [x for x in r0.stdout.splitlines() if "valid mappings" in x][0].split(",")[0]
    res = CV.conversion(d["gnames"], d["gseqs"], [o], threshold=3)
    assert open(t).read() == CV.table(res, meth0=True)[0]
    assert open(rep).read() == CV.report_text(res["bins"], 3)
    assert CV.stderr_line(res, 3) in r.stderr.splitlines()
    assert summary[0].startswith("total %d valid mappings" % res["valid"])


def _map_in_process(case, max_batch, threshold=3, mbias=False, ignore=None, ct_snp=None):
    d = case.data()
    p = B.make_params(**case.param_kwargs())
    ix = B.Index(p, d["gnames"], d["gseqs"])
    mp = B.Mapper(ix, p, max_batch=max_batch, stride=160)
    mh = make_meth(ix, B.meth_opts(), threshold, mbias, ct_snp, ignore)
    mh.attach(mp, sam_rules=bool(p.out_sam))
    if not case.paired:
        buf, lens = B.pack_reads(R.clip(case, d["seqs"]), stride=160)
        mp.map_se(buf, lens)
    else:
        ba, la = B.pack_reads(R.clip(case, d["seqs"]), stride=160)
        bb, lb = B.pack_reads(R.clip(case, d["seqs_b"]), stride=160)
        mp.map_pe(ba, la, bb, lb)
    return d, ix, mp, mh


@pytest.mark.parametrize("name", ["se_cfg2_r0_uR", "pe_sam", "rrbs_pe", "se_cfg2_bsp"])
def test_in_process_equals_the_oracle(tmp_path, name):
    """Mapper + attached Meth, many batches on both streams (Conv, and Conv + M-bias + exclusion + Snp): == oracle on
    the text the records format to"""
    case = CS.BY_NAME[name]
    files = alignment_files(case, str(tmp_path))          # the golden text == what these records format to
    bsp = not files[0].upper().endswith(".SAM")
    for mbias, ct_snp in ((False, None), (not bsp, "correct")):
        ignore = IGNORE if mbias else None
        d, ix, mp, mh = _map_in_process(case, max_batch=256, mbias=mbias, ignore=ignore, ct_snp=ct_snp)
        res = CV.conversion(d["gnames"], d["gseqs"], files, threshold=3, ignore=ignore or (0, 0, 0, 0))
        same_as_oracle(mh, d["gnames"], res, mbias, ct_snp)
        mh.close(); mp.close(); ix.close()


@pytest.mark.parametrize("name", ["se_n1", "pe_sam"])
def test_batch_size_invariance(name):
    """64 and 1 M alignments per batch give the same counters and histograms"""
    res = []
    for mb in (64, 1 << 20):
        d, ix, mp, mh = _map_in_process(CS.BY_NAME[name], max_batch=mb, threshold=1, mbias=True, ignore=(1, 2, 3, 4))
        res.append((mh.conversion(), mh.mbias()[0], [mh.counters(k) for k in range(len(d["gnames"]))]))
        mh.close(); mp.close(); ix.close()
    (c0, m0, k0), (c1, m1, k1) = res
    assert np.array_equal(c0[0], c1[0]) and c0[1] == c1[1] and c0[1] > 0 and np.array_equal(m0, m1)
    for a, b in zip(k0, k1):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_misuse_is_refused(tmp_path):
    ix = B.Index.packed(["c"], [b"ACGT" * 100])
    mh = B.Meth(ix, B.meth_opts())
    for bad in (-1, 256):
        with pytest.raises(B.BsxError, match="threshold must be 0..255"):
            mh.enable_conversion_filter(bad)
    with pytest.raises(B.BsxError, match="not enabled"):
        mh.conversion()
    mh.add([b"ACGTACGT"], [0], [0], [0], [0], [0], [4])
    with pytest.raises(B.BsxError, match="error 1:.*already piled up"):
        mh.enable_conversion_filter(3)
    mh.close(); ix.close()
    case = CS.BY_NAME["se_n1"]
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / "o.sam")
    for opt in (["--meth-conversion-filter", "3"], ["--meth-conversion-report", str(tmp_path / "r")]):
        r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + opt, capture_output=True, text=True)
        assert r.returncode != 0 and "--methratio" in r.stderr
    for bad in ("x", "3.5", "256", "-1"):
        r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", str(tmp_path / "t"), "--meth-conversion-filter", bad], capture_output=True, text=True)
        assert r.returncode != 0 and ("unknown option: " + bad) in r.stdout, bad
        r = subprocess.run([METHRATIO, "-o", str(tmp_path / "t"), "-d", fa, "--conversion-filter", bad, o], capture_output=True, text=True)
        assert r.returncode == 2 and "--conversion-filter" in r.stderr, bad


# ---- unconverted reads end to end -----------------------------------------------------------------------------------
GLEN, RLEN, NREADS = 120_000, 100, 40_000


def chh_ratio(text):
    """sum C / sum CT over the CHH rows of a plain table"""
    c = t = 0
    for line in text.splitlines()[1:]:
        col = line.split("\t")
        ctx = col[3]
        if len(ctx) == 5 and (ctx[3] != "G" and ctx[4] != "G" if col[2] == "+" else ctx[1] != "C" and ctx[0] != "C"):
            c += int(col[6]); t += int(col[5])
    return c / t


def test_unconverted_reads_end_to_end(tmp_path):
    """90 % of the reads converted at 99.5 %, 10 % not converted at all: with --meth-conversion-filter 3 every mapped
    unconverted read is dropped, at most 0.5 % of the converted ones are, and the CHH level falls from about 11 % to
    under 1.5 %; table and report == oracle on the SAM of the same run"""
    import torch
    g = synth.make_genome(7, [GLEN])
    n_u = NREADS // 10
    sims = [synth.simulate_reads(g, NREADS - n_u, RLEN, seed=11, conv=0.995), synth.simulate_reads(g, n_u, RLEN, seed=12, conv=0.0)]
    seqs = torch.cat([s["seq"] for s in sims]).numpy()
    names = ["c%d" % i for i in range(NREADS - n_u)] + ["u%d" % i for i in range(n_u)]
    fa, fq, sam = str(tmp_path / "g.fa"), str(tmp_path / "r.fq"), str(tmp_path / "o.sam")
    synth.write_fasta(fa, g, names=["chr1"])
    synth.write_fastq(fq, seqs, names)
    t0, t, rep = str(tmp_path / "t0"), str(tmp_path / "t"), str(tmp_path / "rep")
    r0 = subprocess.run([BSMAP, "-a", fq, "-d", fa, "-o", sam, "-v", "5", "--methratio", t0, "--meth-zero"], capture_output=True, text=True)
    assert r0.returncode == 0, r0.stdout + r0.stderr
    r = subprocess.run([BSMAP, "-a", fq, "-d", fa, "-o", sam, "-v", "5", "--methratio", t, "--meth-zero", "--meth-conversion-filter", "3",
                        "--meth-conversion-report", rep], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    gb = g[0].numpy().tobytes()
    res = CV.conversion(["chr1"], [gb], [sam], threshold=3)
    assert open(t).read() == CV.table(res, meth0=True)[0]
    assert open(rep).read() == CV.report_text(res["bins"], 3)
    valid = lambda out: [x for x in out.splitlines() if "valid mappings" in x][0].split(",")[0]
    assert valid(r.stdout) == valid(r0.stdout) == "total %d valid mappings" % res["valid"]
    rec = CV.records(sam, {"chr1"})
    drop = {"c": [0, 0], "u": [0, 0]}
    for (_, qn), s in zip(rec, res["scores"][0]):
        drop[qn[0]][0] += 1
        drop[qn[0]][1] += s >= 3
    assert drop["u"][0] > 0.9 * n_u and drop["u"][1] == drop["u"][0], drop
    assert drop["c"][1] <= 0.005 * drop["c"][0], drop
    before, after = chh_ratio(open(t0).read()), chh_ratio(open(t).read())
    assert 0.08 < before < 0.14 and after < 0.015, (before, after)
