"""Read-level CpG concordance (PDR) on the device (the Pdr pile-up kernels of bsx_meth.cu, `methratio --pdr`,
`bsmap --methratio --meth-pdr`) against the numpy restatement (oracle/pdr_oracle.py), randomised rounds on the
generators of tests/meth_fuzz.py, and an end-to-end run that tells bimodal from disordered methylation."""
from __future__ import annotations

import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import cases as CS
import meth_fuzz as MF
import runners as R
from meth_inputs import api_arrays
from test_methratio_cpu import MANIFEST, alignment_files, opts_kwargs
from test_mbias_cpu import oracle_files
from test_pdr_cpu import KATS, NAMES, SEQS, kat_file

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import pdr_oracle as PD  # noqa: E402
import region_oracle as RG  # noqa: E402

import bsmap_b200 as B
from bsmap_b200 import lib as BL

pytestmark = pytest.mark.gpu
BIN = os.path.dirname(BL.LIB_PATH)
METHRATIO, BSMAP = os.path.join(BIN, "methratio"), os.path.join(BIN, "bsmap")
IGNORE = (2, 1, 3, 2)
# name -> (min_cpg, conversion threshold or None, M-bias + exclusion, C/T SNP mode)
VARIANTS = {"pdr": (4, None, False, None), "k2": (2, None, False, None), "conv_mbias": (3, 2, True, None),
            "correct": (4, None, False, "correct"), "all": (2, 2, True, "skip")}


def add_all(mh, cols, batches=1):
    n = len(cols[0])
    cut = [n * k // batches for k in range(batches + 1)]
    for b, e in zip(cut, cut[1:]):
        if e > b:
            mh.add(*[c[b:e] for c in cols[:7]], read2=cols[7][b:e])


def make_meth(ix, opts, min_cpg=4, threshold=None, mbias=False, ct_snp=None, ignore=None):
    mh = B.Meth(ix, opts)
    if min_cpg:
        mh.enable_pdr(min_cpg)
    if threshold is not None:
        mh.enable_conversion_filter(threshold)
    if mbias:
        mh.enable_mbias()
    if ignore:
        mh.set_ignore(*ignore)
    if ct_snp:
        mh.enable_ct_snp(ct_snp)
    return mh


def read_fd(fn):
    with tempfile.TemporaryFile() as f:
        fn(f.fileno())
        f.seek(0)
        return f.read().decode()


def same_as_oracle(mh, names, res, mbias=False, ct_snp=None, threshold=None):
    assert mh.valid() == res["valid"]
    assert mh.pdr() == (res["informative"], res["discordant_alignments"])
    for k, n in enumerate(names):
        m, dp = mh.counters(k)
        exp = res["counters"][n]
        assert np.array_equal(m, exp[0]) and np.array_equal(dp, exp[1]), n
        c, d = mh.pdr_counters(k)
        assert np.array_equal(c, res["concordant"][n]) and np.array_equal(d, res["discordant"][n]), n
        if ct_snp:
            c, s = mh.ct_snp_counters(k)
            assert np.array_equal(c, exp[2]) and np.array_equal(s, exp[3]), n
    if mbias:
        hist, over = mh.mbias()
        assert np.array_equal(hist.astype(np.int64), res["mbias"]) and over == res["mbias_overflow"]
    if threshold is not None:
        bins, dropped = mh.conversion()
        assert np.array_equal(bins.astype(np.int64), res["bins"]) and dropped == res["dropped"]


API_KEYS = ["pe_sam.p_u", "pe_sam.r", "pe_readthrough.p_g", "se_n1.r_t_0", "se_n1.t_5_g", "rrbs_pe.t_0", "se_cfg1.g_z",
            "se_cfg2_bsp.r_u", "pe_bsp_r0.r", "pe_sam.bam.r", "rrbs_se_A.bam.r_u"]


@pytest.mark.parametrize("key", API_KEYS)
def test_meth_add_equals_the_oracle(tmp_path, key):
    """bsx_meth_add in one and in three batches, in every variant: counters, concordance, summary, evidence, M-bias and
    conversion bins == oracle; and the counters, M-bias and bins are those of the same run without PDR"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = opts_kwargs(ent["opts"])
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth")}
    bsp = not files[0].upper().endswith(".SAM")
    cols = api_arrays(files, d["gnames"])
    ix = B.Index.packed(d["gnames"], d["gseqs"])
    informative = 0
    for name, (k, threshold, mbias, ct_snp) in VARIANTS.items():
        if mbias and bsp:
            continue                                          # BSP records carry no read number
        ignore = IGNORE if mbias else None
        res = PD.pdr(d["gnames"], d["gseqs"], files, min_cpg=k, threshold=threshold or 0, ignore=ignore or (0, 0, 0, 0), **ckw)
        informative += res["informative"]
        for batches in (1, 3):
            mh = make_meth(ix, B.meth_opts(**kw), k, threshold, mbias, ct_snp, ignore)
            add_all(mh, cols, batches)
            same_as_oracle(mh, d["gnames"], res, mbias, ct_snp, threshold)
            mh.close()
        plain = make_meth(ix, B.meth_opts(**kw), 0, threshold, mbias, ct_snp, ignore)
        add_all(plain, cols, 3)
        with pytest.raises(B.BsxError, match="not enabled"):
            plain.pdr()
        for kk, n in enumerate(d["gnames"]):
            assert all(np.array_equal(a, b) for a, b in zip(plain.counters(kk), res["counters"][n][:2])), (name, n)
        if mbias:
            assert np.array_equal(plain.mbias()[0].astype(np.int64), res["mbias"])
        if threshold is not None:
            assert np.array_equal(plain.conversion()[0].astype(np.int64), res["bins"])
        plain.close()
    assert informative > 0
    ix.close()


@pytest.mark.parametrize("name", sorted(k for k in KATS if KATS[k][1].get("sam_rules") is not False))   # SAM text takes SAM rules
def test_known_answers_on_the_device(tmp_path, name):
    """the hand-computed cases through bsx_meth_add, one batch per record, upper- and lower-case reference"""
    lines, kw, exp, informative, n_disc = KATS[name]
    sam = kat_file(tmp_path, lines)
    for seqs in (SEQS, [s.lower() for s in SEQS]):
        res = PD.pdr(NAMES, seqs, [sam], **kw)
        assert res["informative"] == informative and res["discordant_alignments"] == n_disc
        ix = B.Index.packed(NAMES, seqs)
        opts = B.meth_opts(trim_fillin=kw.get("trim_fillin", 2), rm_dup=kw.get("rm_dup", False), combine_cpg=kw.get("combine_cpg", False))
        mh = make_meth(ix, opts, kw.get("min_cpg", 4), kw.get("threshold"), mbias=True, ignore=kw.get("ignore"))
        add_all(mh, api_arrays([sam], NAMES), batches=len(lines))
        same_as_oracle(mh, NAMES, res, mbias=True, threshold=kw.get("threshold"))
        mh.close(); ix.close()


def test_files_and_regions_through_the_api(tmp_path):
    """write_pdr, regions_pdr and write_regions on the snp / -m cases of the CPU tests"""
    from test_pdr_cpu import snp_lines
    sam = kat_file(tmp_path, snp_lines())
    regs = [("chrP", s, e) for s in range(0, 20, 3) for e in (s, s + 4, s + 11)] + [("chrQ", 0, 600)]
    ci, st, en = [NAMES.index(c) for c, _, _ in regs], [s for _, s, _ in regs], [e for _, _, e in regs]
    for mode in (None, "skip", "correct"):
        for m in (1, 2):
            res = PD.pdr(NAMES, SEQS, [sam])
            ix = B.Index.packed(NAMES, SEQS)
            mh = make_meth(ix, B.meth_opts(min_depth=m), ct_snp=mode)
            add_all(mh, api_arrays([sam], NAMES))
            assert read_fd(lambda fd: mh.write_pdr(SEQS, fd)) == PD.pdr_text(res, min_depth=m, ct_snp=mode)
            sums, pd = mh.regions_pdr(ci, st, en)
            assert np.array_equal(pd.astype(np.int64), PD.region_pdr(res, regs, min_depth=m, ct_snp=mode))
            assert np.array_equal(sums.astype(np.int64), RG.regions(res["counters"], res["ref"], regs, min_depth=m, ct_snp=mode))
            assert np.array_equal(mh.regions(ci, st, en), sums)
            assert read_fd(lambda fd: mh.write_regions(fd, ci, st, en)) == PD.region_text(res, regs, min_depth=m, ct_snp=mode)
            mh.close(); ix.close()


def run_ok(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return r


CLI_KEYS = ["pe_sam.default", "pe_sam.r", "se_cfg2_bsp.default", "pe_bsp_r0.r", "se_cfg2_r0_uR.bam.default", "se_n1.t_5_g", "rrbs_se_A.z",
            "se_cfg5.m_3"]


@pytest.mark.parametrize("key", CLI_KEYS)
def test_methratio_cli(tmp_path, key):
    """methratio --pdr F [--pdr-min-cpg K] with --region-report (SAM, BAM and BSP): PDR file, region report and stderr
    line == oracle; the table, M-bias report and summary are byte-equal to the run without --pdr"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    fa, _, _ = CS.write_inputs(case, str(tmp_path))
    files = alignment_files(case, str(tmp_path), bam=ent.get("bam", False))
    kw = opts_kwargs(ent["opts"])
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth")}
    ofiles = oracle_files(ent, case, str(tmp_path))
    sam = ofiles[0].upper().endswith(".SAM")
    bed = tmp_path / "r.bed"
    regs = [(n, s, s + w) for n, g in zip(d["gnames"], d["gseqs"]) for s, w in ((0, 500), (len(g) // 3, 2000), (len(g) - 100, 300))
            if not kw.get("chroms") or n in kw["chroms"]]
    bed.write_text("".join("%s\t%d\t%d\n" % r for r in regs))
    t0, t, pdr, rr0, rr, mb0, mb = (str(tmp_path / x) for x in ("t0", "t", "pdr", "rr0", "rr", "mb0", "mb"))
    for k, extra in ((4, []), (2, ["--pdr-min-cpg=2", "--ct-snp", "skip"]), (1, ["--pdr-min-cpg=1", "--conversion-filter", "2"])):
        base = [METHRATIO, "-d", fa, "-q", "--regions", str(bed)] + ent["opts"] + [x for x in extra if not x.startswith("--pdr")]
        if sam:
            base += ["--mbias-ignore", "1,2,0,3"]
        r0 = run_ok(base + ["-o", t0, "--region-report", rr0] + (["--mbias", mb0] if sam else []) + files)
        r = run_ok(base + ["-o", t, "--region-report", rr, "--pdr", pdr] + [x for x in extra if x.startswith("--pdr")] +
                   (["--mbias", mb] if sam else []) + files)
        assert r.stdout == r0.stdout and open(t, "rb").read() == open(t0, "rb").read()
        if sam:
            assert open(mb, "rb").read() == open(mb0, "rb").read()
        mode = "skip" if "skip" in extra else None
        res = PD.pdr(d["gnames"], d["gseqs"], ofiles, min_cpg=k, threshold=2 if "--conversion-filter" in extra else 0,
                     ignore=(1, 2, 0, 3) if sam else (0, 0, 0, 0), **ckw)
        assert open(pdr).read() == PD.pdr_text(res, min_depth=kw.get("min_depth", 1), ct_snp=mode), (k, R.first_diff(open(pdr, "rb").read(), PD.pdr_text(res, min_depth=kw.get("min_depth", 1), ct_snp=mode).encode()))
        assert open(rr).read() == PD.region_text(res, regs, combine_cpg=kw.get("combine_cpg", False), min_depth=kw.get("min_depth", 1), ct_snp=mode)
        assert [ln.split("\t")[:9] for ln in open(rr).read().splitlines()[1:]] == [ln.split("\t") for ln in open(rr0).read().splitlines()[1:]]
        assert PD.stderr_line(res, k) in r.stderr.splitlines()


@pytest.mark.parametrize("name,ext", [("se_cfg2_r0_uR", "sam"), ("pe_sam", "sam"), ("se_cfg2_bsp", "bsp")])
def test_bsmap_cli(tmp_path, name, ext):
    """bsmap --methratio T --meth-pdr F --meth-region-report R (in-process pile-up): == methratio on the alignment file
    the same run wrote, and == the oracle; the table and summary are those of the run without --meth-pdr"""
    case = CS.BY_NAME[name]
    d = case.data()
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / ("out." + ext))
    t0, t, pdr, rr, t2, pdr2, rr2 = (str(tmp_path / x) for x in ("t0", "t", "pdr", "rr", "t2", "pdr2", "rr2"))
    r0 = run_ok([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t0, "--meth-zero", "--meth-tiles", "5000", "--meth-region-report", rr])
    rr0 = open(rr).read()
    r = run_ok([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t, "--meth-zero", "--meth-pdr", pdr, "--meth-pdr-min-cpg", "3",
                                                   "--meth-tiles", "5000", "--meth-region-report", rr])
    summary = lambda out: [x for x in out.splitlines() if "valid mappings" in x]
    assert summary(r.stdout) == summary(r0.stdout) and open(t).read() == open(t0).read()
    assert [ln.split("\t")[:9] for ln in open(rr).read().splitlines()[1:]] == [ln.split("\t") for ln in rr0.splitlines()[1:]]
    m = run_ok([METHRATIO, "-o", t2, "-d", fa, "-z", "--pdr", pdr2, "--pdr-min-cpg", "3", "--tiles", "5000", "--region-report", rr2, o])
    assert open(pdr).read() == open(pdr2).read() and open(rr).read() == open(rr2).read() and open(t).read() == open(t2).read()
    res = PD.pdr(d["gnames"], d["gseqs"], [o], min_cpg=3)
    assert open(pdr).read() == PD.pdr_text(res)
    assert PD.stderr_line(res, 3) in r.stderr.splitlines() and PD.stderr_line(res, 3) in m.stderr.splitlines()
    assert res["informative"] > 0


def _map_in_process(case, max_batch, min_cpg=4, threshold=None, mbias=False, ignore=None, ct_snp=None):
    d = case.data()
    p = B.make_params(**case.param_kwargs())
    ix = B.Index(p, d["gnames"], d["gseqs"])
    mp = B.Mapper(ix, p, max_batch=max_batch, stride=160)
    mh = make_meth(ix, B.meth_opts(), min_cpg, threshold, mbias, ct_snp, ignore)
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
    """Mapper + attached Meth, many batches on both streams (Pdr, and Pdr + Conv + M-bias + exclusion + Snp)"""
    case = CS.BY_NAME[name]
    files = alignment_files(case, str(tmp_path))          # the golden text == what these records format to
    bsp = not files[0].upper().endswith(".SAM")
    for k, threshold, mbias, ct_snp in ((4, None, False, None), (2, 3, not bsp, "correct")):
        ignore = IGNORE if mbias else None
        d, ix, mp, mh = _map_in_process(case, 256, k, threshold, mbias, ignore, ct_snp)
        res = PD.pdr(d["gnames"], d["gseqs"], files, min_cpg=k, threshold=threshold or 0, ignore=ignore or (0, 0, 0, 0))
        same_as_oracle(mh, d["gnames"], res, mbias, ct_snp, threshold)
        mh.close(); mp.close(); ix.close()


@pytest.mark.parametrize("name", ["se_n1", "pe_sam"])
def test_batch_size_invariance(name):
    """64 and 1 M alignments per batch give the same concordance counters and summary"""
    res = []
    for mb in (64, 1 << 20):
        d, ix, mp, mh = _map_in_process(CS.BY_NAME[name], max_batch=mb, min_cpg=2, threshold=3, mbias=True, ignore=(1, 2, 3, 4))
        res.append((mh.pdr(), [mh.pdr_counters(k) for k in range(len(d["gnames"]))]))
        mh.close(); mp.close(); ix.close()
    (s0, k0), (s1, k1) = res
    assert s0 == s1 and s0[0] > 0
    for a, b in zip(k0, k1):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_misuse_is_refused(tmp_path):
    ix = B.Index.packed(["c"], [b"ACGT" * 100])
    mh = B.Meth(ix, B.meth_opts())
    for bad in (0, -1, 256):
        with pytest.raises(B.BsxError, match="1..255"):
            mh.enable_pdr(bad)
    with pytest.raises(B.BsxError, match="not enabled"):
        mh.pdr()
    with pytest.raises(B.BsxError, match="not enabled"):
        mh.pdr_counters(0)
    with pytest.raises(B.BsxError, match="not enabled"):
        mh.regions_pdr([0], [0], [10])
    mh.add([b"ACGTACGT"], [0], [0], [0], [0], [0], [4])
    with pytest.raises(B.BsxError, match="error 1:.*already piled up"):
        mh.enable_pdr(4)
    mh.close(); ix.close()
    case = CS.BY_NAME["se_n1"]
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o, t = str(tmp_path / "o.sam"), str(tmp_path / "t")
    run_ok([BSMAP] + case.cli(a, b, fa, o))
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--meth-pdr", str(tmp_path / "p")], capture_output=True, text=True)
    assert r.returncode == 2 and "--methratio" in r.stderr
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t, "--meth-pdr-min-cpg", "3"], capture_output=True, text=True)
    assert r.returncode == 2 and "--meth-pdr" in r.stderr
    r = subprocess.run([METHRATIO, "-o", t, "-d", fa, "--pdr-min-cpg", "3", o], capture_output=True, text=True)
    assert r.returncode == 2 and "--pdr" in r.stderr
    for bad in ("x", "3.5", "0", "256", "-1"):
        r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t, "--meth-pdr", str(tmp_path / "p"), "--meth-pdr-min-cpg", bad],
                           capture_output=True, text=True)
        assert r.returncode == 2 and "--meth-pdr-min-cpg" in r.stderr, bad
        r = subprocess.run([METHRATIO, "-o", t, "-d", fa, "--pdr", str(tmp_path / "p"), "--pdr-min-cpg", bad, o], capture_output=True, text=True)
        assert r.returncode == 2 and "--pdr-min-cpg" in r.stderr, bad


# ---- randomised rounds on the fuzz generators ------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [3, 4, 5])
def test_fuzz_rounds(tmp_path, seed):
    """generated references, records and options (meth_fuzz), K drawn from 1..6, random batch cuts: every counter,
    the summary, the PDR file, the region report and the unchanged table == the oracle"""
    rng = np.random.default_rng(seed)
    for rnd in range(6):
        names, seqs = MF.make_reference(rng)
        sam = rng.random() < 0.7
        o = MF.draw_options(rng, names, seqs, sam)
        k = int(rng.integers(1, 7))
        recs = MF.make_records(rng, names, seqs, int(rng.choice([60, 400, 2000])), rm_dup=o["rm_dup"])
        path = str(tmp_path / ("a%d_%d.%s" % (seed, rnd, "sam" if sam else "bsp")))
        open(path, "w").write(MF.sam_text(recs, names, seqs) if sam else MF.bsp_text(recs))
        e = MF.expected(names, seqs, [path], o)
        res = PD.pdr(names, seqs, [path], min_cpg=k, threshold=o["conv"] or 0, chroms=o["chroms"], unique=o["unique"], pair=o["pair"],
                     trim_fillin=o["trim_fillin"], combine_cpg=o["combine_cpg"], rm_dup=o["rm_dup"], ignore=o["ignore"] or (0, 0, 0, 0))
        sel = [not o["chroms"] or n in o["chroms"] for n in names]
        cols = api_arrays([path], names) or [[] for _ in range(8)]
        keep = [i for i, c in enumerate(cols[1]) if sel[c]]
        cols = [[c[i] for i in keep] for c in cols]
        cuts = MF.batch_cuts(rng, len(cols[0]))
        ix = B.Index.packed(names, seqs)
        mh = MF.new_meth(B, ix, o)
        mh.enable_pdr(k)
        for b, x in zip(cuts, cuts[1:]):
            mh.add(*[c[b:x] for c in cols[:7]], read2=cols[7][b:x])
        desc = (seed, rnd, k, {x: v for x, v in o.items() if v and x != "regions"})
        assert MF.compare_counters(mh, names, o, e["res"]) is None, desc
        assert mh.pdr() == (res["informative"], res["discordant_alignments"]), desc
        for kk, n in enumerate(names):
            if sel[kk]:
                c, dd = mh.pdr_counters(kk)
                assert np.array_equal(c, res["concordant"][n]) and np.array_equal(dd, res["discordant"][n]), desc
        assert read_fd(lambda fd: mh.write_pdr(seqs, fd, chroms=sel)) == PD.pdr_text(res, o["min_depth"], o["ct_snp"]), desc
        regs = MF.region_list(o, names, seqs)
        if regs is not None:
            idx = {x: i for i, x in enumerate(names)}
            ci, st, en = [idx[c] for c, _, _ in regs], [s for _, s, _ in regs], [x for _, _, x in regs]
            exp = PD.region_text(res, regs, o["combine_cpg"], o["min_depth"], o["ct_snp"])
            assert read_fd(lambda fd: mh.write_regions(fd, ci, st, en)) == exp, desc
        assert read_fd(lambda fd: mh.write(seqs, fd, chroms=sel)) == e["table"], desc
        mh.close(); ix.close()


# ---- end to end: bimodal against disordered methylation ------------------------------------------------------------
GLEN, RLEN, NREADS = 200_000, 100, 60_000
REG_A, REG_B = (40_000, 44_000), (120_000, 124_000)


def _simulate(rng, genome: bytes):
    """directional reads from both strands: the CpGs of a fragment that overlaps A are all methylated or all unmethylated,
    those of one that overlaps B each methylated with p = 1/2, elsewhere with p = 0.8; non-CpG C converted at 99.5 %"""
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    g = np.frombuffer(genome, dtype=np.uint8)
    C, G, T, A = (ord(x) for x in "CGTA")
    cpg_c = np.zeros(len(g), dtype=bool)
    cpg_c[:-1] = (g[:-1] == C) & (g[1:] == G)                 # Watson C of a CpG
    cpg_g = np.zeros(len(g), dtype=bool)
    cpg_g[1:] = cpg_c[:-1]                                    # Crick C of a CpG (the Watson G)
    reads = []
    for _ in range(NREADS):
        s = int(rng.integers(0, len(g) - RLEN))
        sl = slice(s, s + RLEN)
        crick = rng.random() < 0.5
        c_here = (g[sl] == G) if crick else (g[sl] == C)
        cpg = (cpg_g if crick else cpg_c)[sl]
        overlaps = lambda reg: s < reg[1] and s + RLEN > reg[0]
        p_meth = (1.0 if rng.random() < 0.5 else 0.0) if overlaps(REG_A) else (0.5 if overlaps(REG_B) else 0.8)
        meth = np.where(cpg, rng.random(RLEN) < p_meth, rng.random(RLEN) >= 0.995)
        w = g[sl].copy()
        w[c_here & ~meth] = A if crick else T                 # converted C on the read's strand, seen on Watson
        read = w.tobytes()
        reads.append(read.translate(comp)[::-1] if crick else read)
    return reads


def test_bimodal_and_disordered_regions_end_to_end(tmp_path):
    """two planted 4 kb regions at a CpG level of 0.5: A bimodal (fragments fully methylated or fully unmethylated), B
    disordered (each CpG at random).  The region report gives both a level near 0.5, and PDR separates them: near 0
    in A (non-conversion and mismapping only), at least 0.8 in B (1 - 2 / 2^n for n CpG calls)"""
    import torch
    from bsmap_b200 import synth
    gen = synth.make_genome(17, [GLEN])
    gb = gen[0].numpy().tobytes()
    reads = _simulate(np.random.default_rng(5), gb)
    fa, fq, sam, bed = (str(tmp_path / x) for x in ("g.fa", "r.fq", "o.sam", "r.bed"))
    synth.write_fasta(fa, gen, names=["chr1"])
    synth.write_fastq(fq, np.frombuffer(b"".join(reads), dtype=np.uint8).reshape(len(reads), RLEN), ["r%d" % i for i in range(len(reads))])
    open(bed, "w").write("chr1\t%d\t%d\nchr1\t%d\t%d\n" % (REG_A + REG_B))
    t, pdr, rr = (str(tmp_path / x) for x in ("t", "pdr", "rr"))
    r = run_ok([BSMAP, "-a", fq, "-d", fa, "-o", sam, "-v", "5", "--methratio", t, "--meth-pdr", pdr, "--meth-region-report", rr,
                "--meth-regions", bed])
    rows = [ln.split("\t") for ln in open(rr).read().splitlines()[1:] if ln.split("\t")[3] == "CpG"]
    (la, ca, da), (lb, cb, db) = ((float(x[8]), int(x[9]), int(x[10])) for x in rows)
    # A's calls come in blocks of one fragment: the binomial tolerance counts fragments (about 1,200 per region at 30x),
    # not calls, so 4 standard deviations of 0.5 over 1,200 draws
    for level in (la, lb):
        assert abs(level - 0.5) < 4 * (0.25 / 1200) ** 0.5, (la, lb)
    assert ca + da > 2000 and cb + db > 2000
    pdr_a, pdr_b = da / (ca + da), db / (cb + db)
    assert pdr_a <= 0.05 and pdr_b >= 0.8, (pdr_a, pdr_b)
    res = PD.pdr(["chr1"], [gb], [sam])
    assert open(pdr).read() == PD.pdr_text(res)
    assert PD.stderr_line(res, 4) in r.stderr.splitlines()
