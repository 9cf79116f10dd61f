"""4-CpG epialleles on the device (the Epi pile-up kernels and the CpG rank index of bsx_meth.cu, `methratio
--epialleles`, `bsmap --methratio --meth-epialleles`) against the numpy restatement (oracle/epiallele_oracle.py),
randomised rounds on the generators of tests/meth_fuzz.py, and an end-to-end run in which epipolymorphism tells clonal
structure from disorder where PDR cannot."""
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
from test_epiallele_cpu import KATS, NAMES, SEQS, R16, sub
from test_methratio_cpu import MANIFEST, alignment_files, opts_kwargs
from test_mbias_cpu import oracle_files, sam_line
from test_pdr_cpu import kat_file

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import epiallele_oracle as EP  # noqa: E402

import bsmap_b200 as B
from bsmap_b200 import lib as BL

pytestmark = pytest.mark.gpu
BIN = os.path.dirname(BL.LIB_PATH)
METHRATIO, BSMAP = os.path.join(BIN, "methratio"), os.path.join(BIN, "bsmap")
IGNORE = (2, 1, 3, 2)
# name -> (PDR's K or None, conversion threshold or None, M-bias + exclusion, C/T SNP mode)
VARIANTS = {"epi": (None, None, False, None), "pdr": (4, None, False, None), "conv_mbias": (None, 2, True, None),
            "correct": (None, None, False, "correct"), "all": (2, 2, True, "skip")}


def add_all(mh, cols, batches=1):
    n = len(cols[0])
    cut = [n * k // batches for k in range(batches + 1)]
    for b, e in zip(cut, cut[1:]):
        if e > b:
            mh.add(*[c[b:e] for c in cols[:7]], read2=cols[7][b:e])


def make_meth(ix, opts, epi=True, min_cpg=None, threshold=None, mbias=False, ct_snp=None, ignore=None):
    mh = B.Meth(ix, opts)
    if epi:
        mh.enable_epialleles()
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


def same_epi(mh, names, res):
    assert mh.epialleles() == (res["spanning"], res["windows"])
    for k, n in enumerate(names):
        if n not in res["epi"]:
            continue
        pos, counts = mh.epiallele_counters(k)
        assert np.array_equal(pos, res["sites"][n]), n
        assert np.array_equal(counts, res["epi"][n]), n
        assert not counts[max(len(pos) - EP.CPGS + 1, 0):].any(), n      # rows whose window leaves the sequence


def same_as_oracle(mh, names, res, min_cpg=None, mbias=False, ct_snp=None, threshold=None):
    assert mh.valid() == res["valid"]
    same_epi(mh, names, res)
    for k, n in enumerate(names):
        m, dp = mh.counters(k)
        exp = res["counters"][n]
        assert np.array_equal(m, exp[0]) and np.array_equal(dp, exp[1]), n
        if min_cpg:
            c, d = mh.pdr_counters(k)
            assert np.array_equal(c, res["concordant"][n]) and np.array_equal(d, res["discordant"][n]), n
        if ct_snp:
            c, s = mh.ct_snp_counters(k)
            assert np.array_equal(c, exp[2]) and np.array_equal(s, exp[3]), n
    if min_cpg:
        assert mh.pdr() == (res["informative"], res["discordant_alignments"])
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
    """bsx_meth_add in one and in three batches (-r across them), in every variant: pattern counters, summary, counters,
    PDR, evidence, M-bias and conversion bins == oracle; and all but the patterns are those of the run without
    epialleles"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = opts_kwargs(ent["opts"])
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth")}
    bsp = not files[0].upper().endswith(".SAM")
    cols = api_arrays(files, d["gnames"])
    ix = B.Index.packed(d["gnames"], d["gseqs"])
    windows = 0
    for name, (k, threshold, mbias, ct_snp) in VARIANTS.items():
        if mbias and bsp:
            continue                                          # BSP records carry no read number
        ignore = IGNORE if mbias else None
        res = EP.epialleles(d["gnames"], d["gseqs"], files, min_cpg=k or 4, threshold=threshold or 0, ignore=ignore or (0, 0, 0, 0), **ckw)
        windows += res["windows"]
        for batches in (1, 3):
            mh = make_meth(ix, B.meth_opts(**kw), True, k, threshold, mbias, ct_snp, ignore)
            add_all(mh, cols, batches)
            same_as_oracle(mh, d["gnames"], res, k, mbias, ct_snp, threshold)
            plain = make_meth(ix, B.meth_opts(**kw), False, k, threshold, mbias, ct_snp, ignore)
            add_all(plain, cols, batches)
            with pytest.raises(B.BsxError, match="not enabled"):
                plain.epialleles()
            assert plain.valid() == mh.valid()
            for kk in range(len(d["gnames"])):
                assert all(np.array_equal(a, b) for a, b in zip(plain.counters(kk), mh.counters(kk))), name
                if k:
                    assert all(np.array_equal(a, b) for a, b in zip(plain.pdr_counters(kk), mh.pdr_counters(kk))), name
                if ct_snp:
                    assert all(np.array_equal(a, b) for a, b in zip(plain.ct_snp_counters(kk), mh.ct_snp_counters(kk))), name
            if k:
                assert plain.pdr() == mh.pdr()
            if mbias:
                assert all(np.array_equal(a, b) for a, b in zip(plain.mbias(), mh.mbias()))
            if threshold is not None:
                assert all(np.array_equal(a, b) for a, b in zip(plain.conversion(), mh.conversion()))
            mh.close(); plain.close()
    assert windows > 0
    ix.close()


@pytest.mark.parametrize("name", sorted(KATS))
def test_known_answers_on_the_device(tmp_path, name):
    """the hand-computed cases through bsx_meth_add, one batch per record, upper- and lower-case reference"""
    lines, kw, exp, spanning = KATS[name]
    sam = kat_file(tmp_path, lines)
    for seqs in (SEQS, [s.lower() for s in SEQS]):
        res = EP.epialleles(NAMES, seqs, [sam], **kw)
        assert res["spanning"] == spanning
        ix = B.Index.packed(NAMES, seqs)
        opts = B.meth_opts(trim_fillin=kw.get("trim_fillin", 2), rm_dup=kw.get("rm_dup", False), combine_cpg=kw.get("combine_cpg", False))
        mh = make_meth(ix, opts, True, None, kw.get("threshold"), mbias=True, ignore=kw.get("ignore"))
        add_all(mh, api_arrays([sam], NAMES), batches=len(lines))
        same_as_oracle(mh, NAMES, res, mbias=True, threshold=kw.get("threshold"))
        mh.close(); ix.close()


def test_file_through_the_api(tmp_path):
    """write_epialleles in every C/T SNP mode and at -m 1..4, with and without -g"""
    lines = [sam_line(0, "chrP", 1, R16, "++"), sam_line(16, "chrP", 1, sub(R16, 1, "T"), "-+"), sam_line(16, "chrP", 1, R16, "-+"),
             sam_line(0, "chrP", 5, "ACGTACGTACGTACGT", "++"), sam_line(0, "chrQ", 1, "CG" * 50, "++"), sam_line(0, "chrQ", 3, "TG" * 40, "++")]
    sam = kat_file(tmp_path, lines)
    for g in (False, True):
        res = EP.epialleles(NAMES, SEQS, [sam], combine_cpg=g)
        for mode in (None, "no-action", "skip", "correct"):
            for m in (1, 2, 4):
                ix = B.Index.packed(NAMES, SEQS)
                mh = make_meth(ix, B.meth_opts(min_depth=m, combine_cpg=g), ct_snp=mode)
                add_all(mh, api_arrays([sam], NAMES))
                txt = read_fd(lambda fd: mh.write_epialleles(SEQS, fd))
                assert txt == EP.epiallele_text(res, min_depth=m, ct_snp=mode), (g, mode, m)
                assert read_fd(lambda fd: mh.write_epialleles(SEQS, fd, chroms=[0, 1])) == EP.HEADER + "".join(
                    ln + "\n" for ln in txt.splitlines()[1:] if ln.startswith("chrQ"))
                mh.close(); ix.close()


def run_ok(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return r


CLI_KEYS = ["pe_sam.default", "pe_sam.r", "se_cfg2_bsp.default", "pe_bsp_r0.r", "se_cfg2_r0_uR.bam.default", "se_n1.t_5_g", "rrbs_se_A.z",
            "se_cfg5.m_3"]


@pytest.mark.parametrize("key", CLI_KEYS)
def test_methratio_cli(tmp_path, key):
    """methratio --epialleles F (SAM, BAM and BSP), with PDR, the C/T SNP modes and the conversion filter: the file and
    the stderr line == oracle; the table, M-bias report, PDR file and summary are byte-equal to the run without it"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    fa, _, _ = CS.write_inputs(case, str(tmp_path))
    files = alignment_files(case, str(tmp_path), bam=ent.get("bam", False))
    kw = opts_kwargs(ent["opts"])
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth")}
    ofiles = oracle_files(ent, case, str(tmp_path))
    sam = ofiles[0].upper().endswith(".SAM")
    t0, t, epi, mb0, mb, p0, p = (str(tmp_path / x) for x in ("t0", "t", "epi", "mb0", "mb", "p0", "p"))
    for extra in ([], ["--ct-snp", "skip"], ["--ct-snp", "correct", "--conversion-filter", "2"]):
        base = [METHRATIO, "-d", fa, "-q"] + ent["opts"] + extra
        if sam:
            base += ["--mbias-ignore", "1,2,0,3"]
        r0 = run_ok(base + ["-o", t0, "--pdr", p0] + (["--mbias", mb0] if sam else []) + files)
        r = run_ok(base + ["-o", t, "--pdr", p, "--epialleles", epi] + (["--mbias", mb] if sam else []) + files)
        assert r.stdout == r0.stdout and open(t, "rb").read() == open(t0, "rb").read() and open(p, "rb").read() == open(p0, "rb").read()
        if sam:
            assert open(mb, "rb").read() == open(mb0, "rb").read()
        mode = extra[1] if extra else None
        res = EP.epialleles(d["gnames"], d["gseqs"], ofiles, threshold=2 if "--conversion-filter" in extra else 0,
                            ignore=(1, 2, 0, 3) if sam else (0, 0, 0, 0), **ckw)
        exp = EP.epiallele_text(res, min_depth=kw.get("min_depth", 1), ct_snp=mode)
        assert open(epi).read() == exp, (extra, R.first_diff(open(epi, "rb").read(), exp.encode()))
        assert EP.stderr_line(res) in r.stderr.splitlines()
        assert [x for x in r.stderr.splitlines() if not x.startswith("epialleles:")] == r0.stderr.splitlines()


@pytest.mark.parametrize("name,ext", [("se_cfg2_r0_uR", "sam"), ("pe_sam", "sam"), ("se_cfg2_bsp", "bsp")])
def test_bsmap_cli(tmp_path, name, ext):
    """bsmap --methratio T --meth-epialleles F (in-process pile-up): == methratio on the alignment file the same run
    wrote, and == the oracle; the table, PDR file and summary are those of the run without --meth-epialleles"""
    case = CS.BY_NAME[name]
    d = case.data()
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / ("out." + ext))
    t0, t, p0, p, epi, t2, epi2 = (str(tmp_path / x) for x in ("t0", "t", "p0", "p", "epi", "t2", "epi2"))
    r0 = run_ok([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t0, "--meth-zero", "--meth-pdr", p0])
    r = run_ok([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t, "--meth-zero", "--meth-pdr", p, "--meth-epialleles", epi])
    summary = lambda out: [x for x in out.splitlines() if "valid mappings" in x]
    assert summary(r.stdout) == summary(r0.stdout) and open(t).read() == open(t0).read() and open(p).read() == open(p0).read()
    m = run_ok([METHRATIO, "-o", t2, "-d", fa, "-z", "--epialleles", epi2, o])
    assert open(epi).read() == open(epi2).read() and open(t).read() == open(t2).read()
    res = EP.epialleles(d["gnames"], d["gseqs"], [o])
    assert open(epi).read() == EP.epiallele_text(res)
    assert EP.stderr_line(res) in r.stderr.splitlines() and EP.stderr_line(res) in m.stderr.splitlines()
    assert res["windows"] > 0


def _map_in_process(case, max_batch, min_cpg=None, threshold=None, mbias=False, ignore=None, ct_snp=None):
    d = case.data()
    p = B.make_params(**case.param_kwargs())
    ix = B.Index(p, d["gnames"], d["gseqs"])
    mp = B.Mapper(ix, p, max_batch=max_batch, stride=160)
    mh = make_meth(ix, B.meth_opts(), True, min_cpg, threshold, mbias, ct_snp, ignore)
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
    """Mapper + attached Meth, many batches on both streams (Epi, and Epi + Pdr + Conv + M-bias + exclusion + Snp)"""
    case = CS.BY_NAME[name]
    files = alignment_files(case, str(tmp_path))          # the golden text == what these records format to
    bsp = not files[0].upper().endswith(".SAM")
    for k, threshold, mbias, ct_snp in ((None, None, False, None), (2, 3, not bsp, "correct")):
        ignore = IGNORE if mbias else None
        d, ix, mp, mh = _map_in_process(case, 256, k, threshold, mbias, ignore, ct_snp)
        res = EP.epialleles(d["gnames"], d["gseqs"], files, min_cpg=k or 4, threshold=threshold or 0, ignore=ignore or (0, 0, 0, 0))
        same_as_oracle(mh, d["gnames"], res, k, mbias, ct_snp, threshold)
        mh.close(); mp.close(); ix.close()


@pytest.mark.parametrize("name", ["se_n1", "pe_sam"])
def test_batch_size_invariance(name):
    """64 and 1 M alignments per batch give the same pattern counters and summary"""
    res = []
    for mb in (64, 1 << 20):
        d, ix, mp, mh = _map_in_process(CS.BY_NAME[name], max_batch=mb, min_cpg=2, threshold=3, mbias=True, ignore=(1, 2, 3, 4))
        res.append((mh.epialleles(), [mh.epiallele_counters(k) for k in range(len(d["gnames"]))]))
        mh.close(); mp.close(); ix.close()
    (s0, k0), (s1, k1) = res
    assert s0 == s1 and s0[1] > 0
    for a, b in zip(k0, k1):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_misuse_is_refused(tmp_path):
    ix = B.Index.packed(["c"], [b"ACGT" * 100])
    mh = B.Meth(ix, B.meth_opts())
    for call in (mh.epialleles, lambda: mh.epiallele_counters(0), lambda: read_fd(lambda fd: mh.write_epialleles([b"ACGT" * 100], fd))):
        with pytest.raises(B.BsxError, match="not enabled"):
            call()
    mh.enable_epialleles()
    with pytest.raises(B.BsxError, match="already enabled"):
        mh.enable_epialleles()
    with pytest.raises(B.BsxError, match="has 3 bases"):
        read_fd(lambda fd: mh.write_epialleles([b"ACG"], fd))
    mh.close()
    mh = B.Meth(ix, B.meth_opts())
    mh.add([b"ACGTACGT"], [0], [0], [0], [0], [0], [4])
    with pytest.raises(B.BsxError, match="error 1:.*already piled up"):
        mh.enable_epialleles()
    mh.close(); ix.close()
    case = CS.BY_NAME["se_n1"]
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / "o.sam")
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--meth-epialleles", str(tmp_path / "e")], capture_output=True, text=True)
    assert r.returncode == 2 and "--methratio" in r.stderr
    assert not os.path.exists(str(tmp_path / "e"))


# ---- randomised rounds on the fuzz generators ------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [3, 4, 5])
def test_fuzz_rounds(tmp_path, seed):
    """generated references, records and options (meth_fuzz), random batch cuts: every counter, the pattern counters,
    the summary, the epiallele file and the unchanged table == the oracle"""
    rng = np.random.default_rng(seed)
    for rnd in range(6):
        names, seqs = MF.make_reference(rng)
        sam = rng.random() < 0.7
        o = MF.draw_options(rng, names, seqs, sam)
        recs = MF.make_records(rng, names, seqs, int(rng.choice([60, 400, 2000])), rm_dup=o["rm_dup"])
        path = str(tmp_path / ("a%d_%d.%s" % (seed, rnd, "sam" if sam else "bsp")))
        open(path, "w").write(MF.sam_text(recs, names, seqs) if sam else MF.bsp_text(recs))
        e = MF.expected(names, seqs, [path], o)
        res = EP.epialleles(names, seqs, [path], threshold=o["conv"] or 0, chroms=o["chroms"], unique=o["unique"], pair=o["pair"],
                            trim_fillin=o["trim_fillin"], combine_cpg=o["combine_cpg"], rm_dup=o["rm_dup"], ignore=o["ignore"] or (0, 0, 0, 0))
        sel = [not o["chroms"] or n in o["chroms"] for n in names]
        cols = api_arrays([path], names) or [[] for _ in range(8)]
        keep = [i for i, c in enumerate(cols[1]) if sel[c]]
        cols = [[c[i] for i in keep] for c in cols]
        cuts = MF.batch_cuts(rng, len(cols[0]))
        ix = B.Index.packed(names, seqs)
        mh = MF.new_meth(B, ix, o)
        mh.enable_epialleles()
        for b, x in zip(cuts, cuts[1:]):
            mh.add(*[c[b:x] for c in cols[:7]], read2=cols[7][b:x])
        desc = (seed, rnd, {x: v for x, v in o.items() if v and x != "regions"})
        assert MF.compare_counters(mh, names, o, e["res"]) is None, desc
        same_epi(mh, names, res)
        assert read_fd(lambda fd: mh.write_epialleles(seqs, fd, chroms=sel)) == EP.epiallele_text(res, o["min_depth"], o["ct_snp"]), desc
        assert read_fd(lambda fd: mh.write(seqs, fd, chroms=sel)) == e["table"], desc
        mh.close(); ix.close()


# ---- end to end: clonal structure against disorder -------------------------------------------------------------------
GLEN, RLEN, NREADS = 200_000, 100, 120_000
REGIONS = {"A": (20_000, 26_000), "B": (60_000, 66_000), "C": (100_000, 106_000), "D": (140_000, 146_000)}


def _simulate(rng, genome: bytes):
    """directional reads from both strands at 60x; a fragment that overlaps a region takes the region's rule for all its
    CpGs: A all methylated or all unmethylated, B each CpG methylated with p = 1/2, C one of two clones (CpG site of rank
    r methylated when r mod 4 < 2, or its complement), D all methylated; elsewhere p = 0.8.  Non-CpG C converted at
    99.5 %"""
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    g = np.frombuffer(genome, dtype=np.uint8)
    C, G, T, A = (ord(x) for x in "CGTA")
    cpg_c = np.zeros(len(g), dtype=bool)
    cpg_c[:-1] = (g[:-1] == C) & (g[1:] == G)                 # Watson C of a CpG
    cpg_g = np.zeros(len(g), dtype=bool)
    cpg_g[1:] = cpg_c[:-1]                                    # Crick C of a CpG (the Watson G)
    rank = np.cumsum(cpg_c) - 1                               # at a Watson C: its site's rank
    clone_c = np.zeros(len(g), dtype=bool)
    clone_c[cpg_c] = (rank[cpg_c] % 4) < 2
    clone_g = np.zeros(len(g), dtype=bool)
    clone_g[1:] = clone_c[:-1]
    reads = []
    for _ in range(NREADS):
        s = int(rng.integers(0, len(g) - RLEN))
        sl = slice(s, s + RLEN)
        crick = rng.random() < 0.5
        c_here = (g[sl] == G) if crick else (g[sl] == C)
        cpg = (cpg_g if crick else cpg_c)[sl]
        region = next((k for k, (b, e) in REGIONS.items() if s < e and s + RLEN > b), None)
        if region == "A":
            m_cpg = np.full(RLEN, rng.random() < 0.5)
        elif region == "B":
            m_cpg = rng.random(RLEN) < 0.5
        elif region == "C":
            m_cpg = (clone_g if crick else clone_c)[sl] ^ (rng.random() < 0.5)
        elif region == "D":
            m_cpg = np.ones(RLEN, dtype=bool)
        else:
            m_cpg = rng.random(RLEN) < 0.8
        meth = np.where(cpg, m_cpg, rng.random(RLEN) >= 0.995)
        w = g[sl].copy()
        w[c_here & ~meth] = A if crick else T                 # converted C on the read's strand, seen on Watson
        read = w.tobytes()
        reads.append(read.translate(comp)[::-1] if crick else read)
    return reads


def test_epipolymorphism_separates_clones_from_disorder(tmp_path):
    """four planted 6 kb regions.  Over windows with >= 10 reads: the bimodal (A) and two-clone (C) regions have two
    patterns at about 1/2 each, so EPM near 0.5 and entropy near 0.25; the disordered one (B) spreads over all 16, EPM
    and entropy >= 0.85; the methylated one (D) has EPM <= 0.1.  PDR is >= 0.8 in both B and C: it cannot tell them
    apart, EPM can"""
    from bsmap_b200 import synth
    gen = synth.make_genome(17, [GLEN])
    gb = gen[0].numpy().tobytes()
    reads = _simulate(np.random.default_rng(5), gb)
    fa, fq, sam, bed = (str(tmp_path / x) for x in ("g.fa", "r.fq", "o.sam", "r.bed"))
    synth.write_fasta(fa, gen, names=["chr1"])
    synth.write_fastq(fq, np.frombuffer(b"".join(reads), dtype=np.uint8).reshape(len(reads), RLEN), ["r%d" % i for i in range(len(reads))])
    open(bed, "w").write("".join("chr1\t%d\t%d\n" % REGIONS[k] for k in "ABCD"))
    t, pdr, rr, epi = (str(tmp_path / x) for x in ("t", "pdr", "rr", "epi"))
    r = run_ok([BSMAP, "-a", fq, "-d", fa, "-o", sam, "-v", "5", "--methratio", t, "--meth-pdr", pdr, "--meth-region-report", rr,
                "--meth-regions", bed, "--meth-epialleles", epi])
    rows = [ln.split("\t") for ln in open(rr).read().splitlines()[1:] if ln.split("\t")[3] == "CpG"]
    pdrs = {k: int(x[10]) / (int(x[9]) + int(x[10])) for k, x in zip("ABCD", rows)}
    lines = [ln.split("\t") for ln in open(epi).read().splitlines()[1:]]
    stats = {}
    for k, (b, e) in REGIONS.items():
        w = [(float(x[5]), float(x[6])) for x in lines if b <= int(x[1]) - 1 and int(x[2]) <= e and int(x[3]) >= 10]
        assert len(w) > 100, (k, len(w))
        stats[k] = tuple(float(np.mean(v)) for v in zip(*w))  # (entropy, EPM)
    print("mean (entropy, EPM) over windows with >= 10 reads:", stats, "PDR:", pdrs)
    # with N reads, a window of two patterns at 1/2 has E[EPM] = (1 - 1/N) / 2 and entropy just below 0.25; a read
    # crossing a region edge, a non-converted C and a mismapped read add a third pattern now and then
    for k in "AC":
        ent, epm = stats[k]
        assert abs(epm - 0.5) < 0.06 and abs(ent - 0.25) < 0.04, (k, stats)
    assert stats["B"][0] >= 0.85 and stats["B"][1] >= 0.85, stats
    assert stats["D"][1] <= 0.1, stats
    assert pdrs["B"] >= 0.8 and pdrs["C"] >= 0.8, pdrs
    res = EP.epialleles(["chr1"], [gb], [sam])
    assert open(epi).read() == EP.epiallele_text(res)
    assert EP.stderr_line(res) in r.stderr.splitlines()
