"""Methylation haplotype load on the device (the run counters of the Epi pile-up walk, meth_mhl_region_kernel, `methratio
--mhl`, `bsmap --methratio --meth-mhl`) against the numpy restatement (oracle/mhl_oracle.py), randomised rounds on the
generators of tests/meth_fuzz.py, and an end-to-end run in which MHL tells methylation on whole molecules from
scattered methylation at the same mean level."""
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
from test_mhl_cpu import KATS, NAMES, SEQS
from test_pdr_cpu import kat_file

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import epiallele_oracle as EP  # noqa: E402
import mhl_oracle as MH  # noqa: E402
import region_oracle as RG  # noqa: E402

import bsmap_b200 as B
from bsmap_b200 import lib as BL

pytestmark = pytest.mark.gpu
BIN = os.path.dirname(BL.LIB_PATH)
METHRATIO, BSMAP = os.path.join(BIN, "methratio"), os.path.join(BIN, "bsmap")
IGNORE = (2, 1, 3, 2)
# name -> (epialleles, PDR's K or None, conversion threshold or None, M-bias + exclusion, C/T SNP mode)
VARIANTS = {"mhl": (False, None, None, False, None), "epi": (True, None, None, False, None), "pdr": (False, 4, None, False, None),
            "conv_mbias": (False, None, 2, True, None), "correct": (False, None, None, False, "correct"),
            "skip": (False, None, None, False, "skip"), "all": (True, 2, 2, True, "skip")}


def add_all(mh, cols, batches=1):
    n = len(cols[0])
    cut = [n * k // batches for k in range(batches + 1)]
    for b, e in zip(cut, cut[1:]):
        if e > b:
            mh.add(*[c[b:e] for c in cols[:7]], read2=cols[7][b:e])


def make_meth(ix, opts, epi=False, min_cpg=None, threshold=None, mbias=False, ct_snp=None, ignore=None, mhl=True):
    mh = B.Meth(ix, opts)
    if mhl:
        mh.enable_mhl()
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


def run_ok(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return r


def regions_of(names, res, width=60):
    lengths = {n: len(s) for n, s in res["ref"].items()}
    regs = RG.tiles(lengths, width) + [(n, 0, L + 7) for n, L in lengths.items()] + [(n, L // 3, L // 2) for n, L in lengths.items()]
    idx = {n: k for k, n in enumerate(names)}
    return regs, [idx[r[0]] for r in regs], [r[1] for r in regs], [r[2] for r in regs]


def same_as_oracle(mh, names, res, regs, ct_snp=None):
    """counters, summary, region sums and the file == the oracle's"""
    assert mh.valid() == res["valid"]
    assert mh.mhl() == (res["alignments"], res["calls"])
    for k, n in enumerate(names):
        if n not in res["counts"]:
            continue
        pos, counts = mh.mhl_counters(k)
        assert np.array_equal(pos, res["sites"][n]), n
        assert np.array_equal(counts, res["counts"][n]), n
    regs_, c, s, e = regs
    sites, sums = mh.mhl_regions(c, s, e)
    for (n, t), x, y in zip(MH.regions(res, regs_, ct_snp), sites, sums):
        assert n == x and np.array_equal(t, y)
    assert read_fd(lambda fd: mh.write_mhl(fd, c, s, e)) == MH.mhl_text(res, regs_, ct_snp)
    return sums


API_KEYS = ["pe_sam.p_u", "pe_sam.r", "pe_readthrough.p_g", "se_n1.r_t_0", "se_n1.t_5_g", "rrbs_pe.t_0", "se_cfg1.g_z",
            "se_cfg2_bsp.r_u", "pe_bsp_r0.r", "pe_sam.bam.r", "rrbs_se_A.bam.r_u"]


@pytest.mark.parametrize("key", API_KEYS)
def test_meth_add_equals_the_oracle(tmp_path, key):
    """bsx_meth_add in one and in three batches, in every variant: run counters, summary, region sums and file == oracle;
    the other counters are those of the run without MHL; on the device T_4, M_4, U_4 are the windows' reads, UUUU and
    MMMM counts (with epialleles), and T_1, M_1 the region report's CpG CT_count and C_count (-g, no SNP mode)"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = opts_kwargs(ent["opts"])
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth", "combine_cpg")}
    bsp = not files[0].upper().endswith(".SAM")
    cols = api_arrays(files, d["gnames"])
    ix = B.Index.packed(d["gnames"], d["gseqs"])
    calls = 0
    for name, (epi, k, threshold, mbias, ct_snp) in VARIANTS.items():
        if mbias and bsp:
            continue                                          # BSP records carry no read number
        ignore = IGNORE if mbias else None
        res = MH.mhl(d["gnames"], d["gseqs"], files, threshold=threshold or 0, ignore=ignore or (0, 0, 0, 0), **ckw)
        regs = regions_of(d["gnames"], res)
        calls += res["calls"]
        for batches in (1, 3):
            mh = make_meth(ix, B.meth_opts(**kw), epi, k, threshold, mbias, ct_snp, ignore)
            add_all(mh, cols, batches)
            sums = same_as_oracle(mh, d["gnames"], res, regs, ct_snp)
            plain = make_meth(ix, B.meth_opts(**kw), epi, k, threshold, mbias, ct_snp, ignore, mhl=False)
            add_all(plain, cols, batches)
            assert plain.valid() == mh.valid()
            for kk, n in enumerate(d["gnames"]):
                assert all(np.array_equal(a, b) for a, b in zip(plain.counters(kk), mh.counters(kk))), name
                if epi:
                    assert all(np.array_equal(a, b) for a, b in zip(plain.epiallele_counters(kk), mh.epiallele_counters(kk))), name
            if epi:
                assert plain.epialleles() == mh.epialleles()
                if not ct_snp:
                    for (cr, s, e), t in zip(regs[0], sums):
                        kk = d["gnames"].index(cr)
                        pos, ep = mh.epiallele_counters(kk)
                        a, b = np.searchsorted(pos, min(s, len(d["gseqs"][kk]))), np.searchsorted(pos, min(e, len(d["gseqs"][kk])))
                        w = ep[a:max(b - 3, a)].astype(np.int64)
                        assert (t[0, 3], t[1, 3], t[2, 3]) == (w.sum(), w[:, 15].sum(), w[:, 0].sum()), (cr, s, e)
            if k:
                assert plain.pdr() == mh.pdr()
            if kw.get("combine_cpg") and not ct_snp:
                rr = mh.regions(*regs[1:])
                assert np.array_equal(sums[:, 0, 0], rr[:, 0, 3]) and np.array_equal(sums[:, 1, 0], rr[:, 0, 2])
            mh.close(); plain.close()
    assert calls > 0
    ix.close()


@pytest.mark.parametrize("name", sorted(KATS))
def test_known_answers_on_the_device(tmp_path, name):
    """the hand-computed cases through bsx_meth_add, one batch per record, upper- and lower-case reference"""
    lines, regs, ct_snp, _ = KATS[name]
    sam = kat_file(tmp_path, lines)
    for seqs in ([s.encode() for s in SEQS], [s.lower().encode() for s in SEQS]):
        res = MH.mhl(NAMES, seqs, [sam], trim_fillin=0)
        ix = B.Index.packed(NAMES, seqs)
        mh = make_meth(ix, B.meth_opts(trim_fillin=0), ct_snp=ct_snp)
        add_all(mh, api_arrays([sam], NAMES), batches=len(lines))
        c = [0] * len(regs)
        same_as_oracle(mh, NAMES, res, (regs, c, [r[1] for r in regs], [r[2] for r in regs]), ct_snp)
        mh.close(); ix.close()


CLI_KEYS = ["pe_sam.default", "pe_sam.r", "se_cfg2_bsp.default", "pe_bsp_r0.r", "se_cfg2_r0_uR.bam.default", "se_n1.t_5_g", "rrbs_se_A.z"]


@pytest.mark.parametrize("key", CLI_KEYS)
def test_methratio_cli(tmp_path, key):
    """methratio --mhl F with --tiles or --regions (shared with --region-report), with epialleles, PDR, the SNP modes and
    the conversion filter: the file and the stderr line == oracle; every other output is byte-equal to the run without"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    fa, _, _ = CS.write_inputs(case, str(tmp_path))
    files = alignment_files(case, str(tmp_path), bam=ent.get("bam", False))
    kw = opts_kwargs(ent["opts"])
    ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth", "combine_cpg")}
    ofiles = oracle_files(ent, case, str(tmp_path))
    sam = ofiles[0].upper().endswith(".SAM")
    t0, t, mh, rr0, rr, e0, e, bed = (str(tmp_path / x) for x in ("t0", "t", "mh", "rr0", "rr", "e0", "e", "r.bed"))
    lengths = {n: len(s) for n, s in zip(d["gnames"], d["gseqs"])}
    bregs = [(n, L // 4, L // 4 + 300) for n, L in lengths.items()] + [(n, 0, L + 50) for n, L in lengths.items()]
    open(bed, "w").write("".join("%s\t%d\t%d\n" % r for r in bregs))
    for extra, regopt in (([], ["--tiles", "100"]), (["--ct-snp", "skip"], ["--regions", bed]),
                          (["--ct-snp", "correct", "--conversion-filter", "2", "--pdr", str(tmp_path / "p")], ["--tiles", "1000"])):
        base = [METHRATIO, "-d", fa, "-q"] + ent["opts"] + extra + regopt
        if sam:
            base += ["--mbias-ignore", "1,2,0,3"]
        r0 = run_ok(base + ["-o", t0, "--region-report", rr0, "--epialleles", e0] + files)
        r = run_ok(base + ["-o", t, "--region-report", rr, "--epialleles", e, "--mhl", mh] + files)
        assert r.stdout == r0.stdout
        for a, b in ((t, t0), (rr, rr0), (e, e0)):
            assert open(a, "rb").read() == open(b, "rb").read()
        mode = extra[1] if extra else None
        res = MH.mhl(d["gnames"], d["gseqs"], ofiles, threshold=2 if "--conversion-filter" in extra else 0,
                     ignore=(1, 2, 0, 3) if sam else (0, 0, 0, 0), **ckw)
        regs = RG.tiles(lengths, int(regopt[1])) if regopt[0] == "--tiles" else bregs
        exp = MH.mhl_text(res, regs, mode)
        assert open(mh).read() == exp, (extra, R.first_diff(open(mh, "rb").read(), exp.encode()))
        assert MH.stderr_line(res) in r.stderr.splitlines()
        assert [x for x in r.stderr.splitlines() if not x.startswith("MHL:")] == r0.stderr.splitlines()
        only = run_ok([METHRATIO, "-d", fa, "-q", "-o", str(tmp_path / "t1"), "--mhl", str(tmp_path / "m1")] + ent["opts"] + extra + regopt
                      + (["--mbias-ignore", "1,2,0,3"] if sam else []) + files)
        assert open(str(tmp_path / "m1")).read() == exp and MH.stderr_line(res) in only.stderr.splitlines()


@pytest.mark.parametrize("name,ext", [("se_cfg2_r0_uR", "sam"), ("pe_sam", "sam"), ("se_cfg2_bsp", "bsp")])
def test_bsmap_cli(tmp_path, name, ext):
    """bsmap --methratio T --meth-mhl F --meth-tiles W (in-process pile-up): == methratio --mhl on the alignment file the
    same run wrote, and == the oracle; the table, region report and summary are those of the run without --meth-mhl"""
    case = CS.BY_NAME[name]
    d = case.data()
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / ("out." + ext))
    t0, t, r0_, r_, mh, t2, mh2 = (str(tmp_path / x) for x in ("t0", "t", "r0", "r", "mh", "t2", "mh2"))
    reg = ["--meth-tiles", "200"]
    r0 = run_ok([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t0, "--meth-zero", "--meth-region-report", r0_] + reg)
    r = run_ok([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t, "--meth-zero", "--meth-region-report", r_, "--meth-mhl", mh] + reg)
    summary = lambda out: [x for x in out.splitlines() if "valid mappings" in x]
    assert summary(r.stdout) == summary(r0.stdout) and open(t).read() == open(t0).read() and open(r_).read() == open(r0_).read()
    m = run_ok([METHRATIO, "-o", t2, "-d", fa, "-z", "--mhl", mh2, "--tiles", "200", o])
    assert open(mh).read() == open(mh2).read() and open(t).read() == open(t2).read()
    res = MH.mhl(d["gnames"], d["gseqs"], [o])
    assert open(mh).read() == MH.mhl_text(res, MH.tiles(res, 200))
    assert MH.stderr_line(res) in r.stderr.splitlines() and MH.stderr_line(res) in m.stderr.splitlines()
    assert res["calls"] > 0


def _map_in_process(case, max_batch, **kw):
    d = case.data()
    p = B.make_params(**case.param_kwargs())
    ix = B.Index(p, d["gnames"], d["gseqs"])
    mp = B.Mapper(ix, p, max_batch=max_batch, stride=160)
    mh = make_meth(ix, B.meth_opts(), **kw)
    mh.attach(mp, sam_rules=bool(p.out_sam))
    if not case.paired:
        buf, lens = B.pack_reads(R.clip(case, d["seqs"]), stride=160)
        mp.map_se(buf, lens)
    else:
        ba, la = B.pack_reads(R.clip(case, d["seqs"]), stride=160)
        bb, lb = B.pack_reads(R.clip(case, d["seqs_b"]), stride=160)
        mp.map_pe(ba, la, bb, lb)
    return d, ix, mp, mh


@pytest.mark.parametrize("name", ["se_n1", "pe_sam"])
def test_batch_size_invariance(tmp_path, name):
    """64 and 1 M alignments per batch, through the mapped kernel, give the same run counters, summary and file, equal to
    the oracle on the golden text"""
    case = CS.BY_NAME[name]
    files = alignment_files(case, str(tmp_path))
    out = []
    for mb in (64, 1 << 20):
        d, ix, mp, mh = _map_in_process(case, mb, epi=True, min_cpg=2, threshold=3, mbias=True, ignore=(1, 2, 3, 4))
        res = MH.mhl(d["gnames"], d["gseqs"], files, threshold=3, ignore=(1, 2, 3, 4))
        same_as_oracle(mh, d["gnames"], res, regions_of(d["gnames"], res))
        out.append((mh.mhl(), [mh.mhl_counters(k)[1] for k in range(len(d["gnames"]))]))
        mh.close(); mp.close(); ix.close()
    assert out[0][0] == out[1][0] and out[0][0][1] > 0
    assert all(np.array_equal(x, y) for x, y in zip(out[0][1], out[1][1]))


def test_misuse_is_refused(tmp_path):
    ix = B.Index.packed(["c"], [b"ACGT" * 100])
    mh = B.Meth(ix, B.meth_opts())
    for call in (mh.mhl, lambda: mh.mhl_counters(0), lambda: mh.mhl_regions([0], [0], [10]), lambda: read_fd(lambda fd: mh.write_mhl(fd, [0], [0], [10]))):
        with pytest.raises(B.BsxError, match="not enabled"):
            call()
    mh.enable_mhl()
    with pytest.raises(B.BsxError, match="already enabled"):
        mh.enable_mhl()
    with pytest.raises(B.BsxError, match="start 10 > end 5"):
        mh.mhl_regions([0], [10], [5])
    with pytest.raises(B.BsxError, match="sequence 3 of 1"):
        mh.mhl_regions([3], [0], [5])
    mh.enable_epialleles()                                    # shares the rank index
    assert mh.mhl_counters(0)[0].tolist() == mh.epiallele_counters(0)[0].tolist() == list(range(1, 400, 4))
    mh.close()
    mh = B.Meth(ix, B.meth_opts())
    mh.add([b"ACGTACGT"], [0], [0], [0], [0], [0], [4])
    with pytest.raises(B.BsxError, match="error 1:.*already piled up"):
        mh.enable_mhl()
    mh.close(); ix.close()
    case = CS.BY_NAME["se_n1"]
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o, m = str(tmp_path / "o.sam"), str(tmp_path / "m")
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--meth-mhl", m, "--meth-tiles", "100"], capture_output=True, text=True)
    assert r.returncode == 2 and "--methratio" in r.stderr and not os.path.exists(m)
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", str(tmp_path / "t"), "--meth-mhl", m], capture_output=True, text=True)
    assert r.returncode == 2 and "--meth-regions" in r.stderr and not os.path.exists(m)
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", str(tmp_path / "t"), "--meth-tiles", "100"], capture_output=True, text=True)
    assert r.returncode == 1 and "need --meth-region-report" in r.stderr
    for extra, msg in ((["--mhl", m], "--mhl needs --regions"), (["--tiles", "5"], "need --region-report"),
                       (["--mhl", m, "--tiles", "5", "--regions", fa], "exclude each other")):
        r = subprocess.run([METHRATIO, "-d", fa, "-o", str(tmp_path / "t"), o] + extra, capture_output=True, text=True)
        assert r.returncode == 2 and "methratio: error:" in r.stderr and msg in r.stderr, r.stderr
    assert not os.path.exists(m)


# ---- randomised rounds on the fuzz generators ------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [3, 4, 5])
def test_fuzz_rounds(tmp_path, seed):
    """generated references, records and options (meth_fuzz, -r, -u / -p, 1 bp tiles among them), random batch cuts: the
    run counters, summary, region sums, MHL file and the unchanged table == the oracle"""
    rng = np.random.default_rng(seed)
    for rnd in range(6):
        names, seqs = MF.make_reference(rng)
        sam = rng.random() < 0.7
        o = MF.draw_options(rng, names, seqs, sam)
        if rnd == 0 and sum(len(x) for x in seqs) <= 50_000:
            o["regions"] = ("tiles", 1)
        recs = MF.make_records(rng, names, seqs, int(rng.choice([60, 400, 2000])), rm_dup=o["rm_dup"])
        path = str(tmp_path / ("a%d_%d.%s" % (seed, rnd, "sam" if sam else "bsp")))
        open(path, "w").write(MF.sam_text(recs, names, seqs) if sam else MF.bsp_text(recs))
        e = MF.expected(names, seqs, [path], o)
        res = MH.mhl(names, seqs, [path], threshold=o["conv"] or 0, chroms=o["chroms"], unique=o["unique"], pair=o["pair"],
                     trim_fillin=o["trim_fillin"], rm_dup=o["rm_dup"], ignore=o["ignore"] or (0, 0, 0, 0))
        sel = [not o["chroms"] or n in o["chroms"] for n in names]
        cols = api_arrays([path], names) or [[] for _ in range(8)]
        keep = [i for i, c in enumerate(cols[1]) if sel[c]]
        cols = [[c[i] for i in keep] for c in cols]
        cuts = MF.batch_cuts(rng, len(cols[0]))
        ix = B.Index.packed(names, seqs)
        mh = MF.new_meth(B, ix, o)
        mh.enable_mhl()
        for b, x in zip(cuts, cuts[1:]):
            mh.add(*[c[b:x] for c in cols[:7]], read2=cols[7][b:x])
        desc = (seed, rnd, {x: v for x, v in o.items() if v and x != "regions"})
        assert MF.compare_counters(mh, names, o, e["res"]) is None, desc
        regs = MF.region_list(o, names, seqs) or [(n, 0, len(s)) for n, s in zip(names, seqs) if n in res["ref"]]
        idx = {n: k for k, n in enumerate(names)}
        same_as_oracle(mh, names, res, (regs, [idx[r[0]] for r in regs], [r[1] for r in regs], [r[2] for r in regs]), o["ct_snp"])
        assert read_fd(lambda fd: mh.write(seqs, fd, chroms=sel)) == e["table"], desc
        mh.close(); ix.close()


# ---- end to end: methylation on whole molecules against scattered methylation ----------------------------------------
GLEN, RLEN, NREADS = 200_000, 100, 80_000
REGIONS = {"whole": (20_000, 30_000), "scattered": (60_000, 70_000)}


def _simulate(rng, genome: bytes):
    """directional reads from both strands at 40x; a fragment overlapping "whole" is all methylated or all unmethylated
    (p = 1/2), one overlapping "scattered" has each CpG methylated with p = 1/2; elsewhere p = 0.8; non-CpG C converted"""
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    g = np.frombuffer(genome, dtype=np.uint8)
    C, G, T, A = (ord(x) for x in "CGTA")
    cpg_c = np.zeros(len(g), dtype=bool)
    cpg_c[:-1] = (g[:-1] == C) & (g[1:] == G)
    cpg_g = np.zeros(len(g), dtype=bool)
    cpg_g[1:] = cpg_c[:-1]
    reads = []
    for _ in range(NREADS):
        s = int(rng.integers(0, len(g) - RLEN))
        sl = slice(s, s + RLEN)
        crick = rng.random() < 0.5
        c_here = (g[sl] == G) if crick else (g[sl] == C)
        cpg = (cpg_g if crick else cpg_c)[sl]
        region = next((k for k, (b, e) in REGIONS.items() if s < e and s + RLEN > b), None)
        if region == "whole":
            m_cpg = np.full(RLEN, rng.random() < 0.5)
        elif region == "scattered":
            m_cpg = rng.random(RLEN) < 0.5
        else:
            m_cpg = rng.random(RLEN) < 0.8
        meth = np.where(cpg, m_cpg, False)
        w = g[sl].copy()
        w[c_here & ~meth] = A if crick else T
        read = w.tobytes()
        reads.append(read.translate(comp)[::-1] if crick else read)
    return reads


def test_mhl_separates_whole_molecules_from_scattered_methylation(tmp_path):
    """two planted 10 kb regions at a mean CpG level of about 0.5: MHL is near 0.5 where methylation sits on whole
    molecules and far lower where it is scattered; the region report's levels are alike"""
    from bsmap_b200 import synth
    gen = synth.make_genome(23, [GLEN])
    gb = gen[0].numpy().tobytes()
    reads = _simulate(np.random.default_rng(7), gb)
    fa, fq, sam, bed = (str(tmp_path / x) for x in ("g.fa", "r.fq", "o.sam", "r.bed"))
    synth.write_fasta(fa, gen, names=["chr1"])
    synth.write_fastq(fq, np.frombuffer(b"".join(reads), dtype=np.uint8).reshape(len(reads), RLEN), ["r%d" % i for i in range(len(reads))])
    regs = [("chr1",) + REGIONS[k] for k in ("whole", "scattered")]
    open(bed, "w").write("".join("%s\t%d\t%d\n" % r for r in regs))
    t, rr, mh = (str(tmp_path / x) for x in ("t", "rr", "mh"))
    r = run_ok([BSMAP, "-a", fq, "-d", fa, "-o", sam, "-v", "5", "--methratio", t, "--meth-region-report", rr, "--meth-regions", bed,
                "--meth-mhl", mh])
    level = [float(x.split("\t")[8]) for x in open(rr).read().splitlines()[1:] if x.split("\t")[3] == "CpG"]
    rows = [x.split("\t") for x in open(mh).read().splitlines()[1:]]
    mhl = {k: float(x[6]) for k, x in zip(("whole", "scattered"), rows)}
    print("CpG levels:", level, "MHL:", mhl, "L:", [x[5] for x in rows])
    assert all(abs(v - 0.5) < 0.05 for v in level), level
    assert abs(mhl["whole"] - 0.5) < 0.1, mhl           # long haplotypes are few, and weigh l
    assert mhl["scattered"] < 0.2, mhl
    res = MH.mhl(["chr1"], [gb], [sam])
    assert open(mh).read() == MH.mhl_text(res, regs)
    assert MH.stderr_line(res) in r.stderr.splitlines()
