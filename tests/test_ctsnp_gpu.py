"""C/T SNP evidence on the device (the Snp pile-up kernels of bsx_meth.cu, `methratio --ct-snp`, `bsmap --methratio
--meth-ct-snp`) against the numpy restatement (oracle/ctsnp_oracle.py), and planted SNPs mapped end to end."""
from __future__ import annotations

import os
import subprocess
import sys

import numpy as np
import pytest

import cases as CS
import runners as R
from meth_inputs import api_arrays
from test_methratio_cpu import MANIFEST, alignment_files
from test_mbias_cpu import oracle_files
from test_ctsnp_cpu import split_kwargs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ctsnp_oracle as CT  # noqa: E402

import bsmap_b200 as B
from bsmap_b200 import lib as BL
from bsmap_b200 import synth

pytestmark = pytest.mark.gpu
BIN = os.path.dirname(BL.LIB_PATH)
METHRATIO, BSMAP = os.path.join(BIN, "methratio"), os.path.join(BIN, "bsmap")


def add_all(mh, cols, batches=1):
    n = len(cols[0])
    cut = [n * k // batches for k in range(batches + 1)]
    for b, e in zip(cut, cut[1:]):
        mh.add(*[c[b:e] for c in cols[:7]], read2=cols[7][b:e])


def table_bytes(mh, gseqs, tmp_path):
    out = tmp_path / "t.txt"
    fd = os.open(out, os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    mh.write(gseqs, fd)
    os.close(fd)
    return out.read_bytes()


def same_counters(mh, names, cnt):
    for k, n in enumerate(names):
        m, dp = mh.counters(k)
        c, s = mh.ct_snp_counters(k)
        exp = cnt[n]
        assert all(np.array_equal(x, y) for x, y in zip((m, dp, c, s), exp)), n


# SE / PE SAM, BSP, BAM, RRBS, -r (three batches), -g, -u / -p, -z, -t
API_KEYS = ["pe_sam.p_u", "pe_sam.r", "pe_readthrough.p_g", "se_n1.r_t_0", "se_n1.t_5_g", "rrbs_pe.t_0", "pe_sam_v5_R.r_p",
            "se_cfg1.g_z", "se_cfg2_bsp.r_u", "pe_bsp_r0.default", "pe_sam.bam.r", "rrbs_se_A.bam.r_u"]


@pytest.mark.parametrize("key", API_KEYS)
def test_meth_add_ct_snp_equals_the_oracle(tmp_path, key):
    """bsx_meth_add with the evidence on: counters == oracle, table bytes == oracle in each mode"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw, tk = split_kwargs(ent["opts"])
    cnt, nmap, ref = CT.counters(d["gnames"], d["gseqs"], files, **kw)
    cols = api_arrays(files, d["gnames"])
    ix = B.Index.packed(d["gnames"], d["gseqs"])
    for mode in CT.MODES:
        mh = B.Meth(ix, B.meth_opts(**kw, **tk))
        mh.enable_ct_snp(mode)
        add_all(mh, cols, batches=3 if kw.get("rm_dup") else 1)
        assert mh.valid() == nmap
        same_counters(mh, d["gnames"], cnt)
        got = table_bytes(mh, d["gseqs"], tmp_path)
        exp = CT.table(cnt, ref, mode, **tk)[0].encode()
        assert got == exp, (mode, R.first_diff(got, exp))
        mh.close()
    assert sum(int(c[3].sum()) for c in cnt.values()) > 0      # sequencing errors give SNP evidence here too
    ix.close()


CLI_KEYS = ["pe_sam.default", "pe_sam.r", "se_cfg2_bsp.default", "pe_bsp_r0.r", "se_cfg2_r0_uR.bam.default", "se_n1.t_5_g",
            "se_cfg5.r_z", "rrbs_se_A.z", "pe_n1.c_chr2+chr1", "se_cfg2_r0_uR.z_m_2"]


@pytest.mark.parametrize("key", CLI_KEYS)
def test_methratio_cli_ct_snp(tmp_path, key):
    """methratio --ct-snp MODE: table bytes == oracle (BSP included), summary line == the plain run's"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    fa, _, _ = CS.write_inputs(case, str(tmp_path))
    files = alignment_files(case, str(tmp_path), bam=ent.get("bam", False))
    kw, tk = split_kwargs(ent["opts"])
    cnt, _, ref = CT.counters(d["gnames"], d["gseqs"], oracle_files(ent, case, str(tmp_path)), **kw)
    out = str(tmp_path / "meth.txt")
    for mode in CT.MODES:
        r = subprocess.run([METHRATIO, "-o", out, "-d", fa, "-q", "--ct-snp", mode] + ent["opts"] + files, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        assert r.stdout.strip() == ent["stdout"]
        got, exp = open(out, "rb").read(), CT.table(cnt, ref, mode, **tk)[0].encode()
        assert got == exp, (mode, R.first_diff(got, exp))


@pytest.mark.parametrize("name", ["pe_sam", "se_cfg2_r0_uR"])
def test_bsmap_cli_meth_ct_snp(tmp_path, name):
    """bsmap --methratio t --meth-ct-snp MODE (in-process pile-up) == methratio --ct-snp MODE on the SAM the same run wrote"""
    case = CS.BY_NAME[name]
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / "out.sam")
    t1, t2 = str(tmp_path / "t1"), str(tmp_path / "t2")
    for mode in CT.MODES:
        r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t1, "--meth-zero", "--meth-ct-snp", mode], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        r = subprocess.run([METHRATIO, "-o", t2, "-d", fa, "-q", "-z", "--ct-snp", mode, o], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert open(t1, "rb").read() == open(t2, "rb").read()
        assert open(t1).readline().split("\t")[5] == "eff_CT_count"


def test_mbias_unchanged_by_ct_snp(tmp_path):
    """M-bias + exclusion (the Snp + Cycles kernels): report, table columns and calls identical with and without
    --ct-snp; the evidence == oracle with the same exclusion"""
    case = CS.BY_NAME["pe_sam"]
    d = case.data()
    fa, _, _ = CS.write_inputs(case, str(tmp_path))
    files = alignment_files(case, str(tmp_path))
    ign = "2,3,4,1"
    res = []
    for extra in ([], ["--ct-snp", "no-action"]):
        t, mb = str(tmp_path / "t.txt"), str(tmp_path / "mb.txt")
        r = subprocess.run([METHRATIO, "-o", t, "-d", fa, "-q", "--mbias", mb, "--mbias-ignore", ign] + extra + files, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        res.append((open(t).read(), open(mb).read(), r.stdout))
    assert res[0][1] == res[1][1] and res[0][2] == res[1][2]
    assert CT.project_plain(res[1][0]) == res[0][0]
    cnt, nmap, _ = CT.counters(d["gnames"], d["gseqs"], files, ignore=(2, 3, 4, 1))
    ix = B.Index.packed(d["gnames"], d["gseqs"])
    plain, mh = B.Meth(ix, B.meth_opts()), B.Meth(ix, B.meth_opts())
    for h in (plain, mh):
        h.enable_mbias(); h.set_ignore(2, 3, 4, 1)
    mh.enable_ct_snp("skip")
    cols = api_arrays(files, d["gnames"])
    add_all(plain, cols, batches=2); add_all(mh, cols, batches=2)
    assert np.array_equal(plain.mbias()[0], mh.mbias()[0]) and mh.valid() == plain.valid() == nmap
    same_counters(mh, d["gnames"], cnt)
    plain.close(); mh.close(); ix.close()


def _map_in_process(case, max_batch, mode="correct", ignore=None):
    d = case.data()
    p = B.make_params(**case.param_kwargs())
    ix = B.Index(p, d["gnames"], d["gseqs"])
    mp = B.Mapper(ix, p, max_batch=max_batch, stride=160)
    mh = B.Meth(ix, B.meth_opts())
    mh.enable_ct_snp(mode)
    if ignore:
        mh.set_ignore(*ignore)
    mh.attach(mp, sam_rules=bool(p.out_sam))
    if not case.paired:
        buf, lens = B.pack_reads(R.clip(case, d["seqs"]), stride=160)
        mp.map_se(buf, lens)
    else:
        ba, la = B.pack_reads(R.clip(case, d["seqs"]), stride=160)
        bb, lb = B.pack_reads(R.clip(case, d["seqs_b"]), stride=160)
        mp.map_pe(ba, la, bb, lb)
    return d, ix, mp, mh


@pytest.mark.parametrize("name,ignore", [("se_cfg2_r0_uR", None), ("pe_sam", None), ("se_cfg2_bsp", None), ("rrbs_pe", None),
                                         ("pe_readthrough", (1, 2, 3, 4)), ("se_cfg5", (0, 3, 0, 0))])
def test_in_process_equals_the_oracle(tmp_path, name, ignore):
    """Mapper + attached Meth, many batches on both streams (Snp, and Snp + Cycles with exclusion): counters == oracle on
    the text the records format to"""
    case = CS.BY_NAME[name]
    d, ix, mp, mh = _map_in_process(case, max_batch=256, ignore=ignore)
    cnt, _, _ = CT.counters(d["gnames"], d["gseqs"], alignment_files(case, str(tmp_path)), ignore=ignore or (0, 0, 0, 0))
    same_counters(mh, d["gnames"], cnt)
    mh.close(); mp.close(); ix.close()


@pytest.mark.parametrize("name", ["se_n1", "pe_sam"])
def test_batch_size_invariance(name):
    """64 and 1 M alignments per batch give the same counters, with and without exclusion"""
    for ignore in (None, (1, 2, 3, 4)):
        res = []
        for mb in (64, 1 << 20):
            d, ix, mp, mh = _map_in_process(CS.BY_NAME[name], max_batch=mb, ignore=ignore)
            res.append([mh.counters(k) + mh.ct_snp_counters(k) for k in range(len(d["gnames"]))])
            mh.close(); mp.close(); ix.close()
        for a, b in zip(*res):
            assert all(np.array_equal(x, y) for x, y in zip(a, b))
        assert sum(int(a[2].sum()) for a in res[0]) > 0


def test_misuse_is_refused(tmp_path):
    ix = B.Index.packed(["c"], [b"ACGT" * 100])
    mh = B.Meth(ix, B.meth_opts())
    with pytest.raises(ValueError, match="ct-snp mode"):
        mh.enable_ct_snp("fix")
    for bad in (0, 4, -1):
        with pytest.raises(B.BsxError, match="mode must be"):
            BL.check(BL.load().bsx_meth_enable_ct_snp(mh.h, bad))
    with pytest.raises(B.BsxError, match="not enabled"):
        mh.ct_snp_counters(0)
    mh.add([b"ACGTACGT"], [0], [0], [0], [0], [0], [4])
    with pytest.raises(B.BsxError, match="error 1:.*already piled up"):
        mh.enable_ct_snp("skip")
    mh.close(); ix.close()
    case = CS.BY_NAME["se_n1"]
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / "o.sam")
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--meth-ct-snp", "skip"], capture_output=True, text=True)
    assert r.returncode != 0 and "--methratio" in r.stderr
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", str(tmp_path / "t"), "--meth-ct-snp", "fix"], capture_output=True, text=True)
    assert r.returncode != 0 and "fix" in r.stdout
    r = subprocess.run([METHRATIO, "-o", str(tmp_path / "t"), "-d", fa, "--ct-snp", "fix", o], capture_output=True, text=True)
    assert r.returncode == 2 and "--ct-snp" in r.stderr


# ---- planted SNPs ---------------------------------------------------------------------------------------------------
GLEN, RLEN, NREADS = 120_000, 100, 72_000          # 60x over the genome, about 30x per strand


def _sites(g: np.ndarray, base: int, first: int, count: int, step=1000):
    """`count` positions holding `base`, one near each of first, first + step, ..."""
    out = []
    for k in range(count):
        p = first + k * step
        p += int(np.argmax(g[p:p + 50] == base))
        assert g[p] == base
        out.append(p)
    return out


def test_planted_snps_end_to_end(tmp_path):
    """Reads from a genome with homozygous C>T at '+' Cs and G>A at '-' Cs, and half the reads with heterozygous ones at
    other sites, mapped to the original: skip drops every planted site with opposite-strand coverage, correct drops the
    homozygous ones and halves eff_CT_count at the heterozygous ones, other sites read the same in every mode but where
    sequencing errors give evidence; every table == oracle on the SAM of the same run"""
    g = synth.make_genome(5, [GLEN])[0].numpy().copy()
    C, G, T, A = (ord(x) for x in "CGTA")
    hom_p, hom_m = _sites(g, C, 500, 25), _sites(g, G, 700, 25)
    het_p, het_m = _sites(g, C, 900, 25), _sites(g, G, 1100, 25)
    hom = g.copy()
    hom[hom_p], hom[hom_m] = T, A
    het = hom.copy()
    het[het_p], het[het_m] = T, A
    import torch
    sims = [synth.simulate_reads([torch.from_numpy(x)], NREADS // 2, RLEN, seed=s, first_index=s * NREADS) for x, s in ((hom, 1), (het, 2))]
    seqs = torch.cat([s["seq"] for s in sims]).numpy()
    fa, fq, sam = str(tmp_path / "g.fa"), str(tmp_path / "r.fq"), str(tmp_path / "o.sam")
    synth.write_fasta(fa, [torch.from_numpy(g)], names=["chr1"])
    synth.write_fastq(fq, seqs, ["r%d" % i for i in range(len(seqs))])
    tables = {}
    for mode in CT.MODES:
        t = str(tmp_path / ("t_" + mode))
        r = subprocess.run([BSMAP, "-a", fq, "-d", fa, "-o", sam, "-v", "5", "--methratio", t, "--meth-zero", "--meth-ct-snp", mode],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        tables[mode] = open(t).read()
    cnt, _, ref = CT.counters(["chr1"], [g.tobytes()], [sam])
    for mode in CT.MODES:
        assert tables[mode] == CT.table(cnt, ref, mode, meth0=True)[0], mode
    rows = {m: {int(c[1]) - 1: c for c in (x.split("\t") for x in tables[m].splitlines()[1:])} for m in CT.MODES}
    rev_g = lambda c: int(c[8])
    rev_ga = lambda c: int(c[9])
    na = rows["no-action"]
    planted = hom_p + hom_m + het_p + het_m
    # coverage: every planted site is in the no-action table with opposite-strand evidence
    assert all(p in na and rev_ga(na[p]) >= 5 for p in planted)
    assert all(p not in rows["skip"] for p in planted)
    # homozygous: only sequencing errors can confirm the reference; correct drops a site exactly when nothing does
    for p in hom_p + hom_m:
        assert (p not in rows["correct"]) == (rev_g(na[p]) == 0)
    # a substitution shows the reference base in about 1 of 300 opposite-strand reads (1.4 % per base, 1 in 4 of them
    # the reference base), so about 10 % of the sites at this depth keep some confirming evidence
    assert sum(rev_g(na[p]) == 0 for p in hom_p + hom_m) >= 35
    # heterozygous: rev_G ~ Binomial(rev_GA, 1/2), eff_CT = CT * rev_G / rev_GA
    n = k = 0
    for p in het_p + het_m:
        c = rows["correct"][p]
        ga, gg = rev_ga(c), rev_g(c)
        assert abs(gg - ga / 2) <= 4 * (ga / 4) ** 0.5 + 1, (p, gg, ga)
        assert c[5] == "%.2f" % (float(int(c[7])) * gg / ga)
        n += ga; k += gg
    assert abs(k / n - 0.5) < 0.06, (k, n)
    # every other site: the same line in all modes unless it carries SNP evidence (sequencing errors)
    planted = set(planted)
    same = diff = 0
    for p, c in na.items():
        if p in planted:
            continue
        if rev_g(c) == rev_ga(c):
            assert rows["correct"][p] == c and rows["skip"][p] == c
            same += 1
        else:
            diff += 1
    assert same > 2 * diff and diff > 0
