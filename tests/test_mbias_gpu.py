"""M-bias and per-cycle exclusion on the device (the Cycles pile-up kernels of bsx_meth.cu, `methratio --mbias`,
`bsmap --methratio --meth-mbias`) against the numpy restatement (oracle/mbias_oracle.py) and the reference's tables."""
from __future__ import annotations

import gzip
import os
import subprocess
import sys

import numpy as np
import pytest

import cases as CS
import runners as R
from test_methratio_cpu import GOLD, MANIFEST, alignment_files, opts_kwargs
from meth_inputs import api_arrays
from test_mbias_cpu import KATS, NAMES, SEQS, mbias_kwargs, oracle_files, sam_line

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import mbias_oracle as MB  # noqa: E402

import bsmap_b200 as B
from bsmap_b200 import lib as BL

pytestmark = pytest.mark.gpu
BIN = os.path.dirname(BL.LIB_PATH)
METHRATIO, BSMAP = os.path.join(BIN, "methratio"), os.path.join(BIN, "bsmap")


def add_all(mh, cols, batches=1):
    n = len(cols[0])
    cut = [n * k // batches for k in range(batches + 1)]
    for b, e in zip(cut, cut[1:]):
        mh.add(*[c[b:e] for c in cols[:7]], read2=cols[7][b:e])


def table_bytes(mh, gseqs, tmp_path, chroms=None):
    out = tmp_path / "t.txt"
    fd = os.open(out, os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    mh.write(gseqs, fd, chroms=chroms)
    os.close(fd)
    return out.read_bytes()


API_KEYS = ["pe_sam.p_u", "pe_sam.r", "pe_readthrough.p_g", "se_n1.r_t_0", "se_n1.t_5_g", "rrbs_pe.t_0", "pe_sam_v5_R.r_p",
            "se_cfg1.u", "se_cfg2_bsp.r_u", "pe_sam.bam.r", "rrbs_se_A.bam.r_u"]


@pytest.mark.parametrize("key", API_KEYS)
def test_meth_add_mbias_equals_the_oracle(tmp_path, key):
    """bsx_meth_add with M-bias on: histogram == oracle, table bytes == the reference's (-r over three batches)"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = opts_kwargs(ent["opts"])
    ix = B.Index.packed(d["gnames"], d["gseqs"])
    mh = B.Meth(ix, B.meth_opts(**kw))
    mh.enable_mbias()
    add_all(mh, api_arrays(files, d["gnames"]), batches=3 if kw.get("rm_dup") else 1)
    hist, over = mh.mbias()
    exp, exp_over, _, nmap = MB.mbias(d["gnames"], d["gseqs"], files, **mbias_kwargs(ent["opts"]))
    assert over == exp_over == 0 and mh.valid() == nmap
    assert np.array_equal(hist.astype(np.int64), exp)
    got = table_bytes(mh, d["gseqs"], tmp_path)
    gold = gzip.open(os.path.join(GOLD, key + ".txt.gz"), "rb").read()
    assert got == gold, R.first_diff(got, gold)
    mh.close(); ix.close()


@pytest.mark.parametrize("name,kw,ignore", [("pe_sam", dict(trim_fillin=7), (3, 4, 5, 6)), ("pe_readthrough", dict(combine_cpg=True), (0, 0, 2, 0)),
                                            ("se_n1", dict(rm_dup=True, trim_fillin=0), (1, 2, 0, 0)), ("rrbs_pe", dict(unique=True, pair=True), (0, 5, 0, 5))])
def test_exclusion_equals_the_oracle(tmp_path, name, kw, ignore):
    """bsx_meth_set_ignore: the counters and the histogram lose exactly the oracle's excluded calls"""
    case = CS.BY_NAME[name]
    d = case.data()
    files = alignment_files(case, str(tmp_path))
    ix = B.Index.packed(d["gnames"], d["gseqs"])
    mh = B.Meth(ix, B.meth_opts(**kw))
    mh.enable_mbias()
    mh.set_ignore(*ignore)
    add_all(mh, api_arrays(files, d["gnames"]), batches=3)
    hist, _ = mh.mbias()
    exp, _, counters, nmap = MB.mbias(d["gnames"], d["gseqs"], files, ignore=ignore, **kw)
    assert np.array_equal(hist.astype(np.int64), exp) and mh.valid() == nmap
    for k, n in enumerate(d["gnames"]):
        m, dp = mh.counters(k)
        assert np.array_equal(m, counters[n][0]) and np.array_equal(dp, counters[n][1]), n
    assert exp.sum() > 0
    mh.close(); ix.close()


@pytest.mark.parametrize("key", sorted(MANIFEST))
def test_methratio_cli_mbias(tmp_path, key):
    """methratio --mbias: report == the oracle's text; table and stdout unchanged; BSP input is refused"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    fa, _, _ = CS.write_inputs(case, str(tmp_path))
    files = alignment_files(case, str(tmp_path), bam=ent.get("bam", False))
    out, mb = str(tmp_path / "meth.txt"), str(tmp_path / "mbias.txt")
    r = subprocess.run([METHRATIO, "-o", out, "-d", fa, "-q", "--mbias", mb] + ent["opts"] + files, capture_output=True, text=True)
    if case.out_ext == "bsp":
        assert r.returncode == 2 and "BSP" in r.stderr, r.stderr
        r = subprocess.run([METHRATIO, "-o", out, "-d", fa, "-q", "--mbias-ignore=0,0,0,0"] + ent["opts"] + files, capture_output=True, text=True)
        assert r.returncode == 2 and "BSP" in r.stderr, r.stderr
        return
    assert r.returncode == 0, r.stdout + r.stderr
    exp_table = gzip.open(os.path.join(GOLD, key + ".txt.gz"), "rb").read()
    assert open(out, "rb").read() == exp_table and r.stdout.strip() == ent["stdout"]
    hist, _, _, _ = MB.mbias(d["gnames"], d["gseqs"], oracle_files(ent, case, str(tmp_path)), **mbias_kwargs(ent["opts"]))
    assert open(mb).read() == MB.mbias_text(hist)
    r = subprocess.run([METHRATIO, "-o", out, "-d", fa, "-q", "--mbias-ignore", "0,0,0,0"] + ent["opts"] + files, capture_output=True, text=True)
    assert r.returncode == 0 and open(out, "rb").read() == exp_table and r.stdout.strip() == ent["stdout"]


def test_methratio_cli_mbias_grammar(tmp_path):
    case = CS.BY_NAME["pe_sam"]
    fa, _, _ = CS.write_inputs(case, str(tmp_path))
    files = alignment_files(case, str(tmp_path))
    out, mb = str(tmp_path / "m.txt"), str(tmp_path / "b.txt")
    for bad in ("1,2,3", "1,2,3,4,5", "a,0,0,0", "-1,0,0,0", "1,,2,3"):
        r = subprocess.run([METHRATIO, "-o", out, "-d", fa, "--mbias-ignore=" + bad] + files, capture_output=True, text=True)
        assert r.returncode == 2 and "--mbias-ignore" in r.stderr, (bad, r.stderr)
    r = subprocess.run([METHRATIO, "-o", out, "-d", fa, "-q", "--mbias=" + mb, "--mbias-ignore=2,1,3,0"] + files, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    d = case.data()
    hist, _, _, _ = MB.mbias(d["gnames"], d["gseqs"], files, ignore=(2, 1, 3, 0))
    assert open(mb).read() == MB.mbias_text(hist)


@pytest.mark.parametrize("name", sorted(KATS))
def test_known_answers_on_the_device(tmp_path, name):
    """the hand-computed cases through bsx_meth_add: sequence starts and ends, N, both strands, each exclusion bound"""
    lines, kw, exp_sparse = KATS[name]
    sam = tmp_path / "kat.sam"
    sam.write_text("@HD\tVN:1.0\n" + "".join(lines))
    ignore = kw.get("ignore", (0, 0, 0, 0))
    ix = B.Index.packed(NAMES, SEQS)
    mh = B.Meth(ix, B.meth_opts(trim_fillin=kw.get("trim_fillin", 2)))
    mh.enable_mbias()
    mh.set_ignore(*ignore)
    add_all(mh, api_arrays([str(sam)], NAMES))
    hist, over = mh.mbias()
    exp, _, counters, nmap = MB.mbias(NAMES, SEQS, [str(sam)], **kw)
    assert over == 0 and np.array_equal(hist.astype(np.int64), exp) and int(exp.sum()) == sum(exp_sparse.values())
    assert mh.valid() == nmap
    for k, n in enumerate(NAMES):
        m, dp = mh.counters(k)
        assert np.array_equal(m, counters[n][0]) and np.array_equal(dp, counters[n][1]), n
    mh.close(); ix.close()


def test_exclusion_without_mbias(tmp_path):
    """exclusion alone (no histogram kept): the counters equal the oracle's excluded table"""
    case = CS.BY_NAME["pe_sam"]
    d = case.data()
    files = alignment_files(case, str(tmp_path))
    ix = B.Index.packed(d["gnames"], d["gseqs"])
    mh = B.Meth(ix, B.meth_opts())
    mh.set_ignore(4, 3, 2, 5)
    add_all(mh, api_arrays(files, d["gnames"]), batches=2)
    _, _, counters, nmap = MB.mbias(d["gnames"], d["gseqs"], files, ignore=(4, 3, 2, 5))
    assert mh.valid() == nmap
    for k, n in enumerate(d["gnames"]):
        m, dp = mh.counters(k)
        assert np.array_equal(m, counters[n][0]) and np.array_equal(dp, counters[n][1]), n
    with pytest.raises(B.BsxError, match="not enabled"):
        mh.mbias()
    mh.close(); ix.close()


def test_in_process_readset_2_is_read_2(tmp_path):
    """single-end batches mapped as readset 2 (the mates file, FLAG 0x80 when printed) land in read 2, with read 2's
    exclusion: the histogram == the oracle on the SAM those records format to"""
    case = CS.BY_NAME["pe_sam"]
    d = case.data()
    kw = case.param_kwargs()
    kw["pairend"] = 0
    p = B.make_params(**kw)
    ix = B.Index(p, d["gnames"], d["gseqs"])
    mp = B.Mapper(ix, p, max_batch=256, stride=160)
    mh = B.Meth(ix, B.meth_opts())
    mh.enable_mbias()
    mh.set_ignore(0, 0, 3, 0)
    mh.attach(mp, sam_rules=True)
    seqs = R.clip(case, d["seqs_b"])
    buf, lens = B.pack_reads(seqs, stride=160)
    recs, counts = mp.map_se(buf, lens, readset=2)
    hist, _ = mh.mbias()
    txt, _ = mp.format_se(d["names_b"], seqs, d["quals_b"], recs, counts, readset=2)
    sam = tmp_path / "b.sam"
    sam.write_bytes(ix.header() + txt)
    exp, _, _, _ = MB.mbias(d["gnames"], d["gseqs"], [str(sam)], ignore=(0, 0, 3, 0))
    assert hist[0].sum() == 0 and hist[1].sum() > 0 and hist[1][:, :3].sum() == 0
    assert np.array_equal(hist.astype(np.int64), exp)
    BL.check(BL.load().bsx_mapper_attach_meth(mp.h, None, None, 0))
    mh.close(); mp.close(); ix.close()


def _map_in_process(case, max_batch, mbias=True, ignore=None):
    d = case.data()
    p = B.make_params(**case.param_kwargs())
    ix = B.Index(p, d["gnames"], d["gseqs"])
    mp = B.Mapper(ix, p, max_batch=max_batch, stride=160)
    mh = B.Meth(ix, B.meth_opts())
    if mbias:
        mh.enable_mbias()
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


@pytest.mark.parametrize("name", ["se_cfg2_r0_uR", "se_cfg2_bsp", "pe_sam", "pe_readthrough", "rrbs_se_A", "rrbs_pe", "se_cfg5"])
def test_in_process_mbias_equals_the_oracle(tmp_path, name):
    """Mapper + attached Meth, many batches on both streams: histogram == oracle on the text the records format to"""
    case = CS.BY_NAME[name]
    d, ix, mp, mh = _map_in_process(case, max_batch=256)
    hist, over = mh.mbias()
    files = alignment_files(case, str(tmp_path))       # the golden text == what these records format to
    exp, _, counters, _ = MB.mbias(d["gnames"], d["gseqs"], files)
    assert over == 0 and np.array_equal(hist.astype(np.int64), exp)
    m, dp = mh.counters(0)                                 # the device's table agrees with the histogram's marginals
    assert int(hist.sum()) == sum(int(c[1].sum()) for c in counters.values())
    assert np.array_equal(dp, counters[d["gnames"][0]][1]) and np.array_equal(m, counters[d["gnames"][0]][0])
    key = name + ".default"
    if key in MANIFEST:
        got = table_bytes(mh, d["gseqs"], tmp_path)
        assert got == gzip.open(os.path.join(GOLD, key + ".txt.gz"), "rb").read()
    mh.close(); mp.close(); ix.close()


@pytest.mark.parametrize("name", ["se_n1", "pe_sam"])
def test_batch_size_invariance(name):
    """64 and 1 M alignments per batch give the same histogram and table, exclusion on"""
    res = []
    for mb in (64, 1 << 20):
        d, ix, mp, mh = _map_in_process(CS.BY_NAME[name], max_batch=mb, ignore=(1, 2, 3, 4))
        hist, _ = mh.mbias()
        res.append((hist, [mh.counters(k) for k in range(len(d["gnames"]))]))
        mh.close(); mp.close(); ix.close()
    assert np.array_equal(res[0][0], res[1][0]) and res[0][0].sum() > 0
    for (m0, d0), (m1, d1) in zip(res[0][1], res[1][1]):
        assert np.array_equal(m0, m1) and np.array_equal(d0, d1)


@pytest.mark.parametrize("name", ["pe_sam", "se_cfg2_r0_uR"])
def test_bsmap_cli_meth_mbias(tmp_path, name):
    """bsmap --methratio t --meth-mbias f == methratio --mbias on the SAM the same run wrote"""
    case = CS.BY_NAME[name]
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / "out.sam")
    t1, f1, t2, f2 = (str(tmp_path / x) for x in ("t1", "f1", "t2", "f2"))
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--methratio", t1, "--meth-mbias", f1, "--meth-ignore", "1,2,3,4"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([METHRATIO, "-o", t2, "-d", fa, "-q", "--mbias", f2, "--mbias-ignore", "1,2,3,4", o], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(f1, "rb").read() == open(f2, "rb").read() and open(t1, "rb").read() == open(t2, "rb").read()
    assert len(open(f1).read().splitlines()) > 1
    r = subprocess.run([BSMAP] + case.cli(a, b, fa, o) + ["--meth-mbias", f1], capture_output=True, text=True)
    assert r.returncode != 0 and "--methratio" in r.stderr


def test_long_seq_overflow(tmp_path):
    """SEQ past BSX_MBIAS_CYCLES: counted in the table, reported as overflow, warned about by the command line"""
    g = "ACGT" * 200
    fa, sam = tmp_path / "g.fa", tmp_path / "a.sam"
    fa.write_text(">c\n" + g + "\n")
    sam.write_text(sam_line(0, "c", 1, g[:600], "++") + sam_line(0, "c", 5, g[4:100], "++"))
    ix = B.Index.packed(["c"], [g.encode()])
    plain, mh = B.Meth(ix, B.meth_opts()), B.Meth(ix, B.meth_opts())
    mh.enable_mbias()
    cols = api_arrays([str(sam)], ["c"])
    add_all(plain, cols); add_all(mh, cols)
    hist, over = mh.mbias()
    exp, exp_over, _, _ = MB.mbias(["c"], [g.encode()], [str(sam)])
    assert over == exp_over == 22 and np.array_equal(hist.astype(np.int64), exp)
    assert all(np.array_equal(x, y) for x, y in zip(plain.counters(0), mh.counters(0)))
    r = subprocess.run([METHRATIO, "-o", str(tmp_path / "t"), "-d", str(fa), "-q", "--mbias", str(tmp_path / "b"), str(sam)], capture_output=True, text=True)
    assert r.returncode == 0 and "22 methylation calls at cycle 513" in r.stderr, r.stderr
    plain.close(); mh.close(); ix.close()


def test_misuse_is_refused():
    ix = B.Index.packed(["c"], [b"ACGT" * 100])
    mh = B.Meth(ix, B.meth_opts())
    with pytest.raises(B.BsxError, match=">= 0"):
        mh.set_ignore(0, -1, 0, 0)
    with pytest.raises(B.BsxError, match="not enabled"):
        mh.mbias()
    mh.add([b"ACGTACGT"], [0], [0], [0], [0], [0], [4])
    for call in (mh.enable_mbias, lambda: mh.set_ignore(1, 0, 0, 0)):
        with pytest.raises(B.BsxError, match="error 1:.*already piled up"):
            call()
    mh.close(); ix.close()
