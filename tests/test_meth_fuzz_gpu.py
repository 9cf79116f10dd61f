"""Randomised and large-launch differential tests of methratio on the device (bsx_meth.cu) against the composed numpy
oracles, through tests/meth_fuzz.py's generator: fixed-seed rounds; every pile-up instantiation at launch sizes where
each warp of the capped grid loops over several alignments (text and mapped); -r under heavy duplication across many
batches and both in-process streams; more regions than one device slice; the command lines on generated SAM, BSP and
BAM; and SEQ lengths around the 16-bit limit of bsx_meth_add."""
from __future__ import annotations

import os
import subprocess
import sys

import numpy as np
import pytest

import bamio
import meth_fuzz as F
from meth_inputs import api_arrays
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
METHRATIO = os.path.join(BIN, "methratio")
IGNORE = (3, 2, 4, 1)
PLAIN = dict(unique=False, pair=False, meth0=True, combine_cpg=False, rm_dup=False, trim_fillin=2, min_depth=1, chroms=None,
             mbias=False, ignore=None, ct_snp=None, conv=None, regions=None)


def opts(**kw):
    return dict(PLAIN, **kw)


def oracle(names, seqs, files, o, sam_rules=None):
    return CV.conversion(names, seqs, files, threshold=o["conv"] or 0, chroms=o["chroms"], unique=o["unique"], pair=o["pair"],
                         trim_fillin=o["trim_fillin"], combine_cpg=o["combine_cpg"], rm_dup=o["rm_dup"], ignore=o["ignore"] or (0, 0, 0, 0),
                         sam_rules=sam_rules)


def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- randomised rounds ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [21, 22, 23, 24])
def test_meth_fuzz_rounds(seed):
    rng = np.random.default_rng(seed)
    for k in range(4):
        desc, bad = F.one_round(rng, k)
        assert bad is None, f"{desc} -> {bad}"


# ---- launch sizes where warps loop ------------------------------------------------------------------------------------
# (M-bias, exclusion, C/T SNP mode, conversion threshold): every instantiation of the pile-up kernels (plain, Snp,
# Cycles, Cycles + Snp, Conv, Conv + Snp), Cycles and Conv with and without the M-bias histogram
LAUNCH_VARIANTS = [(False, None, None, None), (False, None, "correct", None), (True, None, None, None), (True, None, "skip", None),
                   (False, IGNORE, None, None), (False, None, None, 0), (True, IGNORE, "no-action", 3)]


def launch_opts(v):
    mbias, ignore, ct_snp, conv = v
    return opts(mbias=mbias, ignore=ignore, ct_snp=ct_snp, conv=conv)


def oracle_cached(cache, names, seqs, files, o):
    key = (o["ignore"], o["conv"] or 0)
    if key not in cache:
        cache[key] = oracle(names, seqs, files, o)
    return cache[key]


def test_pileup_at_launch_sizes_where_warps_loop(tmp_path):
    """One bsx_meth_add of more than 4 x 64 x SMs alignments (every warp of the capped grid takes several, and the
    per-CTA histograms gather many before their flush), then the mapped kernels on 2 x 2^16 SE reads and 2^16 pairs
    in batches of 2^16 reads: counters, evidence, M-bias and score histograms == oracle for every instantiation"""
    rng = np.random.default_rng(5)
    g = synth.make_genome(77, [14_000_000, 6_000_000])
    names, seqs = ["chrB", "chrA"], [x.numpy().tobytes() for x in g]
    recs = F.make_records(rng, names, seqs, 60_000, dup_frac=0.02)
    path = str(tmp_path / "a.sam")
    open(path, "w").write(F.sam_text(recs, names, seqs))
    cols = api_arrays([path], names)
    n = len(cols[0])
    assert n > 4 * 64 * sms(), n
    ix = B.Index.packed(names, seqs)
    cache = {}
    for v in LAUNCH_VARIANTS:
        o = launch_opts(v)
        res = oracle_cached(cache, names, seqs, [path], o)
        mh = F.new_meth(B, ix, o)
        mh.add(*cols[:7], read2=cols[7])
        bad = F.compare_counters(mh, names, o, res)
        assert bad is None, (v, bad)
        mh.close()
    ix.close()

    # the mapped kernels: reads simulated on the same genome, mapped with Meth attached; the oracle reads the SAM text
    # the same records format to
    p_se, p_pe = B.make_params(), B.make_params(pairend=1, m=28, x=500)
    sim = synth.simulate_reads(g, 1 << 17, 100, seed=9, conv=0.9)
    se = [bytes(r) for r in sim["seq"].numpy()]
    simp = synth.simulate_pairs(g, 1 << 16, 100, seed=10, conv=0.9)
    pa, pb = [bytes(r) for r in simp["seq1"].numpy()], [bytes(r) for r in simp["seq2"].numpy()]
    for pe, p in ((False, p_se), (True, p_pe)):
        ix = B.Index(p, names, seqs)
        sam = str(tmp_path / ("pe.sam" if pe else "se.sam"))
        cache = {}
        for v in LAUNCH_VARIANTS:
            if v[1] and not v[3]:
                continue                                               # exclusion alone: the same instantiation as M-bias
            o = launch_opts(v)
            mp = B.Mapper(ix, p, max_batch=1 << 16, stride=160)
            mh = F.new_meth(B, ix, o)
            mh.attach(mp, sam_rules=True)
            if not pe:
                buf, lens = B.pack_reads(se, stride=160)
                recs_, counts = mp.map_se(buf, lens)
                if not cache:
                    txt, _ = mp.format_se(["s%d" % i for i in range(len(se))], se, [b"I" * len(s) for s in se], recs_, counts)
            else:
                ba, la = B.pack_reads(pa, stride=160)
                bb, lb = B.pack_reads(pb, stride=160)
                pr, ra, rb, ca, cb = mp.map_pe(ba, la, bb, lb)
                if not cache:
                    q = [b"I" * len(s) for s in pa]
                    txt, _, _ = mp.format_pe(["p%d" % i for i in range(len(pa))], pa, q, ["p%d" % i for i in range(len(pb))], pb, q, pr, ra, rb, ca, cb)
            if not cache:
                open(sam, "wb").write(txt)
            res = oracle_cached(cache, names, seqs, [sam], o)
            assert res["valid"] > 4 * 64 * sms()
            bad = F.compare_counters(mh, names, o, res)
            assert bad is None, (pe, v, bad)
            mh.close(); mp.close()
        ix.close()


# ---- -r under heavy duplication ---------------------------------------------------------------------------------------
def test_rm_dup_under_heavy_duplication(tmp_path):
    """~100k alignments, about half of them duplicates, a few keys claimed by thousands: through Meth.add in batches of
    1 (the first 3000), 7 and 257, and in-process with 257 reads per batch (hundreds of batches alternating between the
    two streams): counters == oracle, the same for every batching"""
    rng = np.random.default_rng(8)
    names, seqs = ["d1", "d0"], [x.numpy().tobytes() for x in synth.make_genome(3, [700_000, 300_000])]
    base = F.make_records(rng, names, seqs, 50_000, dup_frac=0.0)
    hot = [base[int(i)] for i in rng.integers(0, len(base), 5)]
    dups = []
    for i in range(50_000):
        r = dict(hot[i % 5] if i % 10 < 3 else base[int(rng.integers(0, len(base)))])
        if i % 2 and r["seq"] != "*":                                  # shared fragment end, another read
            r["seq"] = r["seq"][::-1]
        dups.append(r)
    recs = base + dups
    order = rng.permutation(len(recs))
    recs = [recs[int(i)] for i in order]
    size = dict(zip(names, (len(s) for s in seqs)))
    recs = [r for r in recs if r["chrom"] not in size or (r["pos"] + len(r["seq"]) if r["strand"] in ("+-", "-+") else r["pos"]) < size[r["chrom"]]]
    path = str(tmp_path / "a.sam")
    open(path, "w").write(F.sam_text(recs, names, seqs))
    o = opts(rm_dup=True, ct_snp="no-action", mbias=True, conv=0)
    res = oracle(names, seqs, [path], o)
    assert sum(s is None for s in res["scores"][0]) > 40_000              # -r losers
    cols = api_arrays([path], names)
    n = len(cols[0])
    ix = B.Index.packed(names, seqs)
    for cuts in (list(range(0, 3001)) + [n], list(range(0, n, 7)) + [n], list(range(0, n, 257)) + [n]):
        mh = F.new_meth(B, ix, o)
        for b, e in zip(cuts, cuts[1:]):
            mh.add(*[c[b:e] for c in cols[:7]], read2=cols[7][b:e])
        assert F.compare_counters(mh, names, o, res) is None, len(cuts)
        mh.close()
    ix.close()

    # in-process: 20k simulated reads, each repeated 1-9 times (identical reads map to the same key), 257 per batch
    g = synth.make_genome(4, [400_000])
    sim = synth.simulate_reads(g, 20_000, 90, seed=5, conv=0.9)
    uniq = [bytes(r) for r in sim["seq"].numpy()]
    reads = [uniq[int(i)] for i in np.repeat(np.arange(len(uniq)), rng.integers(1, 10, len(uniq)))]
    reads = [reads[int(i)] for i in rng.permutation(len(reads))]
    p = B.make_params()
    ix = B.Index(p, ["chr1"], [g[0].numpy().tobytes()])
    for mb in (257, 1 << 20):
        mp = B.Mapper(ix, p, max_batch=mb, stride=160)
        mh = F.new_meth(B, ix, o)
        mh.attach(mp)
        buf, lens = B.pack_reads(reads, stride=160)
        recs_, counts = mp.map_se(buf, lens)
        if mb == 257:
            txt, _ = mp.format_se(["r%d" % i for i in range(len(reads))], reads, [b"I" * len(s) for s in reads], recs_, counts)
            sam = str(tmp_path / "ip.sam")
            open(sam, "wb").write(txt)
            res = oracle(["chr1"], [g[0].numpy().tobytes()], [sam], o)
            assert sum(s is None for s in res["scores"][0]) > len(reads) // 3
        assert F.compare_counters(mh, ["chr1"], o, res) is None, mb
        mh.close(); mp.close()
    ix.close()


# ---- more regions than one slice --------------------------------------------------------------------------------------
def test_regions_past_one_slice(tmp_path):
    """1 bp tiles and a random BED of more than 2^20 regions over a 1.5 Mb genome: Meth.regions, Meth.write_regions and
    methratio --tiles 1 == region_oracle"""
    rng = np.random.default_rng(12)
    names, seqs = ["r2", "r1"], [x.numpy().tobytes() for x in synth.make_genome(12, [1_100_000, 400_000])]
    recs = F.make_records(rng, names, seqs, 30_000, dup_frac=0.0)
    path, fa = str(tmp_path / "a.sam"), str(tmp_path / "g.fa")
    open(path, "w").write(F.sam_text(recs, names, seqs))
    F.write_fasta(fa, names, seqs)
    o = opts(ct_snp="skip", combine_cpg=True, min_depth=2)
    res = oracle(names, seqs, [path], o)
    lengths = dict(zip(names, (len(s) for s in seqs)))
    tiles = RO.tiles(lengths, 1)
    bed = random_regions(lengths, (1 << 20) + 5000, seed=3)
    assert len(tiles) > 1 << 20 and len(bed) > 1 << 20
    cols = api_arrays([path], names)
    ix = B.Index.packed(names, seqs)
    mh = F.new_meth(B, ix, o)
    mh.add(*cols[:7], read2=cols[7])
    idx = {x: i for i, x in enumerate(names)}
    for regs in (tiles, bed):
        exp = RO.regions(res["counters"], res["ref"], regs, combine_cpg=True, min_depth=2, ct_snp="skip")
        assert exp[:, :, 1].sum() > 0
        ci, st, en = [idx[c] for c, _, _ in regs], [s for _, s, _ in regs], [e for _, _, e in regs]
        assert F.first_diff("region sums", mh.regions(ci, st, en), exp) is None
        if regs is tiles:
            text = RO.report_text(regs, exp)
            assert F.read_fd(lambda fd: mh.write_regions(fd, ci, st, en))[1] == text
    mh.close(); ix.close()
    rep = str(tmp_path / "rep")
    r = subprocess.run([METHRATIO, "-o", str(tmp_path / "t"), "-d", fa, "-q", "-g", "-m", "2", "--ct-snp", "skip", "--region-report", rep,
                        "--tiles", "1", path], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(rep).read() == text


# ---- the command lines on generated inputs ----------------------------------------------------------------------------
def cli_args(o, td, fa, kind):
    a = ["-d", fa, "-q", "-t", str(o["trim_fillin"]), "-m", str(o["min_depth"])]
    a += [f for f, on in (("-u", o["unique"]), ("-p", o["pair"]), ("-z", o["meth0"]), ("-r", o["rm_dup"]), ("-g", o["combine_cpg"])) if on]
    if o["chroms"]:
        a += ["-c", ",".join(o["chroms"])]
    if o["mbias"]:
        a += ["--mbias", os.path.join(td, kind + ".mbias")]
    if o["ignore"]:
        a += ["--mbias-ignore", ",".join(map(str, o["ignore"]))]
    if o["ct_snp"]:
        a += ["--ct-snp", o["ct_snp"]]
    if o["conv"] is not None:
        a += ["--conversion-filter", str(o["conv"]), "--conversion-report", os.path.join(td, kind + ".conv")]
    if o["regions"] is not None:
        a += ["--region-report", os.path.join(td, kind + ".reg")]
        if o["regions"][0] == "tiles":
            a += ["--tiles", str(o["regions"][1])]
        else:
            bed = os.path.join(td, "r.bed")
            open(bed, "w").write("".join("%s\t%d\t%d\n" % r for r in o["regions"][1]) + F.UNKNOWN + "\t0\t10\n")
            a += ["--regions", bed]
    return a


@pytest.mark.parametrize("seed", [31, 32, 33])
def test_cli_on_fuzz_inputs(tmp_path, seed):
    """methratio on a generated round written as SAM (FLAG partly as samtools view -X letters), BSP and BAM, with the
    round's options: table, summary, M-bias, conversion and region reports byte-equal to the oracle's texts"""
    rng = np.random.default_rng(seed)
    names, seqs = F.make_reference(rng)
    o = F.draw_options(rng, names, seqs, True)
    recs = F.make_records(rng, names, seqs, 1500, rm_dup=o["rm_dup"])
    td = str(tmp_path)
    fa = os.path.join(td, "g.fa")
    F.write_fasta(fa, names, seqs)
    numeric = F.sam_text(recs, names, seqs)
    files = {"sam": os.path.join(td, "a.sam"), "bsp": os.path.join(td, "a.bsp"), "bam": os.path.join(td, "a.bam")}
    open(files["sam"], "w").write(F.sam_text(recs, names, seqs, letters=list(rng.random(len(recs)) < 0.5)))
    open(files["bsp"], "w").write(F.bsp_text(recs))
    bamio.aligned_bam_from_sam(files["bam"], numeric, extra_names=[F.UNKNOWN])
    ofiles = {"sam": os.path.join(td, "o.sam"), "bsp": files["bsp"], "bam": os.path.join(td, "ob.sam")}
    open(ofiles["sam"], "w").write(numeric)
    open(ofiles["bam"], "w").write(bamio.bam_to_sam_text(files["bam"]))
    for kind in ("sam", "bsp", "bam"):
        ok = o if kind != "bsp" else dict(o, mbias=False, ignore=None)       # BSP records carry no read number
        e = F.expected(names, seqs, [ofiles[kind]], ok)
        out = os.path.join(td, kind + ".txt")
        r = subprocess.run([METHRATIO, "-o", out] + cli_args(ok, td, fa, kind) + [files[kind]], capture_output=True, text=True)
        assert r.returncode == 0, (kind, r.stderr)
        assert F.first_diff(kind + " table", open(out).read(), e["table"]) is None
        assert r.stdout.strip() == e["summary"], kind
        if ok["mbias"]:
            assert open(os.path.join(td, kind + ".mbias")).read() == e["mbias_text"], kind
        if ok["conv"] is not None:
            assert open(os.path.join(td, kind + ".conv")).read() == e["conv_text"], kind
            assert e["conv_line"] in r.stderr.splitlines(), kind
        if ok["regions"] is not None:
            assert F.first_diff(kind + " regions", open(os.path.join(td, kind + ".reg")).read(), e["region_text"]) is None


# ---- SEQ lengths at the 16-bit limit ----------------------------------------------------------------------------------
@pytest.mark.parametrize("length", [65_535, 65_536, 70_000])
def test_long_reads(tmp_path, length):
    """a SAM / BAM record of 65,535 bases is counted exactly; a longer one is either counted exactly or refused with an
    error naming the file (exit status 1), never piled up cut short; Meth.add refuses it"""
    rng = np.random.default_rng(length)
    names, seqs = ["big"], [synth.make_genome(6, [200_000])[0].numpy().tobytes()]
    recs = F.make_records(rng, names, seqs, 50, dup_frac=0.0)
    recs.append(dict(qname="long", flag=0, chrom="big", pos=1000, strand="++", insert=0, pnext=0,
                     seq=F.read_at(rng, seqs[0], 1000, length, "++", 0.5, [])))
    recs.append(dict(qname="long2", flag=0x10, chrom="big", pos=2000, strand="-+", insert=0, pnext=0,
                     seq=F.read_at(rng, seqs[0], 2000, length, "-+", 0.5, [])))
    td = str(tmp_path)
    fa, sam, bam = (os.path.join(td, x) for x in ("g.fa", "a.sam", "a.bam"))
    F.write_fasta(fa, names, seqs)
    text = F.sam_text(recs, names, seqs)
    open(sam, "w").write(text)
    bamio.aligned_bam_from_sam(bam, text, extra_names=[F.UNKNOWN])
    o = opts(meth0=True, trim_fillin=0)
    e = F.expected(names, seqs, [sam], o)
    bam_text = os.path.join(td, "b.sam")                                 # BAM keeps no lowercase: its own oracle text
    open(bam_text, "w").write(bamio.bam_to_sam_text(bam))
    for f, ef in ((sam, e), (bam, F.expected(names, seqs, [bam_text], o))):
        out = os.path.join(td, "t.txt")
        r = subprocess.run([METHRATIO, "-o", out, "-d", fa, "-q", "-z", "-t", "0", f], capture_output=True, text=True)
        if length <= 65_535:
            assert r.returncode == 0, r.stderr
        if r.returncode == 0:
            assert open(out).read() == ef["table"] and r.stdout.strip() == ef["summary"], f
        else:
            assert r.returncode == 1 and f in r.stderr and "longer than 65535" in r.stderr, r.stderr
    ix = B.Index.packed(names, seqs)
    mh = F.new_meth(B, ix, o)
    cols = api_arrays([sam], names)
    if length <= 65_535:
        mh.add(*cols[:7], read2=cols[7])
        assert F.compare_counters(mh, names, o, e["res"]) is None
    else:
        with pytest.raises(ValueError, match="at most 65535"):
            mh.add(*cols[:7], read2=cols[7])
    mh.close(); ix.close()


# ---- known answers from the generated rounds ----------------------------------------------------------------------------
def test_table_context_of_short_sequences(tmp_path):
    """the context column is refcr[i-2:i+3] with Python's slice rules: at i < 2 of a sequence of 4 bases or fewer the
    negative start counts from the end (found by the fuzz rounds: the writer printed nothing there)"""
    names, seqs = ["s1", "s3", "s4", "s5"], [b"C", b"CGa", b"GCCG", b"CCAGG"]
    recs = [dict(qname="r%d" % i, flag=0, chrom=n, pos=0, strand=st, insert=0, pnext=0, seq=s.decode().upper())
            for i, (n, s) in enumerate(zip(names, seqs)) for st in ("++", "-+")]
    path = str(tmp_path / "a.sam")
    open(path, "w").write(F.sam_text(recs, names, seqs))
    o = opts(meth0=True, trim_fillin=0)
    e = F.expected(names, seqs, [path], o)
    assert "s3\t1\t+\tGA\t" in e["table"] and "s4\t2\t+\tG\t" in e["table"] and "s5\t1\t+\t\t" in e["table"]
    assert F.device_check(B, names, seqs, [path], o, e, cuts=[0, len(recs)]) is None


def test_lettered_flag_that_starts_with_a_digit(tmp_path):
    """samtools view -X letters put '1' (0x40) and '2' (0x80) before 's' (0x100): "2s" is a secondary read 2, not FLAG 2
    (found by the fuzz rounds: methratio read it as a number)"""
    names, seqs = ["c"], [b"ACGTTCGACG" * 20]
    fa = str(tmp_path / "g.fa")
    F.write_fasta(fa, names, seqs)
    body = "".join("%s\t%s\tc\t%d\t255\t10M\t*\t0\t0\tACGTTTGACG\tIIIIIIIIII\tZS:Z:++\n" % (q, f, p) for q, f, p in
                   (("a", "2s", 1), ("b", "1s", 11), ("c", "pP1", 21), ("d", "0", 31)))
    sam = str(tmp_path / "a.sam")
    open(sam, "w").write(body)
    for args, covered in (([], [1, 11, 21, 31]), (["-u"], [21, 31]), (["-p"], [21])):
        out = str(tmp_path / "t")
        r = subprocess.run([METHRATIO, "-o", out, "-d", fa, "-q", "-z", "-t", "0"] + args + [sam], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        starts = sorted({int(x.split("\t")[1]) // 10 * 10 + 1 for x in open(out).read().splitlines()[1:]})
        assert starts == covered, (args, starts)
