"""GPU parity tests (run on the B200 box with `-m gpu`): the CUDA path, called through the C ABI,
against the oracle restatement on the same inputs and against the committed golden outputs of the
unmodified reference.  Bit-exact: every index word, every record field, every output byte."""
import os
import subprocess

import numpy as np
import pytest

import cases as CS
import oracle_lib as O
import runners as R

import bsmap_b200 as B
from bsmap_b200 import lib as BL

pytestmark = pytest.mark.gpu


def _have_gpu():
    try:
        return BL.load().bsx_device_count() > 0
    except Exception:
        return False


@pytest.fixture(scope="module", autouse=True)
def _require_gpu():
    if not _have_gpu():
        pytest.fail("no CUDA device / libbsmap_b200.so missing: the product path has no CPU fallback")


def _diff_arrays(name, got, exp, limit=5):
    if got.shape != exp.shape:
        return f"{name}: shape {got.shape} vs {exp.shape}"
    bad = np.nonzero(got != exp)[0]
    if bad.size == 0:
        return None
    rows = ", ".join(f"[{i}] got {got[i]} exp {exp[i]}" for i in bad[:limit])
    return f"{name}: {bad.size} of {got.size} differ; first: {rows}"


INDEX_CASES = ["se_cfg1", "se_mixed_A", "se_cfg5", "se_I16_s10", "se_mixed_fa", "rrbs_se_A", "rrbs_pe"]


@pytest.mark.parametrize("name", INDEX_CASES)
def test_index_matches_oracle(name):
    """K0/K1: packed strands, anchors, CSR table and every position list (order included)"""
    case = CS.BY_NAME[name]
    d = case.data()
    kw = case.param_kwargs()
    po, pb = O.make_params(**kw), B.make_params(**kw)
    oref = O.OracleRef(po, d["gnames"], d["gseqs"])
    ix = B.Index(pb, d["gnames"], d["gseqs"])
    info = ix.info
    assert (info.n_words, info.n_keys, info.n_entries) == (oref.n_words, oref.n_keys, oref.n_entries)
    f, c = np.array(oref.refcat).astype(np.uint64), np.array(oref.crefcat).astype(np.uint64)

    def window(coord, strand):
        w, sh = coord >> 4, ((coord & 15) * 2).astype(np.uint64)
        lo_f, hi_f = f[w + 1], f[w]; lo_c, hi_c = c[w + 1], c[w]
        hi, lo = np.where(strand, hi_c, hi_f), np.where(strand, lo_c, lo_f)
        return ((((hi << np.uint64(32)) | lo) << sh) >> np.uint64(32)) & np.uint64(0xffffffff)

    s_ = 12 if kw.get("D") else kw.get("s", 16)   # -D forces seed 12 (param.cpp:95-106)
    for what in ("refcat", "crefcat", "anchor"):
        msg = _diff_arrays(what, ix.download(what), np.array(getattr(oref, what)))
        assert msg is None, msg
    tab, pos = np.array(oref.tab).astype(np.int64), np.array(oref.pos).astype(np.int64)
    if kw.get("D"):
        # RRBS: every list of the reference, stably partitioned by its (segment, mirrored) tag -- the entries one
        # SnpAlign call does not skip become contiguous, in the reference's order -- and a CSR over (key, group)
        tag = np.array(oref.pos_tag).astype(np.int64)
        G = 2 * (144 // s_)
        key = np.repeat(np.arange(info.n_keys, dtype=np.int64), tab[2::2] - tab[0:-1:2])
        comp = key * G + 2 * ((tag >> 16) & 0xff) + (tag >> 24)
        order = np.argsort(comp, kind="stable")
        exp_tab = np.concatenate([[0], np.cumsum(np.bincount(comp, minlength=int(info.n_keys) * G))])
        assert info.n_tab == len(exp_tab)
        for what, exp in (("tab", exp_tab), ("pos", pos[order]), ("tag", tag[order])):
            msg = _diff_arrays(what, ix.download(what), exp.astype(np.uint32))
            assert msg is None, msg
        chr_ = tag[order] & 0xffff
        coord, strand = np.array(oref.anchor).astype(np.int64)[chr_ >> 1] + pos[order], (chr_ & 1).astype(bool)
    else:
        for what in ("tab", "pos"):
            msg = _diff_arrays(what, ix.download(what), np.array(getattr(oref, what)))
            assert msg is None, msg
        strand = np.zeros(len(pos) + 1, dtype=np.int64)
        np.add.at(strand, tab[1::2], 1); np.add.at(strand, tab[2::2], -1)
        strand = np.cumsum(strand)[:-1] > 0
        coord = pos
    # inline context: the 16 reference bases before / after every entry's seed, on the entry's strand
    wide = not kw.get("D") and kw.get("v", 2) >= 8     # built for high -v: 16-byte entries, the next 16 bases outwards as well
    assert info.ctx_words == (4 if wide else 2)
    ctx = ix.download("ctx").reshape(-1, info.ctx_words)
    inner = ctx[:, 1:3] if wide else ctx
    assert np.array_equal(inner[:, 0].astype(np.uint64), window(coord - 16, strand)), "ctx.before differs"
    assert np.array_equal(inner[:, 1].astype(np.uint64), window(coord + s_, strand)), "ctx.after differs"
    if wide:
        assert np.array_equal(ctx[:, 0].astype(np.uint64), window(coord - 32, strand)), "outer ctx.before differs"
        assert np.array_equal(ctx[:, 3].astype(np.uint64), window(coord + s_ + 16, strand)), "outer ctx.after differs"
    ix.close(); oref.close()


def test_index_of_a_long_masked_sequence():
    """UnmaskRegion on a sequence long enough for the piecewise host scan (bsx_index.cu: pieces of >= 1 Mb stitched in order):
    N / X runs, IUPAC letters that neither start nor end a block, lower case, islands shorter than 30 nt, runs across
    piece borders, a block that reaches the sequence end -- table and every list equal the oracle's"""
    rng = np.random.default_rng(5)
    L = 5_300_000
    g = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, L)].copy()
    lower = rng.random(L) < 0.05
    g[lower] += 32
    for _ in range(4000):                                    # masked runs of every length, some back to back
        b, n = int(rng.integers(0, L)), int(rng.choice([1, 2, 5, 29, 30, 31, 200, 5000]))
        g[b:b + n] = rng.choice(np.frombuffer(b"NXnx", dtype=np.uint8))
    for _ in range(3000):                                    # letters of class 0: inside a block they continue it, outside they do not start one
        b, n = int(rng.integers(0, L)), int(rng.integers(1, 40))
        g[b:b + n] = rng.choice(np.frombuffer(b"RYKMryBD-", dtype=np.uint8))
    for piece in range(1, 20):                               # runs straddling the borders of the scan pieces (any thread count up to 64)
        for parts in (4, 8, 16, 20, 32, 64, 128, 256):
            q = L * piece // parts
            if 0 < q < L - 50:
                g[q - 3:q + 4] = ord("N") if piece % 2 else ord("R")
    g[:40] = ord("N"); g[-100:] = np.frombuffer(b"ACGT" * 25, dtype=np.uint8)
    names, seqs = ["long", "short"], [g.tobytes(), (b"ACGTTGCA" * 40) + b"N" * 7 + (b"GATTACA" * 30)]
    kw = dict(s=12, I=4)
    oref = O.OracleRef(O.make_params(**kw), names, seqs)
    ix = B.Index(B.make_params(**kw), names, seqs)
    assert (ix.info.n_words, ix.info.n_entries) == (oref.n_words, oref.n_entries)
    for what in ("refcat", "crefcat", "anchor", "tab", "pos"):
        msg = _diff_arrays(what, ix.download(what), np.array(getattr(oref, what)))
        assert msg is None, msg
    ix.close(); oref.close()


def _run_gpu(case, max_batch=4096, stride=160):
    d = case.data()
    p = B.make_params(**case.param_kwargs())
    ix = B.Index(p, d["gnames"], d["gseqs"])
    mp = B.Mapper(ix, p, max_batch=max_batch, stride=stride)
    out = {}
    head = ix.header() if p.out_sam else b""
    if not case.paired:
        buf, lens = B.pack_reads(R.clip(case, d["seqs"]), stride=stride)
        recs, counts = mp.map_se(buf, lens)
        txt, na = mp.format_se(d["names"], d["seqs"], R.case_quals(case), recs, counts)
        out.update(main=head + txt, unpair=b"", recs=recs, counts=counts, n_aligned=na)
    else:
        ba, la = B.pack_reads(R.clip(case, d["seqs"]), stride=stride)
        bb, lb = B.pack_reads(R.clip(case, d["seqs_b"]), stride=stride)
        pr, ra, rb, ca, cb = mp.map_pe(ba, la, bb, lb)
        txt, un, st = mp.format_pe(d["names"], d["seqs"], d["quals"], d["names_b"], d["seqs_b"], d["quals_b"], pr, ra, rb, ca, cb)
        out.update(main=head + txt, unpair=un, pr=pr, ra=ra, rb=rb, ca=ca, cb=cb, n_aligned=st)
    out["stats"] = mp.stats()
    out["launches"] = mp.launches
    mp.close(); ix.close()
    return out


@pytest.mark.parametrize("name", ["se_cfg2_r0_uR", "pe_sam", "se_n1"])
def test_read_stride_is_only_8_byte_aligned(name):
    """100-nt reads in 104-byte slots (the bench layout): same records and text as in 160-byte slots"""
    case = CS.BY_NAME[name]
    a, b = _run_gpu(case), _run_gpu(case, stride=104)
    assert a["main"] == b["main"] and a["unpair"] == b["unpair"]
    assert a["main"] == R.golden_load(case)[0]
    with pytest.raises(B.BsxError, match="multiple of 8"):
        B.Mapper(B.Index(B.make_params(), ["c"], [b"ACGT" * 100]), B.make_params(), max_batch=4, stride=100)


@pytest.mark.parametrize("name", [c.name for c in CS.CASES])
def test_packed_read_input_gives_the_same_records(name):
    """bsx_map_se_packed / bsx_map_pe_packed (2-bit bases + valid mask, 40 bytes per 100-nt slot) == the ASCII entry
    points on every parity case: adapters, RRBS remnants, N-rich and short reads, -n 1, paired ends.  Cases whose reads
    hold lower-case bases while adapters are trimmed are the documented exception (the reference compares case-sensitively)."""
    case = CS.BY_NAME[name]
    d = case.data()
    p = B.make_params(**case.param_kwargs())
    ix = B.Index(p, d["gnames"], d["gseqs"])
    mp = B.Mapper(ix, p, max_batch=1024, stride=152)
    bufs = [B.pack_reads(R.clip(case, d[k]), stride=152) for k in (("seqs", "seqs_b") if case.paired else ("seqs",))]
    packed = [B.pack_reads_2bit(b, l) for b, l in bufs]
    assert packed[0][0].shape[1] == 60      # 38 + 19 bytes rounded up to a multiple of 4
    lower = sum(x[1] for x in packed)
    if lower and p.n_adapter:
        mp.close(); ix.close()
        pytest.skip(f"{lower} lower-case bases with adapter trimming: the ASCII entry point is the exact one")
    if not case.paired:
        a = mp.map_se(*bufs[0])
        b = mp.map_se_packed(packed[0][0], bufs[0][1])
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    else:
        a = mp.map_pe(bufs[0][0], bufs[0][1], bufs[1][0], bufs[1][1])
        b = mp.map_pe_packed(packed[0][0], bufs[0][1], packed[1][0], bufs[1][1])
        for nm, x, y in zip(("pairs", "recs_a", "recs_b", "counts_a", "counts_b"), a, b):
            bad = np.nonzero(x != y)[0]
            assert bad.size == 0, f"{nm}: {bad.size} differ; first idx {bad[0]}: ascii {x[bad[0]]} packed {y[bad[0]]}"
    mp.close(); ix.close()


def test_packed_input_refuses_what_it_cannot_compare():
    p = B.make_params(A=["AGATCGGAAGAGCNNN"])
    ix = B.Index(p, ["c"], [b"ACGTTGCA" * 200])
    mp = B.Mapper(ix, p, max_batch=8, stride=64)
    buf, lens = B.pack_reads([b"ACGTTGCA" * 6], stride=64)
    pk, _ = B.pack_reads_2bit(buf, lens)
    with pytest.raises(B.BsxError, match="upper-case ACGT adapters"):
        mp.map_se_packed(pk, lens)
    mp.close(); ix.close()


def _rec_diff(name, got, exp, reads=None):
    for f in exp.dtype.names:
        bad = np.nonzero(got[f] != exp[f])[0]
        if bad.size:
            i = int(bad[0])
            extra = f" read={reads[i][:60]!r}" if reads else ""
            return f"{name}.{f}: {bad.size} reads differ; first idx {i}: got {got[i]} exp {exp[i]}{extra}"
    return None


SE_CASES = [c for c in CS.CASES if not c.paired]
PE_CASES = [c for c in CS.CASES if c.paired]


@pytest.mark.parametrize("case", SE_CASES, ids=lambda c: c.name)
def test_se_matches_oracle_and_reference(case):
    got = _run_gpu(case)
    exp = R.oracle_run(case)
    msg = _rec_diff("rec", got["recs"], exp["recs"], case.data()["seqs"])
    assert msg is None, msg
    assert np.array_equal(got["counts"], exp["counts"]), "per-level hit counts differ"
    exp_main, _ = R.golden_load(case)
    assert got["main"] == exp_main, R.first_diff(got["main"], exp_main)
    # work counters: C (candidates the reference semantics extend) and P (distinct headers) are
    # functions of the input, so the kernel's own counts must equal the oracle's
    assert got["stats"]["candidates"] == int(exp["stats"][0]), (got["stats"], exp["stats"])
    # P: the kernel reads every header the selection COULD touch once; the reference touches a subset
    assert int(exp["stats"][1]) <= got["stats"]["probes"] <= int(exp["stats"][2]) + len(case.data()["seqs"]), (got["stats"], exp["stats"])
    assert got["launches"] >= 1


@pytest.mark.parametrize("case", PE_CASES, ids=lambda c: c.name)
def test_pe_matches_oracle_and_reference(case):
    got = _run_gpu(case)
    exp = R.oracle_run(case)
    for k in ("pr", "ra", "rb"):
        msg = _rec_diff(k, got[k], exp[k])
        assert msg is None, msg
    assert np.array_equal(got["ca"], exp["ca"]) and np.array_equal(got["cb"], exp["cb"])
    exp_main, exp_un = R.golden_load(case)
    assert got["main"] == exp_main, R.first_diff(got["main"], exp_main)
    assert got["unpair"] == exp_un, R.first_diff(got["unpair"], exp_un)


def test_batching_is_invisible():
    """sub-batch pipelining (two slots / streams) must not change any record"""
    case = CS.BY_NAME["se_cfg2_r0_uR"]
    a = _run_gpu(case, max_batch=1 << 16)
    b = _run_gpu(case, max_batch=257)
    assert np.array_equal(a["recs"], b["recs"]) and a["main"] == b["main"]
    n = len(case.data()["seqs"])
    first = 257 // 8                      # the host pipeline opens with a small sub-batch (bsx_api.cu::map_host)
    assert b["launches"] == 1 + -(-(n - first) // 257)


def test_empty_and_ragged_batches():
    case = CS.BY_NAME["se_cfg1"]
    d = case.data()
    p = B.make_params(**case.param_kwargs())
    ix = B.Index(p, d["gnames"], d["gseqs"])
    mp = B.Mapper(ix, p, max_batch=64, stride=160)
    buf, lens = B.pack_reads([], stride=160)
    recs, _ = mp.map_se(buf.reshape(0, 160), lens)
    assert len(recs) == 0
    # zero-length, 1-nt and over-long (truncated to 144) reads, next to ordinary ones
    seqs = [b"", b"A", b"ACGT" * 50] + d["seqs"][:29]
    buf, lens = B.pack_reads(seqs, stride=208)
    mp2 = B.Mapper(ix, p, max_batch=64, stride=208)
    recs, counts = mp2.map_se(buf, lens)
    assert list(recs["status"][:2]) == [1, 1] and recs["len"][2] == 144
    oref = O.OracleRef(O.make_params(**case.param_kwargs()), d["gnames"], d["gseqs"])
    obuf, olens = O.pack_reads(seqs, stride=208)
    orec, ocnt, _ = oref.map_se(obuf, olens)
    msg = _rec_diff("rec", recs, orec, seqs)
    assert msg is None, msg
    assert np.array_equal(counts, ocnt)
    mp.close(); mp2.close(); ix.close(); oref.close()


def test_mapper_with_less_shared_memory_does_not_break_an_earlier_mapper():
    """The kernels' dynamic shared-memory limit belongs to (kernel, device), not to a mapper: creating and running a
    mapper that needs less (-v 0 on a wide -v 12 index) must not leave the earlier mapper unable to launch."""
    from bsmap_b200 import synth
    g = synth.make_genome(12, [150_000, 90_000])
    names, gseqs = ["chr1", "chr2"], [x.numpy().tobytes() for x in g]
    sim = synth.simulate_pairs(g, 2000, 100, seed=12, subs="cfg1")
    buf_a, lens_a = B.pack_reads([bytes(r) for r in sim["seq1"].numpy()], stride=160)
    buf_b, lens_b = B.pack_reads([bytes(r) for r in sim["seq2"].numpy()], stride=160)
    ix = B.Index(B.make_params(s=12, I=4, v=12), names, gseqs)
    assert ix.info.ctx_words == 4                    # 16-byte context entries: the wide kernels
    # single-end
    a = B.Mapper(ix, B.make_params(s=12, I=4, v=12), max_batch=4096, stride=160)
    first, _ = a.map_se(buf_a, lens_a)
    b = B.Mapper(ix, B.make_params(s=12, I=4, v=0), max_batch=4096, stride=160)
    b.map_se(buf_a, lens_a)
    again, _ = a.map_se(buf_a, lens_a)
    assert np.array_equal(first, again)
    assert (first["nhits"] > 0).mean() > 0.9
    # paired-end
    pa = B.Mapper(ix, B.make_params(s=12, I=4, v=12, pairend=1), max_batch=4096, stride=160)
    first = pa.map_pe(buf_a, lens_a, buf_b, lens_b)
    pb = B.Mapper(ix, B.make_params(s=12, I=4, v=0, pairend=1), max_batch=4096, stride=160)
    pb.map_pe(buf_a, lens_a, buf_b, lens_b)
    again = pa.map_pe(buf_a, lens_a, buf_b, lens_b)
    for x, y in zip(first, again):
        assert np.array_equal(x, y)
    assert (first[0]["paired"] > 0).mean() > 0.9
    for m in (a, b, pa, pb):
        m.close()
    ix.close()


@pytest.mark.parametrize("L,opts,n_reads", [
    (100, dict(s=16, v=5, I=4, S=13), 60000),
    (50, dict(s=16, v=2, I=4, S=13), 60000),
])
def test_larger_random_workload_matches_oracle(L, opts, n_reads):
    """20 Mb genome: lists are long enough that chunks of 32 candidates, threshold lowering and
    early exits all occur many times"""
    import torch
    from bsmap_b200 import synth
    g = synth.make_genome(5, [4_000_000] * 5)
    g = synth.plant_repeats(g, 5, unit_len=250, copies=300)
    sim = synth.simulate_reads(g, n_reads, L, seed=99, subs="cfg2" if L == 100 else "cfg1")
    names = [f"chr{i + 1}" for i in range(5)]
    gb = [x.numpy().tobytes() for x in g]
    seqs = [bytes(r) for r in sim["seq"].numpy()]
    kw = dict(s=opts["s"], v=opts["v"], I=opts["I"], S=opts["S"])
    oref = O.OracleRef(O.make_params(**kw), names, gb)
    obuf, olens = O.pack_reads(seqs)
    orec, ocnt, ostats = oref.map_se(obuf, olens)
    p = B.make_params(**kw)
    ix = B.Index(p, names, gb)
    mp = B.Mapper(ix, p, max_batch=1 << 15, stride=112)
    buf, lens = B.pack_reads(seqs, stride=112)
    recs, counts = mp.map_se(buf, lens)
    msg = _rec_diff("rec", recs, orec, seqs)
    assert msg is None, msg
    assert np.array_equal(counts, ocnt)
    st = mp.stats()
    assert st["candidates"] == int(ostats[0]) and int(ostats[1]) <= st["probes"] <= 1.35 * int(ostats[1]), (st, ostats)
    assert (recs["nhits"] > 0).mean() > 0.9
    mp.close(); ix.close(); oref.close()


def test_packed_reference_cache_rebuilds_the_same_index(tmp_path):
    """bsx_index_save_packed / bsx_index_create_from_packed: every device array equals the FASTA build, also for
    other -s / -I than the cache was written with, with N runs (blocks) and lower case in the reference"""
    rng = np.random.default_rng(5)
    seqs = []
    for n in (300_017, 1_234, 90_000):
        a = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=n)
        a[n // 3:n // 3 + 500] = ord("N"); a[10:40] = ord("n"); a[n // 2:n // 2 + 77] |= 0x20
        seqs.append(bytes(a))
    names = ["chrA", "chrB", "chrC"]
    p0 = B.make_params(s=16, I=4)
    ix0 = B.Index(p0, names, seqs)
    path = str(tmp_path / "ref.bsxpack")
    ix0.save_packed(path)
    for kw in (dict(s=16, I=4), dict(s=12, I=1), dict(s=10, I=16)):
        p = B.make_params(**kw)
        a, b = B.Index(p, names, seqs), B.Index.from_packed(p, path)
        assert a.header() == b.header() and a.info.n_entries == b.info.n_entries
        for what in ("refcat", "crefcat", "anchor", "tab", "pos", "ctx"):
            assert np.array_equal(a.download(what), b.download(what)), (kw, what)
        a.close(); b.close()
    with pytest.raises(B.BsxError, match="RRBS"):
        B.Index.from_packed(B.make_params(D="C-CGG"), path)
    (tmp_path / "junk").write_bytes(b"hello")
    with pytest.raises(B.BsxError, match="not a packed reference"):
        B.Index.from_packed(p0, str(tmp_path / "junk"))
    ix0.close()


@pytest.mark.parametrize("name", ["bam_se", "bam_se_quirks_B11_E400", "bam_pe_interleaved", "bam_pe_odd_tail"])
def test_cli_bam_read_input(tmp_path, name):
    """BAM read files through the command line == the unmodified reference fed the same BAM (tests/golden/bam)"""
    import gzip
    import bam_cases as BC
    argv, out = BC.build(name, str(tmp_path))
    exe = os.path.join(os.path.dirname(BL.LIB_PATH), "bsmap")
    r = subprocess.run([exe] + argv, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    exp = gzip.open(os.path.join(R.GOLDEN, "bam", name + ".sam.gz"), "rb").read()
    got = open(out, "rb").read()
    assert got == exp, R.first_diff(got, exp)


def test_cli_bam_output(tmp_path):
    """-o out.bam: coordinate-sorted BAM + .bai in process; decompressed it equals what samtools 0.1.7 (the reference's
    sam2bam.sh) makes of the reference's SAM for the same run (digest committed by tests/test_bam_output_cpu.py)"""
    import gzip, hashlib, json
    case = CS.BY_NAME["pe_sam"]
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    exe = os.path.join(os.path.dirname(BL.LIB_PATH), "bsmap")
    out = str(tmp_path / "out.bam")
    r = subprocess.run([exe] + case.cli(a, b, fa, out, None), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    digests = json.load(open(os.path.join(R.GOLDEN, "bam_output_sha256.json")))
    assert hashlib.sha256(gzip.open(out, "rb").read()).hexdigest() == digests["pe_sam"]
    assert os.path.exists(out + ".bai") and not os.path.exists(out + ".sam.tmp")


def test_cli_reference_cache(tmp_path):
    """BSX_REF_CACHE: the second run starts from the packed reference and writes the same file"""
    case = CS.BY_NAME["se_cfg2_r0_uR"]
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    cache = tmp_path / "cache"; cache.mkdir()
    exe = os.path.join(os.path.dirname(BL.LIB_PATH), "bsmap")
    outs = []
    for k in range(2):
        o = str(tmp_path / f"out{k}.sam")
        r = subprocess.run([exe] + case.cli(a, b, fa, o, None), capture_output=True, text=True, env=dict(os.environ, BSX_REF_CACHE=str(cache), BSX_CLI_TIMING="1"))
        assert r.returncode == 0, r.stdout + r.stderr
        outs.append(open(o, "rb").read())
        assert len(list(cache.iterdir())) == 1
    assert outs[0] == outs[1] == R.golden_load(case)[0]


def test_index_replica_over_nvlink_or_same_device():
    """bsx_index_replicate: metadata blob + peer copy of the device arrays gives an identical index"""
    case = CS.BY_NAME["se_cfg1"]
    d = case.data()
    p = B.make_params(**case.param_kwargs())
    ix = B.Index(p, d["gnames"], d["gseqs"])
    dev = 1 if BL.load().bsx_device_count() > 1 else 0
    rep = ix.replicate(dev)
    for what in ("refcat", "crefcat", "anchor", "tab", "pos"):
        assert np.array_equal(ix.download(what), rep.download(what)), what
    mp = B.Mapper(rep, p, max_batch=4096, stride=160)
    buf, lens = B.pack_reads(d["seqs"], stride=160)
    recs, _ = mp.map_se(buf, lens)
    exp = R.oracle_run(case)
    assert _rec_diff("rec", recs, exp["recs"]) is None
    mp.close(); rep.close(); ix.close()


CLI_CASES = ["se_cfg1", "se_mixed_A", "se_mixed_fa", "se_cfg2_bsp", "se_L60", "pe_sam", "pe_bsp_r0", "rrbs_se_A", "rrbs_pe"]


@pytest.mark.parametrize("name", CLI_CASES)
def test_cli_writes_the_reference_files(name, tmp_path):
    """the `bsmap` drop-in executable: same options, FASTA/FASTQ files in, SAM/BSP files out,
    byte-identical to what the unmodified reference wrote (-p 1)"""
    import subprocess
    case = CS.BY_NAME[name]
    exe = os.path.join(os.path.dirname(BL.LIB_PATH), "bsmap")
    assert os.path.exists(exe), "bsmap CLI not built (python -m bsmap_b200.build)"
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / ("out." + case.out_ext))
    o2 = str(tmp_path / "out_unpair.bsp") if (case.paired and case.out_ext != "sam") else None
    r = subprocess.run([exe] + case.cli(a, b, fa, o, o2) + ["-p", "4"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    exp_main, exp_un = R.golden_load(case)
    got = open(o, "rb").read()
    assert got == exp_main, R.first_diff(got, exp_main)
    if o2:
        got_un = open(o2, "rb").read()
        assert got_un == exp_un, R.first_diff(got_un, exp_un)
    assert "Total number of aligned reads" in r.stdout


@pytest.mark.parametrize("name", ["se_cfg1", "pe_sam", "rrbs_se_A", "se_cfg2_bsp"])
def test_cli_maps_on_several_devices_in_input_order(name, tmp_path):
    """`bsmap -g`: one mapper thread per listed device, each with its own replica of the index (cudaMemcpyPeer), small
    batches dealt to whichever is free, text written in input order -> the same bytes as the one-device run and the
    reference.  On a one-GPU box the list names device 0 three times (three replicas, three mapper threads); with more
    devices visible it is every device."""
    import subprocess
    case = CS.BY_NAME[name]
    exe = os.path.join(os.path.dirname(BL.LIB_PATH), "bsmap")
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / ("out." + case.out_ext))
    o2 = str(tmp_path / "out_unpair.bsp") if (case.paired and case.out_ext != "sam") else None
    n = BL.load().bsx_device_count()
    devs = ",".join(str(i) for i in range(n)) if n > 1 else "0,0,0"
    r = subprocess.run([exe] + case.cli(a, b, fa, o, o2) + ["-p", "4", "-g", devs], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, BSX_CLI_BATCH="257", BSX_CLI_TIMING="1", BSX_CLI_WAIT_DEVICES="1"))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    exp_main, exp_un = R.golden_load(case)
    got = open(o, "rb").read()
    assert got == exp_main, R.first_diff(got, exp_main)
    if o2:
        assert open(o2, "rb").read() == exp_un
    used = [ln for ln in r.stderr.splitlines() if "[bsx timing] device" in ln and " 0 reads" not in ln]
    assert len(used) >= 2, r.stderr[-1500:]     # more than one mapper thread took batches


@pytest.mark.parametrize("name", ["se_mixed_A", "pe_sam"])
def test_cli_streams_gzipped_reads(name, tmp_path):
    """gzip'ed read files go through the windowed stream reader; with small batches several windows are alive in the cut ->
    map -> format pipeline at once (the views of a batch keep theirs) -> the reference's bytes all the same"""
    import gzip, subprocess
    case = CS.BY_NAME[name]
    exe = os.path.join(os.path.dirname(BL.LIB_PATH), "bsmap")
    fa, a, b = CS.write_inputs(case, str(tmp_path))
    for f in (a, b):
        if f:
            with gzip.open(f + ".gz", "wb", compresslevel=1) as g:
                g.write(open(f, "rb").read())
    o = str(tmp_path / ("out." + case.out_ext))
    r = subprocess.run([exe] + case.cli(a + ".gz", b + ".gz" if b else None, fa, o, None) + ["-p", "4"], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, BSX_CLI_BATCH="193"))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    got, exp = open(o, "rb").read(), R.golden_load(case)[0]
    assert got == exp, R.first_diff(got, exp)


def test_cli_option_grammar(tmp_path):
    """-x=val form, unknown option exit code = argv index (main.cpp:452-455)"""
    import subprocess
    exe = os.path.join(os.path.dirname(BL.LIB_PATH), "bsmap")
    case = CS.BY_NAME["se_cfg1"]
    fa, a, _ = CS.write_inputs(case, str(tmp_path))
    o = str(tmp_path / "o.sam")
    r = subprocess.run([exe, f"-a={a}", f"-d={fa}", f"-o={o}", "-s=16", "-v=2", "-I=4", "-S=7"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert open(o, "rb").read() == R.golden_load(case)[0]
    r = subprocess.run([exe, "-a", a, "-Q", "3"], capture_output=True, text=True)
    assert r.returncode == 3 and "unknown option: -Q" in r.stdout
