#!/usr/bin/env python
"""Cost of the methylation haplotype load (the MHL walk in the Epi pile-up kernels, meth_mhl_region_kernel and the MHL
writer) next to the plain and Epi pile-up, on one GPU.

Workload: tests/epiallele_bench.py's, a 200 Mb synthetic genome and 4 M x 100 nt reads mapped by `bsmap` to SAM.
  * kernel: CUDA time of the pile-up kernels alone (torch.profiler, CUDA activities) at 131072 alignments per launch,
    alternated: plain; Epi; MHL; Epi + MHL; everything (Epi + MHL + Pdr + Conv + M-bias + exclusion + Snp);
    meth_pileup_kernel over bsx_meth_add batches from the SAM, meth_pileup_mapped_kernel over in-process mapped batches
  * the parent: with --parent DIR (a built checkout of the parent commit), Epi-only in a child process on that
    checkout's library, alternated with this one's Epi-only in the same call
  * regions: CUDA time of meth_mhl_region_kernel (with the span, scan and cut kernels) and the wall time of
    bsx_meth_regions_mhl for --tiles 1000 and for a 100 k-line BED, and the wall time of bsx_meth_write_mhl for both
  * whole process: `methratio` and fused `bsmap --methratio` (no -o), each without and with --mhl / --meth-mhl over
    --tiles 1000, runs alternated
The genome is uniform random: about 6 % of its dinucleotides are CpG against about 1 % in mammals, so the run atomics
here are an upper bound of what a mammalian genome costs.

    python tests/mhl_bench.py [--reads 4000000] [--len 100] [--genome-mb 200] [--runs 3] [--parent DIR] [--out FILE]
Prints one JSON line (and writes it to --out when given).
"""
import argparse, json, os, subprocess, sys, tempfile, time

ap = argparse.ArgumentParser()
ap.add_argument("--reads", type=int, default=4_000_000)
ap.add_argument("--len", type=int, default=100)
ap.add_argument("--genome-mb", type=float, default=200.0)
ap.add_argument("--runs", type=int, default=3)
ap.add_argument("--kernel-batches", type=int, default=8)
ap.add_argument("--parent", default=None)
ap.add_argument("--out", default=None)
ap.add_argument("--child", default=None, help=argparse.SUPPRESS)     # internal: ROOT,td -> Epi-only kernel times of ROOT
a = ap.parse_args()
ROOT = a.child.split(",")[0] if a.child else os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np
import torch
from bsmap_b200 import synth
import bsmap_b200 as B
from meth_inputs import api_arrays

if not torch.cuda.is_available():
    sys.exit("mhl_bench: needs a CUDA device")
BATCH, n_chr = 131072, 5
names = ["chr%d" % (i + 1) for i in range(n_chr)]
STRIDE = (a.len + 15) // 16 * 16
map_args_of = lambda fa, fq: ["-a", fq, "-d", fa, "-s", "16", "-v", "5", "-S", "7"]


def kernel_us(run, keys):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    return sum(e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total for e in prof.key_averages()
               if any(k in e.key for k in keys))


def workload(td, g):
    gseqs = [bytes(x.cpu().numpy()) for x in g]
    head = os.path.join(td, "head.sam")
    cols = api_arrays([head], names)
    reads = np.load(os.path.join(td, "reads.npy"))
    return gseqs, cols, reads


def meth(ix, var):
    mh = B.Meth(ix, B.meth_opts())
    if "epi" in var or var == "all":
        mh.enable_epialleles()
    if "mhl" in var or var == "all":
        mh.enable_mhl()
    if var == "all":
        mh.enable_pdr(4); mh.enable_conversion_filter(3); mh.enable_mbias(); mh.enable_ct_snp("correct"); mh.set_ignore(2, 2, 2, 2)
    return mh


def pileup_times(pix, mix, mp, cols, reads, variants, rounds):
    """{path: {variant: [us per batch]}}, round 0 (warm-up) not recorded; and the last Meth of each text variant's counts"""
    kern = {"text": {v: [] for v in variants}, "mapped": {v: [] for v in variants}}
    rlens = np.full(len(reads), a.len, dtype=np.uint16)
    for rnd in range(rounds + 1):
        for var in variants:
            mh = meth(pix, var)
            us = kernel_us(lambda: [mh.add(*[c[b:b + BATCH] for c in cols[:7]], read2=cols[7][b:b + BATCH]) for b in range(0, len(cols[0]), BATCH)],
                           ("meth_pileup_kernel",))
            if rnd:
                kern["text"][var].append(round(us / ((len(cols[0]) + BATCH - 1) // BATCH), 1))
            mh.close()
            mh = meth(mix, var)
            mh.attach(mp, sam_rules=True)
            us = kernel_us(lambda: mp.map_se(reads, rlens), ("meth_pileup_mapped_kernel",))
            if rnd:
                kern["mapped"][var].append(round(us / ((len(reads) + BATCH - 1) // BATCH), 1))
            B.lib.check(B.lib.load().bsx_mapper_attach_meth(mp.h, None, None, 0))
            mh.close()
    return kern


def indexes(gseqs):
    pix = B.Index.packed(names, gseqs)
    p = B.make_params(s=16, v=5, S=7)
    mix = B.Index(p, names, gseqs)
    return pix, mix, B.Mapper(mix, p, max_batch=BATCH, stride=STRIDE)


if a.child:                                                   # Epi-only on ROOT's library, one round after a warm-up
    td = a.child.split(",")[1]
    g = synth.make_genome(1, [int(a.genome_mb * 1e6 / n_chr)] * n_chr, device="cuda")
    gseqs, cols, reads = workload(td, g)
    pix, mix, mp = indexes(gseqs)
    print(json.dumps(pileup_times(pix, mix, mp, cols, reads, ("epi",), 1)))
    sys.exit(0)

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.splitlines()
res = {"gpu": smi[0].strip() if smi else torch.cuda.get_device_name(0), "reads": a.reads, "read_len": a.len, "genome_mb": a.genome_mb}
td = tempfile.mkdtemp(prefix="bsx_mhl_")
g = synth.make_genome(1, [int(a.genome_mb * 1e6 / n_chr)] * n_chr, device="cuda")
sim = synth.simulate_reads(g, a.reads, a.len, seed=11, subs="cfg2")
fa, fq, sam = os.path.join(td, "ref.fa"), os.path.join(td, "reads.fq"), os.path.join(td, "aln.sam")
synth.write_fasta(fa, [x.cpu() for x in g])
synth.write_fastq(fq, sim["seq"].cpu(), synth.read_names({k: v.cpu() for k, v in sim.items() if k != "seq"}))
BSMAP, METHRATIO = os.path.join(ROOT, "bsmap_b200", "bsmap"), os.path.join(ROOT, "bsmap_b200", "methratio")
map_args = map_args_of(fa, fq)
subprocess.run([BSMAP] + map_args + ["-o", sam], check=True, capture_output=True)
NB = a.kernel_batches
with open(sam) as f, open(os.path.join(td, "head.sam"), "w") as o:
    n = 0
    for line in f:
        if line.startswith("@"):
            continue
        o.write(line); n += 1
        if n >= BATCH * NB:
            break
nr = min(a.reads, BATCH * NB)
rbuf = np.zeros((nr, STRIDE), dtype=np.uint8)
rbuf[:, :a.len] = sim["seq"][:nr].cpu().numpy()
np.save(os.path.join(td, "reads.npy"), rbuf)


def timed(argv):
    t0 = time.perf_counter()
    r = subprocess.run(argv, capture_output=True, text=True)
    dt = time.perf_counter() - t0
    assert r.returncode == 0, r.stderr[-400:]
    return dt


runs = {"methratio": [], "methratio_mhl": [], "fused": [], "fused_mhl": []}
out, mout = os.path.join(td, "t.txt"), os.path.join(td, "mhl.txt")
for k in range(a.runs):                                       # alternate without / with in every round
    runs["methratio"].append(timed([METHRATIO, "-o", out, "-d", fa, "-q", sam]))
    runs["methratio_mhl"].append(timed([METHRATIO, "-o", out, "-d", fa, "-q", sam, "--mhl", mout, "--tiles", "1000"]))
    runs["fused"].append(timed([BSMAP] + map_args + ["--methratio", out]))
    runs["fused_mhl"].append(timed([BSMAP] + map_args + ["--methratio", out, "--meth-mhl", mout, "--meth-tiles", "1000"]))
res["seconds_runs"] = {k: [round(x, 3) for x in v] for k, v in runs.items()}
res["seconds_min"] = {k: round(min(v), 3) for k, v in runs.items()}

gseqs, cols, reads = workload(td, g)
pix, mix, mp = indexes(gseqs)
VARIANTS = ("plain", "epi", "mhl", "epi_mhl", "all")
kern = pileup_times(pix, mix, mp, cols, reads, VARIANTS, 3)
res["kernel_batch_alignments"] = BATCH
res["kernel_text_batches"], res["kernel_mapped_batches"] = (len(cols[0]) + BATCH - 1) // BATCH, (nr + BATCH - 1) // BATCH
res["variant_all"] = "epi + mhl + pdr(4) + conversion filter(3) + mbias + exclusion(2,2,2,2) + ct_snp correct"
for path in ("text", "mapped"):
    res["pileup_%s_kernel_us_per_batch" % path] = kern[path]
    res["pileup_%s_kernel_ratio_to_plain" % path] = {v: round(min(kern[path][v]) / min(kern[path]["plain"]), 3) for v in VARIANTS[1:]}

if a.parent:                                                  # Epi-only: the parent's library against this one, alternated
    par = {"text": [], "mapped": []}
    cur = {"text": [], "mapped": []}
    for rnd in range(3):
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "%s,%s" % (os.path.abspath(a.parent), td),
                            "--genome-mb", str(a.genome_mb), "--len", str(a.len)], capture_output=True, text=True, cwd=os.path.abspath(a.parent))
        assert r.returncode == 0, r.stderr[-800:]
        p = json.loads(r.stdout.strip().splitlines()[-1])
        c = pileup_times(pix, mix, mp, cols, reads, ("epi",), 1)
        for path in ("text", "mapped"):
            par[path] += p[path]["epi"]; cur[path] += c[path]["epi"]
    res["epi_only_parent_us_per_batch"], res["epi_only_this_us_per_batch"] = par, cur
    res["epi_only_ratio_to_parent"] = {path: round(min(cur[path]) / min(par[path]), 3) for path in ("text", "mapped")}
else:
    res["epi_only_ratio_to_parent"] = "not measured"

# regions: one Meth with MHL over the text batches, then --tiles 1000 and a 100 k-line BED
mh = meth(pix, "mhl")
for b in range(0, len(cols[0]), BATCH):
    mh.add(*[c[b:b + BATCH] for c in cols[:7]], read2=cols[7][b:b + BATCH])
res["mhl_alignments_calls_valid"] = list(mh.mhl()) + [mh.valid()]
lens = [len(s) for s in gseqs]
tiles = [(k, s, min(s + 1000, L)) for k, L in enumerate(lens) for s in range(0, L, 1000)]
rng = np.random.default_rng(3)
bk = rng.integers(0, n_chr, 100_000)
bs = np.array([int(rng.integers(0, lens[k] - 5000)) for k in bk])
bed = list(zip(bk.tolist(), bs.tolist(), (bs + rng.integers(200, 5000, len(bs))).tolist()))
RKEYS = ("meth_mhl_region_kernel", "mhl_span_kernel", "scan_tile_kernel", "scan_add_kernel")
for name, regs in (("tiles_1000", tiles), ("bed_100k", bed)):
    c, s, e = (np.array([r[i] for r in regs]) for i in range(3))
    kus, wall, wr = [], [], []
    for rnd in range(4):
        t0 = time.perf_counter()
        us = kernel_us(lambda: mh.mhl_regions(c, s, e), RKEYS)
        dt = time.perf_counter() - t0
        with open(os.path.join(td, "w.txt"), "wb") as f:
            t1 = time.perf_counter()
            mh.write_mhl(f.fileno(), c, s, e)
            dw = time.perf_counter() - t1
        if rnd:
            kus.append(round(us, 1)); wall.append(round(dt, 4)); wr.append(round(dw, 3))
    res["regions_%s" % name] = {"regions": len(regs), "region_kernels_us": kus, "regions_mhl_seconds_profiled": wall, "write_mhl_seconds": wr}
mh.close()
line = json.dumps(res)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    open(a.out, "w").write(line + "\n")
