#!/usr/bin/env python
"""Cost of the region report (meth_region_kernel) on one GPU, next to a device-to-device copy of the same bytes.

Workload: tests/conversion_bench.py's, a 200 Mb synthetic genome and 4 M x 100 nt reads; the counters (1.6 GB of
meth / depth, well past the L2) are piled up in process by an attached Meth.
  * kernel: CUDA time of meth_region_kernel (torch.profiler, CUDA activities) for 1 kb tiles over the whole genome and
    for 50 k random 1-5 kb regions; bytes = 8 per position in the regions (meth + depth) + the 2-bit reference; the
    bandwidth reference is a cudaMemcpyAsync device-to-device copy (torch copy_, listed as Memcpy DtoD) of as many
    bytes, timed the same way, counted as read + write
  * whole process: `methratio` on the SAM and fused `bsmap --methratio` (no -o), each without and with a 1 kb tile
    report, runs alternated

    python tests/region_bench.py [--reads 4000000] [--len 100] [--genome-mb 200] [--runs 3] [--out FILE]
Prints one JSON line (and writes it to --out when given).
"""
import argparse, json, os, subprocess, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
from bsmap_b200 import synth
import bsmap_b200 as B

ap = argparse.ArgumentParser()
ap.add_argument("--reads", type=int, default=4_000_000)
ap.add_argument("--len", type=int, default=100)
ap.add_argument("--genome-mb", type=float, default=200.0)
ap.add_argument("--runs", type=int, default=3)
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--out", default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("region_bench: needs a CUDA device")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.splitlines()
res = {"gpu": smi[0].strip() if smi else torch.cuda.get_device_name(0), "reads": a.reads, "read_len": a.len, "genome_mb": a.genome_mb}
td = tempfile.mkdtemp(prefix="bsx_region_")
n_chr = 5
g = synth.make_genome(1, [int(a.genome_mb * 1e6 / n_chr)] * n_chr, device="cuda")
sim = synth.simulate_reads(g, a.reads, a.len, seed=11, subs="cfg2")
names = ["chr%d" % (i + 1) for i in range(n_chr)]
lens = {n: int(x.numel()) for n, x in zip(names, g)}
fa, fq, sam = os.path.join(td, "ref.fa"), os.path.join(td, "reads.fq"), os.path.join(td, "aln.sam")
synth.write_fasta(fa, [x.cpu() for x in g])
synth.write_fastq(fq, sim["seq"].cpu(), synth.read_names({k: v.cpu() for k, v in sim.items() if k != "seq"}))
map_args = ["-a", fq, "-d", fa, "-s", "16", "-v", "5", "-S", "7"]
BSMAP, METHRATIO = os.path.join(ROOT, "bsmap_b200", "bsmap"), os.path.join(ROOT, "bsmap_b200", "methratio")
subprocess.run([BSMAP] + map_args + ["-o", sam], check=True, capture_output=True)


def timed(argv):
    t0 = time.perf_counter()
    r = subprocess.run(argv, capture_output=True, text=True)
    dt = time.perf_counter() - t0
    assert r.returncode == 0, r.stderr[-400:]
    return dt


out, rep = os.path.join(td, "t.txt"), os.path.join(td, "rep.txt")
runs = {"methratio": [], "methratio_tiles1k": [], "fused": [], "fused_tiles1k": []}
for k in range(a.runs):                                       # alternate without / with in every round
    runs["methratio"].append(timed([METHRATIO, "-o", out, "-d", fa, "-q", sam]))
    runs["methratio_tiles1k"].append(timed([METHRATIO, "-o", out, "-d", fa, "-q", sam, "--region-report", rep, "--tiles", "1000"]))
    runs["fused"].append(timed([BSMAP] + map_args + ["--methratio", out]))
    runs["fused_tiles1k"].append(timed([BSMAP] + map_args + ["--methratio", out, "--meth-region-report", rep, "--meth-tiles", "1000"]))
res["seconds_runs"] = {k: [round(x, 3) for x in v] for k, v in runs.items()}
res["seconds_min"] = {k: round(min(v), 3) for k, v in runs.items()}
res["region_report_bytes_tiles1k"] = os.path.getsize(rep)

# the counters of all reads, piled up in process
gseqs = [bytes(x.cpu().numpy()) for x in g]
p = B.make_params(s=16, v=5, S=7)
ix = B.Index(p, names, gseqs)
STRIDE = (a.len + 15) // 16 * 16
rbuf = np.zeros((a.reads, STRIDE), dtype=np.uint8)
rbuf[:, :a.len] = sim["seq"].cpu().numpy()
mp = B.Mapper(ix, p, max_batch=131072, stride=STRIDE)
mh = B.Meth(ix, B.meth_opts())
mh.attach(mp, sam_rules=True)
mp.map_se(rbuf, np.full(a.reads, a.len, dtype=np.uint16))
res["valid_mappings"] = mh.valid()

rnd = np.random.default_rng(5)
tiles = [(k, s, min(s + 1000, lens[n])) for k, n in enumerate(names) for s in range(0, lens[n], 1000)]
bed_chr = rnd.integers(0, n_chr, 50_000)
bed_len = rnd.integers(1000, 5001, 50_000)
bed_start = np.array([rnd.integers(0, lens[names[c]] - l) for c, l in zip(bed_chr, bed_len)])
WORKLOADS = {
    "tiles_1kb": ([t[0] for t in tiles], [t[1] for t in tiles], [t[2] for t in tiles]),
    "bed_50k_1to5kb": (bed_chr, bed_start, bed_start + bed_len),
}


def cuda_us(run, name):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    return sum(e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total for e in prof.key_averages() if name in e.key)


for w, (c, s, e) in WORKLOADS.items():
    positions = int(np.sum(np.asarray(e) - np.asarray(s)))
    nbytes = positions * 8 + positions // 4
    src = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    first = mh.regions(c, s, e)                               # warm-up, and the result every repeat must reproduce
    k_us, c_us = [], []
    for _ in range(a.repeats):                                # alternated
        k_us.append(cuda_us(lambda: mh.regions(c, s, e), "meth_region_kernel"))
        c_us.append(cuda_us(lambda: dst.copy_(src), "Memcpy DtoD"))
        assert np.array_equal(mh.regions(c, s, e), first)
    del src, dst
    res[w] = {"regions": len(c), "positions": positions, "bytes": nbytes, "kernel_us": [round(x, 1) for x in k_us],
              "kernel_GBps": round(nbytes / min(k_us) / 1e3, 1), "copy_us": [round(x, 1) for x in c_us],
              "copy_GBps_read_plus_write": round(2 * nbytes / min(c_us) / 1e3, 1),
              "kernel_over_copy_time": round(min(k_us) / min(c_us), 3), "covered": int(first[:, :, 1].sum())}
mh.close(); mp.close(); ix.close()
line = json.dumps(res)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    open(a.out, "w").write(line + "\n")
