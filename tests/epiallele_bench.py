#!/usr/bin/env python
"""Cost of 4-CpG epialleles (the Epi pile-up kernels, the CpG rank index and the epiallele writer) next to the plain
and Pdr pile-up, on one GPU.

Workload: tests/pdr_bench.py's, a 200 Mb synthetic genome and 4 M x 100 nt reads (97 % conversion) mapped by `bsmap` to
SAM.
  * whole process: `methratio` and fused `bsmap --methratio` (no -o), each without and with --epialleles /
    --meth-epialleles, runs alternated in the same process tree
  * kernel: CUDA time of the pile-up kernels alone (torch.profiler, CUDA activities) at 131072 alignments per launch
    (the command line's 128 k-read batch), alternated: plain; Pdr (K = 4); Epi; Epi + Pdr + Conv (threshold 3) + M-bias
    + exclusion + Snp; meth_pileup_kernel over bsx_meth_add batches from the same SAM, meth_pileup_mapped_kernel over
    in-process mapped batches of the same reads
  * the rank index: CUDA time of its three kernels, and the wall time of bsx_meth_enable_epialleles (index, counters
    and their zeroing)
  * the writer: wall time of bsx_meth_write_epialleles after the text-path batches
The genome is uniform random: about 6 % of its dinucleotides are CpG against about 1 % in mammals, so the window
atomics here are an upper bound of what a mammalian genome costs.

    python tests/epiallele_bench.py [--reads 4000000] [--len 100] [--genome-mb 200] [--runs 3] [--out FILE]
Prints one JSON line (and writes it to --out when given).
"""
import argparse, json, os, subprocess, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
from bsmap_b200 import synth
import bsmap_b200 as B

ap = argparse.ArgumentParser()
ap.add_argument("--reads", type=int, default=4_000_000)
ap.add_argument("--len", type=int, default=100)
ap.add_argument("--genome-mb", type=float, default=200.0)
ap.add_argument("--runs", type=int, default=3)
ap.add_argument("--kernel-batches", type=int, default=8)
ap.add_argument("--out", default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("epiallele_bench: needs a CUDA device")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.splitlines()
res = {"gpu": smi[0].strip() if smi else torch.cuda.get_device_name(0), "reads": a.reads, "read_len": a.len, "genome_mb": a.genome_mb}
td = tempfile.mkdtemp(prefix="bsx_epi_")
n_chr = 5
g = synth.make_genome(1, [int(a.genome_mb * 1e6 / n_chr)] * n_chr, device="cuda")
sim = synth.simulate_reads(g, a.reads, a.len, seed=11, subs="cfg2")
fa, fq, sam = os.path.join(td, "ref.fa"), os.path.join(td, "reads.fq"), os.path.join(td, "aln.sam")
synth.write_fasta(fa, [x.cpu() for x in g])
synth.write_fastq(fq, sim["seq"].cpu(), synth.read_names({k: v.cpu() for k, v in sim.items() if k != "seq"}))
map_args = ["-a", fq, "-d", fa, "-s", "16", "-v", "5", "-S", "7"]
subprocess.run([os.path.join(ROOT, "bsmap_b200", "bsmap")] + map_args + ["-o", sam], check=True, capture_output=True)
EPI_ARGS = ["--epialleles", os.path.join(td, "epi.txt")]
FUSED_EPI = ["--meth-epialleles", os.path.join(td, "epi.txt")]


def timed(argv):
    t0 = time.perf_counter()
    r = subprocess.run(argv, capture_output=True, text=True)
    dt = time.perf_counter() - t0
    assert r.returncode == 0, r.stderr[-400:]
    return dt


runs = {"methratio": [], "methratio_epi": [], "fused": [], "fused_epi": []}
for k in range(a.runs):                                       # alternate without / with in every round
    out = os.path.join(td, "t.txt")
    runs["methratio"].append(timed([os.path.join(ROOT, "bsmap_b200", "methratio"), "-o", out, "-d", fa, "-q", sam]))
    runs["methratio_epi"].append(timed([os.path.join(ROOT, "bsmap_b200", "methratio"), "-o", out, "-d", fa, "-q", sam] + EPI_ARGS))
    runs["fused"].append(timed([os.path.join(ROOT, "bsmap_b200", "bsmap")] + map_args + ["--methratio", out]))
    runs["fused_epi"].append(timed([os.path.join(ROOT, "bsmap_b200", "bsmap")] + map_args + ["--methratio", out] + FUSED_EPI))
res["seconds_runs"] = {k: [round(x, 3) for x in v] for k, v in runs.items()}
res["seconds_min"] = {k: round(min(v), 3) for k, v in runs.items()}

# kernel time: the pile-up kernels alone (CUDA time from torch.profiler), plain vs Pdr vs Epi vs Epi + Pdr + Conv +
# M-bias + exclusion + Snp, alternated, 131072 alignments per launch: the text path (bsx_meth_add, meth_pileup_kernel) on the first lines of the
# SAM, the in-process path (Mapper + attached Meth, meth_pileup_mapped_kernel) on the first reads
from meth_inputs import api_arrays
names = ["chr%d" % (i + 1) for i in range(n_chr)]
gseqs = [bytes(x.cpu().numpy()) for x in g]
BATCH = 131072
NB = a.kernel_batches
head = os.path.join(td, "head.sam")
with open(sam) as f, open(head, "w") as o:
    n = 0
    for line in f:
        if line.startswith("@"):
            continue
        o.write(line); n += 1
        if n >= BATCH * NB:
            break
cols = api_arrays([head], names)
pix = B.Index.packed(names, gseqs)
p = B.make_params(s=16, v=5, S=7)
mix = B.Index(p, names, gseqs)
STRIDE = (a.len + 15) // 16 * 16
nr = min(a.reads, BATCH * NB)
rbuf = np.zeros((nr, STRIDE), dtype=np.uint8)
rbuf[:, :a.len] = sim["seq"][:nr].cpu().numpy()
rlens = np.full(nr, a.len, dtype=np.uint16)
mp = B.Mapper(mix, p, max_batch=BATCH, stride=STRIDE)


def kernel_us(run, name):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    return sum(e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total for e in prof.key_averages() if name in e.key)


VARIANTS = ("plain", "pdr", "epi", "epi_pdr_conv3_mbias_exclusion_ct_snp")


def meth(ix, var):
    mh = B.Meth(ix, B.meth_opts())
    if var.startswith("epi"):
        mh.enable_epialleles()
    if var in ("pdr", "epi_pdr_conv3_mbias_exclusion_ct_snp"):
        mh.enable_pdr(4)
    if var == "epi_pdr_conv3_mbias_exclusion_ct_snp":
        mh.enable_conversion_filter(3); mh.enable_mbias(); mh.enable_ct_snp("correct"); mh.set_ignore(2, 2, 2, 2)
    return mh


kern = {"text": {v: [] for v in VARIANTS}, "mapped": {v: [] for v in VARIANTS}}
spanning, writer_s = {}, []
for rnd in range(4):                                          # round 0 warms up every shape; not recorded
    for var in VARIANTS:
        mh = meth(pix, var)
        us = kernel_us(lambda: [mh.add(*[c[b:b + BATCH] for c in cols[:7]], read2=cols[7][b:b + BATCH]) for b in range(0, len(cols[0]), BATCH)],
                       "meth_pileup_kernel")
        if rnd:
            kern["text"][var].append(us / ((len(cols[0]) + BATCH - 1) // BATCH))
        if var.startswith("epi"):
            spanning[var] = list(mh.epialleles()) + [mh.valid()]
            if var == "epi" and rnd:
                with open(os.path.join(td, "w.txt"), "wb") as f:
                    t0 = time.perf_counter()
                    mh.write_epialleles(gseqs, f.fileno())
                    writer_s.append(round(time.perf_counter() - t0, 3))
        mh.close()
        mh = meth(mix, var)
        mh.attach(mp, sam_rules=True)
        us = kernel_us(lambda: mp.map_se(rbuf, rlens), "meth_pileup_mapped_kernel")
        if rnd:
            kern["mapped"][var].append(us / ((nr + BATCH - 1) // BATCH))
        B.lib.check(B.lib.load().bsx_mapper_attach_meth(mp.h, None, None, 0))
        mh.close()
res["kernel_batch_alignments"] = BATCH
res["kernel_text_spanning_windows_valid"] = spanning
res["writer_seconds"] = writer_s

# the rank index: its kernels' CUDA time, and the wall time of enable_epialleles (index + counters + zeroing)
build_us, build_s = [], []
for rnd in range(4):
    mh = B.Meth(pix, B.meth_opts())
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mh.enable_epialleles()
        dt = time.perf_counter() - t0
    us = sum(e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total for e in prof.key_averages()
             if any(k in e.key for k in ("cpg_count_kernel", "scan_tile_kernel", "scan_add_kernel")))
    if rnd:
        build_us.append(round(us, 1)); build_s.append(round(dt, 4))
    n_sites = sum(len(mh.epiallele_counters(k)[0]) for k in range(n_chr)) if rnd == 1 else None
    if n_sites is not None:
        res["cpg_sites"] = n_sites
    mh.close()
res["rank_index_kernels_us"] = build_us
res["enable_epialleles_seconds"] = build_s
res["kernel_text_batches"], res["kernel_mapped_batches"] = (len(cols[0]) + BATCH - 1) // BATCH, (nr + BATCH - 1) // BATCH
for path in ("text", "mapped"):
    k = kern[path]
    res["pileup_%s_kernel_us_per_batch" % path] = {v: [round(x, 1) for x in k[v]] for v in VARIANTS}
    res["pileup_%s_kernel_ratio_to_plain" % path] = {v: round(min(k[v]) / min(k["plain"]), 3) for v in VARIANTS[1:]}
line = json.dumps(res)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    open(a.out, "w").write(line + "\n")
