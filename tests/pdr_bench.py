#!/usr/bin/env python
"""Cost of the proportion of discordant reads (the Pdr pile-up kernels) next to the plain and Cycles pile-up, on one GPU.

Workload: tests/ctsnp_bench.py's, a 200 Mb synthetic genome and 4 M x 100 nt reads mapped by `bsmap` to SAM.
  * whole process: `methratio` and fused `bsmap --methratio` (no -o), each without and with --pdr / --meth-pdr (K = 4),
    runs alternated in the same process tree
  * kernel: CUDA time of the pile-up kernels alone (torch.profiler, CUDA activities) at 131072 alignments per launch
    (the command line's 128 k-read batch): plain; Cycles with exclusion of 2 cycles at every read end; Pdr (K = 4);
    Pdr + Conv (threshold 3) + M-bias + exclusion + Snp; meth_pileup_kernel over bsx_meth_add batches from the same
    SAM, meth_pileup_mapped_kernel over in-process mapped batches of the same reads
The genome is uniform random: about 6 % of its dinucleotides are CpG against about 1 % in mammals, so the concordance
atomics here are an upper bound of what a mammalian genome costs.

    python tests/pdr_bench.py [--reads 4000000] [--len 100] [--genome-mb 200] [--runs 3] [--out FILE]
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
    sys.exit("pdr_bench: needs a CUDA device")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.splitlines()
res = {"gpu": smi[0].strip() if smi else torch.cuda.get_device_name(0), "reads": a.reads, "read_len": a.len, "genome_mb": a.genome_mb}
td = tempfile.mkdtemp(prefix="bsx_pdr_")
n_chr = 5
g = synth.make_genome(1, [int(a.genome_mb * 1e6 / n_chr)] * n_chr, device="cuda")
sim = synth.simulate_reads(g, a.reads, a.len, seed=11, subs="cfg2")
fa, fq, sam = os.path.join(td, "ref.fa"), os.path.join(td, "reads.fq"), os.path.join(td, "aln.sam")
synth.write_fasta(fa, [x.cpu() for x in g])
synth.write_fastq(fq, sim["seq"].cpu(), synth.read_names({k: v.cpu() for k, v in sim.items() if k != "seq"}))
map_args = ["-a", fq, "-d", fa, "-s", "16", "-v", "5", "-S", "7"]
subprocess.run([os.path.join(ROOT, "bsmap_b200", "bsmap")] + map_args + ["-o", sam], check=True, capture_output=True)
PDR_ARGS = ["--pdr", os.path.join(td, "pdr.txt")]
FUSED_PDR = ["--meth-pdr", os.path.join(td, "pdr.txt")]


def timed(argv):
    t0 = time.perf_counter()
    r = subprocess.run(argv, capture_output=True, text=True)
    dt = time.perf_counter() - t0
    assert r.returncode == 0, r.stderr[-400:]
    return dt


runs = {"methratio": [], "methratio_pdr": [], "fused": [], "fused_pdr": []}
for k in range(a.runs):                                       # alternate without / with in every round
    out = os.path.join(td, "t.txt")
    runs["methratio"].append(timed([os.path.join(ROOT, "bsmap_b200", "methratio"), "-o", out, "-d", fa, "-q", sam]))
    runs["methratio_pdr"].append(timed([os.path.join(ROOT, "bsmap_b200", "methratio"), "-o", out, "-d", fa, "-q", sam] + PDR_ARGS))
    runs["fused"].append(timed([os.path.join(ROOT, "bsmap_b200", "bsmap")] + map_args + ["--methratio", out]))
    runs["fused_pdr"].append(timed([os.path.join(ROOT, "bsmap_b200", "bsmap")] + map_args + ["--methratio", out] + FUSED_PDR))
res["seconds_runs"] = {k: [round(x, 3) for x in v] for k, v in runs.items()}
res["seconds_min"] = {k: round(min(v), 3) for k, v in runs.items()}

# kernel time: the pile-up kernels alone (CUDA time from torch.profiler), plain vs Cycles (exclusion 2,2,2,2) vs Pdr
# vs Pdr + Conv + M-bias + exclusion + Snp, alternated, 131072 alignments per launch: the text path (bsx_meth_add, meth_pileup_kernel) on the first lines of the
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


VARIANTS = ("plain", "exclusion", "pdr", "pdr_conv3_mbias_exclusion_ct_snp")


def meth(ix, var):
    mh = B.Meth(ix, B.meth_opts())
    if var.startswith("pdr"):
        mh.enable_pdr(4)
    if var == "pdr_conv3_mbias_exclusion_ct_snp":
        mh.enable_conversion_filter(3); mh.enable_mbias(); mh.enable_ct_snp("correct")
    if var in ("exclusion", "pdr_conv3_mbias_exclusion_ct_snp"):
        mh.set_ignore(2, 2, 2, 2)
    return mh


kern = {"text": {v: [] for v in VARIANTS}, "mapped": {v: [] for v in VARIANTS}}
informative = {}
for rnd in range(4):                                          # round 0 warms up every shape; not recorded
    for var in VARIANTS:
        mh = meth(pix, var)
        us = kernel_us(lambda: [mh.add(*[c[b:b + BATCH] for c in cols[:7]], read2=cols[7][b:b + BATCH]) for b in range(0, len(cols[0]), BATCH)],
                       "meth_pileup_kernel")
        if rnd:
            kern["text"][var].append(us / ((len(cols[0]) + BATCH - 1) // BATCH))
        if var.startswith("pdr"):
            informative[var] = list(mh.pdr()) + [mh.valid()]
        mh.close()
        mh = meth(mix, var)
        mh.attach(mp, sam_rules=True)
        us = kernel_us(lambda: mp.map_se(rbuf, rlens), "meth_pileup_mapped_kernel")
        if rnd:
            kern["mapped"][var].append(us / ((nr + BATCH - 1) // BATCH))
        B.lib.check(B.lib.load().bsx_mapper_attach_meth(mp.h, None, None, 0))
        mh.close()
res["kernel_batch_alignments"] = BATCH
res["kernel_text_informative_discordant_valid"] = informative
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
