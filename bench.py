#!/usr/bin/env python
"""bench.py -- BSMAP hot path on B200: reads (pairs) mapped per second, one JSON line (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg1..cfg5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workloads (BASELINE.json configs; default cfg2 = the configuration the metric is quoted on):
    cfg1  100 k x 50 nt SE vs 5 Mb genome,        -s 16 -v 2 -I 4          (the reference's own CPU-runnable case)
    cfg2  20 M x 100 nt SE vs 3.1 Gb genome,      -s 16 -v 5 -I 4          (headline)
    cfg3  10 M x 2x100 nt PE vs 3.1 Gb genome,    -m 28 -x 500             (PairAlign on the device; unit = pairs)
    cfg4  10 M x 75 nt RRBS vs 3.1 Gb genome,     -D C-CGG -A <adapter>    (seed 12, interval 1, adapter trimming)
    cfg5  1 M x 144 nt SE vs 3.1 Gb genome,       -s 12 -v 15 -w 1000      (planted 2 000-copy repeat; wide-context kernel)
Genomes and reads are synthetic (counter-based generators, bsmap_b200/synth.py), generated in HBM.

One step = one pass of the hot path (trim / pack / seed selection / probe / extension / best-hit selection [/ pairing])
over the whole read set of a rank.  Reads shard across ranks (independent units, no collective on the data path):
weak scaling, every rank maps its own read set against its own replica of the index, which rank 0 builds and
broadcasts once over NVLink (NCCL, outside the timed region).

    value     units/s, inputs resident in HBM, CUDA events around K launches of the mapping kernel
    e2e       same metric through the C ABI with pinned HOST buffers (bsx_map_*_packed: 2-bit reads in, records out;
              H2D + kernel + D2H inside the timed region); e2e.ascii = the ASCII entry point (bsx_map_se / bsx_map_pe)
    roofline  algorithmic bytes (SURVEY.md 8(d): B = mates*2*ceil(L/4) + 12 P + C (4 + L/4) + 32 per unit, with the kernel's
              exact C counter and the header count P) / kernel time vs the measured HBM copy peak
    cpu_baseline  the oracle port (oracle/bsmap_oracle.c) on the host cores over a bounded sample of the same reads;
              EVERY record of the sample is compared with the GPU's
    strong    (N > 1, cfg2) rank 0's read set sharded over the N ranks, mapped end to end, gathered, merged in input
              order on the host and compared with rank 0's own single-GPU records: the multi-GPU product path

--impl reference times the CPU implementation with all host threads: the oracle port by default (index arrays
imported, mapping only), or with --reference-binary the UNMODIFIED reference (oracle/_ref/bsmap -p <threads>) on the
first 1 M reads of cfg2, whose 280-s single-threaded seed-table build is reported separately (BASELINE.md 3).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ADAPTER = "AGATCGGAAGAGCGGTTCAGCAGGAATGCCGAGA"
BIG = [124_000_000] * 25

CONFIGS = {
    "cfg1": dict(kind="se", gseed=1, lens=[1_000_000] * 5, n=100_000, L=50, stride=56, rseed=11, subs="cfg1", opts=dict(s=16, v=2, I=4, S=7),
                 desc="5x1Mb synthetic genome, {n} x 50nt SE reads per GPU per step, -s 16 -v 2 -I 4"),
    "cfg2": dict(kind="se", gseed=2, lens=BIG, n=20_000_000, L=100, stride=104, rseed=2024, subs="cfg2", opts=dict(s=16, v=5, I=4, S=7),
                 desc="25x124Mb synthetic genome, {n} x 100nt SE reads per GPU per step, -s 16 -v 5 -I 4"),
    "cfg3": dict(kind="pe", gseed=2, lens=BIG, n=10_000_000, L=100, stride=104, rseed=33, subs="cfg2", opts=dict(s=16, v=2, I=4, m=28, x=500, S=7, pairend=1),
                 desc="25x124Mb synthetic genome, {n} x 2x100nt PE pairs per GPU per step (fragments 150-450), -s 16 -v 2 -I 4 -m 28 -x 500"),
    "cfg4": dict(kind="rrbs", gseed=2, lens=BIG, n=10_000_000, L=75, stride=80, rseed=44, subs=None, opts=dict(D="C-CGG", v=2, S=5, A=[ADAPTER]),
                 desc="25x124Mb synthetic genome, {n} x 75nt RRBS reads per GPU per step (C-CGG fragments 40-400, adapter read-through), -D C-CGG -v 2 -A"),
    "cfg5": dict(kind="se", gseed=5, lens=BIG, repeats=2000, n=1_000_000, L=144, stride=144, rseed=55, subs="cfg5", opts=dict(s=12, v=15, I=4, w=1000, S=7),
                 desc="25x124Mb synthetic genome with a planted 2000-copy repeat, {n} x 144nt SE reads per GPU per step, -s 12 -v 15 -I 4 -w 1000"),
}
CPU_UNITS_PER_THREAD = {"cfg2": 40_000, "cfg1": 100_000, "cfg3": 6_000, "cfg4": 100_000, "cfg5": 150}   # ~1 s of oracle work per thread


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 5; --reference-binary: 1)")
    ap.add_argument("--warmup", type=int, default=None, help="untimed steps before them (default 3; --reference-binary: 0)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--reads", type=int, default=0, help="units (reads / pairs) per GPU per step (0 = the config's)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="units in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling / merge leg (N > 1)")
    ap.add_argument("--batch", type=int, default=1 << 20, help="sub-batch of the end-to-end pipeline")
    ap.add_argument("--reference-binary", action="store_true", help="--impl reference: run the unmodified oracle/_ref/bsmap (cfg2, first 1 M reads)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the records of the last timed step for rank 0's read set as DIR/<array>_<field>.npy (float64; a "
                         "fixed, seeded sample of the units when all of them would exceed 64 MB, their positions in DIR/unit_index.npy)")
    a = ap.parse_args()
    if a.reference_binary:
        # one run of the binary is one step: every run repeats its FASTA load and seed-table build (minutes at 3.1 Gb)
        if a.steps not in (None, 1) or a.warmup not in (None, 0):
            ap.error("--reference-binary times one run of the binary: --steps 1 --warmup 0")
        a.steps, a.warmup = 1, 0
    a.steps = 5 if a.steps is None else a.steps
    a.warmup = 3 if a.warmup is None else a.warmup
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.reference_binary:
        ap.error("--dump-outputs: the reference binary's output is SAM text, not records")
    return a


DUMP_BYTES = 64_000_000


def dump_outputs(path, arrays, first):
    """Every field of the record arrays (same length, one entry per unit) as float64 .npy files, exact for the u32 / i32 /
    u8 fields.  When they exceed DUMP_BYTES, a sorted sample of units drawn with a fixed seed: the same units every run,
    so two builds can be compared output for output.  unit_index.npy holds the units' global indices (first + row)."""
    n = len(next(iter(arrays.values())))
    fields = [(name, f) for name, arr in arrays.items() for f in arr.dtype.names]
    k = min(n, (DUMP_BYTES - 128 * (len(fields) + 1)) // (8 * (len(fields) + 1)))     # 128: the .npy header of a 1-D array
    rows = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "unit_index.npy"), (first + rows).astype(np.float64))
    for name, f in fields:
        np.save(os.path.join(path, f"{name}_{f}.npy"), arrays[name][f][rows].astype(np.float64))


class _DevBuf:
    """zero-copy torch view of a raw device pointer (for the NCCL index broadcast)"""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class ClockSampler:
    """nvidia-smi clocks and throttle reasons during the timed region (B200_PROFILING.md)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.p, self.lines = gpu, None, []

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for ln in self.p.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_map_parallel(oref, op, kind, bufs, lens, first_index, threads):
    """oracle port over `threads` host threads (ctypes releases the GIL) -> (seconds, stats, list of record arrays)"""
    from concurrent.futures import ThreadPoolExecutor
    n = len(lens)
    cuts = np.linspace(0, n, threads + 1).astype(int)
    stats, parts = [], [None] * threads

    def work(i):
        a, b = int(cuts[i]), int(cuts[i + 1])
        if b <= a:
            return
        if kind == "pe":
            pr, ra, rb, _, _, st = oref.map_pe(bufs[0][a:b], lens[a:b], bufs[1][a:b], lens[a:b], first_index=first_index + a, params=op)
            parts[i] = (pr, ra, rb)
        else:
            r, _, st = oref.map_se(bufs[0][a:b], lens[a:b], first_index=first_index + a, want_counts=False, params=op)
            parts[i] = (r,)
        stats.append(st)

    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(work, range(threads)))
    dt = time.perf_counter() - t0
    parts = [p for p in parts if p is not None]
    return dt, np.sum(stats, axis=0), [np.concatenate([p[k] for p in parts]) for k in range(len(parts[0]))]


def bind_near_gpu(torch, local):
    """Host side of the end-to-end path: run this rank (and first-touch its pinned buffers) on the CPUs of the NUMA
    node its GPU hangs off, so that eight ranks do not pull their input through one socket.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1} & os.sched_getaffinity(0)
        if cpus and len(cpus) < len(os.sched_getaffinity(0)):
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def run_reference_binary(a, cfg, names, genome, make_reads, synth):
    """The UNMODIFIED reference on the first 1 M reads of the workload, -p <host threads>: phases from its own progress
    lines stamped with the wall clock (BASELINE.md 2/3)."""
    import tempfile
    import oracle_lib as O
    import scale_cases as SC
    T = host_threads()
    n = min(1_000_000, a.reads or cfg["n"])
    td = tempfile.mkdtemp(prefix="bsx_ref_")
    fa, fq, sam = (os.path.join(td, f) for f in ("ref.fa", "reads.fq", "out.sam"))
    synth.write_fasta(fa, genome, names)
    seq = make_reads(0, n)[0].cpu().numpy()
    sim_names = SC.se_read_names(genome, SC.SE, 0, n) if n <= SC.SE["n"] else [f"r{i}" for i in range(n)]
    synth.write_fastq(fq, seq[:, :cfg["L"]], sim_names)
    o = cfg["opts"]
    args = [O.REF_BIN, "-a", fq, "-d", fa, "-o", sam, "-s", o["s"], "-v", o["v"], "-I", o["I"], "-S", o["S"], "-p", T]
    t0 = time.perf_counter()
    p = subprocess.Popen([str(x) for x in args], cwd=td, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    stamps = [(time.perf_counter() - t0, ln.rstrip("\n")) for ln in p.stdout]
    if p.wait() != 0:
        raise SystemExit(f"reference binary failed: {stamps[-3:]}")
    t_load = next(t for t, ln in stamps if ln.startswith("Load in"))
    t_tab = next(t for t, ln in stamps if ln.startswith("Create seed table") or ln.startswith("max mismatches"))
    t_done = next(t for t, ln in stamps if ln.startswith("Done."))
    dig, nl = SC.sorted_sam_digest(open(sam, "rb").read())
    for f in (fa, fq, sam):
        os.remove(f)
    os.rmdir(td)
    info = dict(reads=n, threads=T, fasta_load_s=t_load, seed_table_s=t_tab - t_load, mapping_s=t_done - t_tab,
                reads_per_s=n / (t_done - t_tab), sorted_sam_sha256=dig, sam_lines=nl)
    try:   # the same digest the CUDA path reproduces in tests/test_scale_gpu.py
        info["equals_committed_golden"] = dig == json.load(open(SC.REFRUN))["sorted_sam_sha256"]
    except Exception:
        pass
    return info


def main():
    a = parse()
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    if a.impl == "reference" and rank != 0:
        return 0
    import torch
    import torch.distributed as dist
    import bsmap_b200 as B
    from bsmap_b200 import shard, synth
    from bsmap_b200.lib import PAIR_REC, REC

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = bind_near_gpu(torch, local) if world > 1 else 0
    multi = world > 1 and a.impl == "ours"
    if multi:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    cfg = CONFIGS[a.config]
    kind, L, STRIDE = cfg["kind"], cfg["L"], cfg["stride"]
    pe = kind == "pe"
    unit = "pairs/s" if pe else "reads/s"
    lens = list(cfg["lens"])
    names = [f"chr{i + 1}" for i in range(len(lens))]
    n = a.reads or cfg["n"]
    t_setup = time.perf_counter()

    # ---- synthetic genome on the GPU; host copy only where the index is built
    genome = synth.make_genome(cfg["gseed"], lens, device=dev)
    if cfg.get("repeats"):
        genome = synth.plant_repeats(genome, cfg["gseed"], unit_len=300, copies=cfg["repeats"], divergence=0.03)
    p = B.make_params(**cfg["opts"])
    build_s, bcast_s, host_g = None, None, None
    if (rank == 0 or not multi) and not a.reference_binary:
        host_g = [torch.empty(ln, dtype=torch.uint8, pin_memory=True) for ln in lens]
        for h, g in zip(host_g, genome):
            h.copy_(g)
        torch.cuda.synchronize()
        ix = B.Index.from_pointers(p, names, [h.data_ptr() for h in host_g], lens, device=local)
        build_s = ix.info.build_seconds
        if kind != "rrbs":
            host_g = None            # RRBS: the CPU checker builds its own index from the text
    if multi:
        # one-time index broadcast over NVLink: metadata by object broadcast, arrays by NCCL broadcast
        meta = shard.broadcast_blob(ix.meta() if rank == 0 else None, src=0, device=dev)
        if rank != 0:
            ix = B.Index.shell(p, meta, local)
        t_b = time.perf_counter()
        shard.broadcast_buffers([torch.as_tensor(_DevBuf(ptr, nbytes), device=dev) for ptr, nbytes in ix.device_buffers() if nbytes], src=0)
        torch.cuda.synchronize()
        bcast_s = time.perf_counter() - t_b

    # ---- simulated reads, generated in HBM: make_reads(first, count) -> [mate a (, mate b)] uint8[count, STRIDE]
    frags = synth.rrbs_fragments(genome) if kind == "rrbs" else None

    def make_reads(first, count):
        outs = [torch.zeros((count, STRIDE), dtype=torch.uint8, device=dev) for _ in range(2 if pe else 1)]
        CH = 1 << 20
        for s0 in range(0, count, CH):
            m = min(CH, count - s0)
            if pe:
                sim = synth.simulate_pairs(genome, m, L, seed=cfg["rseed"], frag_min=150, frag_max=450, subs=cfg["subs"], first_index=first + s0)
                outs[0][s0:s0 + m, :L] = sim["seq1"]; outs[1][s0:s0 + m, :L] = sim["seq2"]
            elif kind == "rrbs":
                outs[0][s0:s0 + m, :L] = synth.simulate_rrbs_reads(genome, frags, m, L, cfg["rseed"], ADAPTER.encode(), first_index=first + s0)
            else:
                outs[0][s0:s0 + m, :L] = synth.simulate_reads(genome, m, L, seed=cfg["rseed"], subs=cfg["subs"], first_index=first + s0)["seq"]
        return outs

    metric = {"cfg2": "wgbs_100nt_reads_mapped_per_sec", "cfg1": "wgbs_50nt_reads_mapped_per_sec", "cfg3": "wgbs_2x100nt_pairs_mapped_per_sec",
              "cfg4": "rrbs_75nt_reads_mapped_per_sec", "cfg5": "wgbs_144nt_v15_reads_mapped_per_sec"}[a.config]

    if a.impl == "reference" and a.reference_binary:
        if a.config != "cfg2":
            raise SystemExit("--reference-binary is set up for cfg2")
        info = run_reference_binary(a, cfg, names, genome, make_reads, synth)
        val = info["reads_per_s"]
        print(json.dumps({"metric": metric, "value": val, "unit": unit, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                          "ms_per_step": 1e3 * info["mapping_s"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
                          "data": "synthetic", "impl": "reference", "config": {"workload": "cfg2: " + cfg["desc"].format(n=info["reads"])},
                          "cpu_baseline": {"value": val, "unit": unit, "cores": info["threads"], "kind": "reference",
                                           "sample": f"first {info['reads']} reads; mapping phase only (FASTA load {info['fasta_load_s']:.0f} s and the single-threaded "
                                                     f"seed-table build {info['seed_table_s']:.0f} s reported apart)"},
                          "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "reference_binary": info, "gpu_launches": 0}))
        return 0

    first_index = rank * n
    seqs_dev = make_reads(first_index, n)
    if os.environ.get("BSX_BENCH_REPEAT_READS"):
        # diagnostic only (never a bench value): the first K reads repeated, so that every table / list / image access
        # hits cache -- same instruction stream, no DRAM; tells how far the memory system holds the kernel back
        k = int(os.environ["BSX_BENCH_REPEAT_READS"])
        for t in seqs_dev:
            t[:] = t[:k].repeat((n + k - 1) // k, 1)[:n]
    do_strong = multi and not a.no_strong and a.config == "cfg2"
    if not do_strong:
        del genome
        frags = None
    torch.cuda.empty_cache()

    def pin(t):
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t)
        return h

    seq_host = [pin(t) for t in seqs_dev]
    len_host = pin(torch.full((n,), L, dtype=torch.int16, device=dev))
    torch.cuda.synchronize()
    del seqs_dev
    torch.cuda.empty_cache()
    # packed form of the same reads (2-bit bases + valid mask): what the end-to-end leg uploads
    L_ = B.lib.load()
    PS = int(L_.bsx_packed_stride(STRIDE))
    pk_host = []
    for h in seq_host:
        pk = torch.empty((n, PS), dtype=torch.uint8, pin_memory=True)
        B.lib.check(L_.bsx_pack_reads(n, h.data_ptr(), STRIDE, len_host.data_ptr(), pk.data_ptr(), None, 0))
        pk_host.append(pk)
    rec_host = torch.empty((n, 16), dtype=torch.uint8, pin_memory=True)
    recb_host = torch.empty((n, 16), dtype=torch.uint8, pin_memory=True) if pe else None
    pair_host = torch.empty((n, 28), dtype=torch.uint8, pin_memory=True) if pe else None
    setup_s = time.perf_counter() - t_setup

    conf = {"workload": f"{a.config}: " + cfg["desc"].format(n=n),
            "l2_policy": ("working set larger than L2 (index + reads per step vs 126 MB L2)" if sum(lens) > 1e9 else
                          "the index of this small genome is L2-resident by nature of the config; reads stream from HBM"),
            "units_per_gpu_per_step": n, "genome_bp": sum(lens), "e2e_input": f"packed 2-bit read slots, {PS} B per read (ASCII slots: {STRIDE} B)",
            "resident_input": f"`value`: the packed slots resident in HBM (the device batch format of the product path); `value_ascii_resident`: {STRIDE}-byte ASCII slots resident"}
    if numa_cpus:
        conf["host_binding"] = f"each rank pinned to the {numa_cpus} CPUs NVML reports as local to its GPU (pinned buffers first-touched there)"

    def oracle_for_sample():
        """the CPU checker for this workload: the port over imported index arrays (WGBS), or its own build (RRBS)"""
        import oracle_lib as O
        op = O.make_params(**cfg["opts"])
        if kind == "rrbs":
            return O, op, O.OracleRef(op, names, [h.numpy() for h in host_g])
        arrs = [ix.download(w) for w in ("refcat", "crefcat", "tab", "pos")]
        return O, op, O.OracleRef.imported(op, names, lens, *arrs)

    def gpu_records_host(mapper):
        """records of the whole read set through the ASCII entry point, as numpy"""
        if pe:
            pr = np.empty(n, dtype=PAIR_REC); ra = np.empty(n, dtype=REC); rb = np.empty(n, dtype=REC)
            mapper.map_pe_ptr(n, seq_host[0].data_ptr(), len_host.data_ptr(), seq_host[1].data_ptr(), len_host.data_ptr(),
                              pr.ctypes.data, ra.ctypes.data, rb.ctypes.data, first_index=first_index)
            return [pr, ra, rb]
        r = np.empty(n, dtype=REC)
        mapper.map_se_ptr(n, seq_host[0].data_ptr(), len_host.data_ptr(), r.ctypes.data, first_index=first_index)
        return [r]

    def count_diff(orecs, grecs, lo, hi):
        return int(sum(int((o != g[lo:hi].astype(o.dtype)).sum()) for o, g in zip(orecs, grecs)))

    # =====================================================================================
    if a.impl == "reference":
        # CPU arm: the oracle port with every host thread, on bounded samples of the same reads; every record it produces is
        # compared with the GPU's record for the same read (computed outside the timed region)
        gm = B.Mapper(ix, p, max_batch=min(n, 1 << 20), stride=STRIDE)
        grecs = gpu_records_host(gm)
        gm.close()
        O, op, oref = oracle_for_sample()
        ix.close()
        T = host_threads()
        sample = a.cpu_sample or min(n, CPU_UNITS_PER_THREAD[a.config] * T)
        bufs = [h.numpy() for h in seq_host]; ln = len_host.numpy().view(np.uint16)
        times, compared, differing = [], 0, 0
        for it in range(a.warmup + a.steps):
            s0 = (it * sample) % max(1, n - sample + 1)
            dt, _, orecs = cpu_map_parallel(oref, op, kind, [b[s0:s0 + sample] for b in bufs], ln[s0:s0 + sample], first_index + s0, T)
            compared += sample
            differing += count_diff(orecs, grecs, s0, s0 + sample)
            if it >= a.warmup:
                times.append(dt)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, dict(zip(("pairs", "recs_a", "recs_b") if pe else ("recs",), orecs)), first_index + s0)
        tot = sum(times)
        val = sample * a.steps / tot
        line = {"metric": metric, "value": val, "unit": unit, "n_gpus": a.gpus, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": 1e3 * tot / a.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": conf, "impl": "reference",
                "cpu_baseline": {"value": val, "unit": unit, "cores": T, "kind": "port",
                                 "sample": f"{sample} units per step of the same read set; " + ("oracle's own index build" if kind == "rrbs" else "index arrays imported") + " (mapping only)",
                                 "records_compared_with_gpu": compared, "records_differing_from_gpu": differing},
                "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # =====================================================================================
    mp = B.Mapper(ix, p, max_batch=n, stride=STRIDE)
    # the kernel is launched on this (non-default) torch stream, so torch.cuda.Event brackets it
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    def upload_resident(packed):
        src, up = (pk_host, mp.upload_packed) if packed else (seq_host, mp.upload)
        if pe:
            up(n, src[0].data_ptr(), len_host.data_ptr(), src[1].data_ptr(), len_host.data_ptr(), stream=stream)
        else:
            up(n, src[0].data_ptr(), len_host.data_ptr(), stream=stream)
        torch.cuda.synchronize()
    run = (lambda: mp.run_pe(n, first_index=first_index, stream=stream)) if pe else (lambda: mp.run_se(n, first_index=first_index, stream=stream))

    def barrier():
        if multi:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_resident():
        for _ in range(a.warmup):
            run()
        barrier()
        mp.stats(reset=True)
        l0 = mp.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(tstream)
        for _ in range(a.steps):
            run()
        e1.record(tstream)
        barrier()
        return e0.elapsed_time(e1), mp.launches - l0

    # ---- kernel-only: inputs resident in HBM.  First as ASCII slots (what the reference-facing bsx_map_se takes), then --
    # the headline `value` -- as the packed 2-bit slots the product path keeps on the device (bsx_map_se_packed)
    clocks = ClockSampler(local); clocks.start()
    upload_resident(False)
    ms_ascii, launches_value_ascii = timed_resident()
    upload_resident(True)
    ms, launches_value = timed_resident()
    st = mp.stats(reset=True)
    if pe:
        pr_d = np.empty(n, dtype=PAIR_REC); ra_d = np.empty(n, dtype=REC); rb_d = np.empty(n, dtype=REC)
        B.lib.check(L_.bsx_batch_download_pe(mp.h, n, pr_d.ctypes.data, ra_d.ctypes.data, rb_d.ctypes.data, None, None, stream))
        recs_dev = [pr_d, ra_d, rb_d]
        mapped_frac = float(pr_d["paired"].mean())
    else:
        r_d, _ = mp.download_se(n, stream=stream)
        recs_dev = [r_d]
        mapped_frac = float((r_d["nhits"] > 0).mean())
    mp.close()

    # ---- end to end: pinned host buffers in (packed 2-bit reads), host records out, every step
    small = B.Mapper(ix, p, max_batch=min(n, a.batch), stride=STRIDE)

    def e2e_call(packed):
        src = pk_host if packed else seq_host
        if pe:
            f = L_.bsx_map_pe_packed if packed else L_.bsx_map_pe
            B.lib.check(f(small.h, n, src[0].data_ptr(), len_host.data_ptr(), src[1].data_ptr(), len_host.data_ptr(), first_index,
                          pair_host.data_ptr(), rec_host.data_ptr(), recb_host.data_ptr(), None, None))
        else:
            f = L_.bsx_map_se_packed if packed else L_.bsx_map_se
            B.lib.check(f(small.h, n, src[0].data_ptr(), len_host.data_ptr(), first_index, 0, rec_host.data_ptr(), None))

    def e2e_time(packed):
        for _ in range(max(1, a.warmup // 2)):
            e2e_call(packed)
        barrier()
        l1 = small.launches
        t0 = time.perf_counter()
        for _ in range(a.steps):
            e2e_call(packed)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        got = [pair_host.numpy().view(PAIR_REC).reshape(-1), rec_host.numpy().view(REC).reshape(-1), recb_host.numpy().view(REC).reshape(-1)] if pe \
            else [rec_host.numpy().view(REC).reshape(-1)]
        same = all(bool(np.array_equal(g, r)) for g, r in zip(got, recs_dev))
        return dt, small.launches - l1, same

    e2e_s, launches_e2e, same = e2e_time(True)
    e2e_ascii_s, launches_ascii, same_ascii = e2e_time(False)
    clk = clocks.stop()

    # ---- strong scaling + in-order merge across the ranks (the multi-GPU product path): rank 0's read set, sharded
    strong = None
    if do_strong:
        share = n // world
        lo = rank * share
        mine = make_reads(lo, share)[0]                    # reads lo .. lo+share of the set rank 0 mapped above (first_index 0)
        mine_h = pin(mine); del mine
        pk = torch.empty((share, PS), dtype=torch.uint8, pin_memory=True)
        B.lib.check(L_.bsx_pack_reads(share, mine_h.data_ptr(), STRIDE, len_host.data_ptr(), pk.data_ptr(), None, 0))
        out = torch.empty((share, 16), dtype=torch.uint8, pin_memory=True)

        def call():
            B.lib.check(L_.bsx_map_se_packed(small.h, share, pk.data_ptr(), len_host.data_ptr(), lo, 0, out.data_ptr(), None))
        call()
        barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            call()
        torch.cuda.synchronize()
        dt = shard.reduce_max([time.perf_counter() - t0], device=dev)[0]
        parts = shard.gather_records(out.numpy().view(REC).reshape(-1), device=dev)
        if rank == 0:
            merged = shard.merge_in_order(share * world, world, share, parts)
            strong = {"value": share * world * a.steps / dt, "unit": unit, "reads_total_per_step": share * world, "ms_per_step": 1e3 * dt / a.steps,
                      "what": f"one {share * world}-read set sharded over {world} ranks, end to end from packed host buffers; records gathered and merged "
                              "in input order on the host",
                      "merged_records_equal_single_gpu_run": bool(np.array_equal(merged, recs_dev[0][:share * world]))}
    small.close()

    # max over ranks
    ms, ms_ascii, e2e_s, e2e_ascii_s = shard.reduce_max([ms, ms_ascii, e2e_s, e2e_ascii_s], device=dev)
    tot_c, tot_p, tot_over, tot_full, tot_list, tot_gather = shard.reduce_sum(
        [st[k] for k in ("candidates", "probes", "overfetch", "full_extensions", "list_entries", "gathers")], device=dev)
    units_total = n * world * a.steps
    value = units_total / (ms * 1e-3)
    e2e_val = units_total / e2e_s

    # ---- roofline of the mapping kernel (per launch, this rank's view scaled by world)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    c_per = tot_c / units_total
    p_per = tot_p / units_total
    mates = 2 if pe else 1
    bytes_per_unit = mates * 2 * ((L + 3) // 4) + 12 * p_per + c_per * (4 + L / 4) + 32
    kernel_s = (ms * 1e-3) / a.steps
    achieved = bytes_per_unit * n / kernel_s / 1e9
    kname = ("bsx_map_pe_rrbs_kernel" if kind == "rrbs" else "bsx_map_pe_wgbs_kernel") if pe else ("bsx_map_se_rrbs_kernel" if kind == "rrbs" else
                                            ("bsx_map_se_wide_kernel" if cfg["opts"].get("v", 2) >= 8 else "bsx_map_se_wgbs_kernel"))
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
            "peak_source": peak_src, "kernel": kname, "algorithmic_bytes_per_unit": bytes_per_unit,
            "candidates_per_unit": c_per, "headers_per_unit": p_per,
            "overfetch_per_unit": tot_over / units_total, "full_extensions_per_unit": tot_full / units_total,
            "hbm_gathers_per_unit": tot_gather / units_total}
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        k = prof.get("kernels", {}).get(kname)
        if k:
            roof["traffic"] = k["dram_bytes_per_unit"] * n
            roof["traffic_source"] = k.get("source", "") + " -- an ncu capture scaled by the units of one launch, not a measurement of this run"
    except Exception:
        pass

    # ---- CPU baseline (rank 0, N = 1 only): oracle port on a bounded sample, mapping only; every record compared
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        O, op, oref = oracle_for_sample()
        T = host_threads()
        sample = a.cpu_sample or min(n, CPU_UNITS_PER_THREAD[a.config] * T)
        bufs = [h.numpy() for h in seq_host]; ln = len_host.numpy().view(np.uint16)
        dt, ost, orecs = cpu_map_parallel(oref, op, kind, [b[:sample] for b in bufs], ln[:sample], first_index, T)
        cpu = {"value": sample / dt, "unit": unit, "cores": T, "kind": "port",
               "sample": f"first {sample} units of the step ({dt:.1f} s wall on {T} threads); " +
                         ("oracle's own index build" if kind == "rrbs" else "index arrays imported") + " (mapping only)",
               "candidates_per_unit": float(ost[0]) / sample, "headers_per_unit": float(ost[1]) / sample,
               "records_compared_with_gpu": int(sample), "records_differing_from_gpu": count_diff(orecs, recs_dev, 0, sample)}
        if a.config == "cfg2":
            try:
                ref = json.load(open(os.path.join(ROOT, "tests", "golden", "scale", "cfg2_reference_binary.json")))
                cpu["unmodified_reference_binary"] = {
                    "reads_per_s": ref["reads_per_s"], "threads": ref["host_threads"], "seed_table_s": ref["seed_table_s"],
                    "note": "oracle/_ref/bsmap on this genome and the first 1 M reads, measured in the CPU container when the golden was generated "
                            "(tests/golden/make_scale_golden.py); not a measurement of this run -- `--impl reference --reference-binary` measures it here"}
            except Exception:
                pass
        oref.close()

    if rank == 0:
        if a.dump_outputs:
            # recs_dev: downloaded after the last launch of the timed packed-resident loop that `value` measures
            dump_outputs(a.dump_outputs, dict(zip(("pairs", "recs_a", "recs_b") if pe else ("recs",), recs_dev)), first_index)
        h2d = n * mates * (PS + 2)
        d2h = n * (16 if not pe else 28 + 32)
        line = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u32", "data": "synthetic", "config": conf, "clocks": clk,
                "value_ascii_resident": units_total / (ms_ascii * 1e-3),
                "e2e": {"value": e2e_val, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": 1e3 * e2e_s / a.steps, "records_identical_to_resident_run": same,
                        "ascii": {"value": units_total / e2e_ascii_s, "h2d_bytes_per_step": n * mates * (STRIDE + 2), "records_identical_to_resident_run": same_ascii}},
                "gpu_launches": int(launches_value + launches_value_ascii + launches_e2e + launches_ascii),
                "roofline": roof, "cpu_baseline": cpu, "strong": strong,
                "mapped_fraction": mapped_frac, "index_build_seconds": build_s, "index_broadcast_seconds": bcast_s,
                "setup_seconds": setup_s}
        print(json.dumps(line))
    ix.close()
    if multi:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
