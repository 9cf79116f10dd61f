#!/usr/bin/env python
"""Randomised differential test of methratio on the device: the text pile-up kernels (plain, Cycles, Snp, Conv), the
-r claims, the -g combine and region kernels and the table / region / M-bias / conversion writers of bsx_meth.cu,
against the composed numpy oracles (oracle/conversion_oracle.py, ctsnp_oracle.py, region_oracle.py, mbias_oracle.py).

The inputs are generated rather than written by BSMAP, so they hold what BSMAP never prints: sequences of 1-5 bases and
lengths at multiples of 16 and one either side; lowercase, N and IUPAC runs in the reference; alignments that end at or
one past the sequence end; reads of 1-700 bases and '*'; N, lowercase and '=' in reads; inserts shorter than the read;
PNEXT before, inside and after the read; the FLAG bits the filters read; records on sequences the FASTA lacks; exact
duplicates and shared fragment ends for -r.  Options are drawn from every combination the command line accepts, and
the alignments go in over 1-6 batches (empty and one-alignment batches included).  Every round compares exactly: the
counters and the C/T SNP evidence, the valid count, the M-bias bins and overflow, the conversion bins and dropped
count, the region sums, and the bytes of the table, the summary line and the region, M-bias and conversion reports.

    python tests/meth_fuzz.py [--rounds 40] [--seed 1]
"""
import argparse
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))   # repo root (this script lives in tests/)
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)
import conversion_oracle as CV   # noqa: E402  (test infrastructure: the checker)
import mbias_oracle as MB        # noqa: E402
import region_oracle as RO       # noqa: E402
from meth_inputs import api_arrays    # noqa: E402
from test_region_cpu import random_regions   # noqa: E402
from bsmap_b200 import synth     # noqa: E402

NAME_POOL = ["chr1", "chr2", "chr10", "chrX", "Chr_3", "MT", "scaffold_7", "lambda", "c.1", "seqA"]
UNKNOWN = "chrUn_fuzz"                   # a sequence name the FASTA lacks
IUPAC = b"RYKMSWBDHVNrykn"
STRANDS = ("++", "+-", "-+", "--")
FLAG_LETTERS = "pPuUrR12sfd"             # samtools view -X: one letter per FLAG bit, 0x1 .. 0x400
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
A, C, G, T = (ord(x) for x in "ACGT")


# ---- reference ------------------------------------------------------------------------------------------------------
def make_reference(rng, n_seq=None, big=(10_000, 400_000)):
    """-> (names, sequences as bytes): 1-5 sequences of 1-5 bases, 16k - 1 .. 16k + 1 or 10-400 kb, with lowercase, N
    and IUPAC runs; the names are unique and often not in sorted order"""
    n = n_seq or int(rng.integers(1, 6))
    names = [str(x) for x in rng.choice(NAME_POOL, n, replace=False)]
    lens = []
    for _ in range(n):
        u = rng.random()
        if u < 0.25:
            lens.append(int(rng.integers(1, 6)))
        elif u < 0.55:
            lens.append(max(1, 16 * int(rng.integers(1, 1200)) + int(rng.integers(-1, 2))))
        else:
            lens.append(int(rng.integers(*big)))
    seqs = []
    for t in synth.make_genome(int(rng.integers(1, 1 << 30)), lens):
        b = bytearray(t.numpy().tobytes())
        L = len(b)
        for _ in range(int(rng.integers(0, 4))):
            s = int(rng.integers(0, L)); e = min(L, s + int(rng.integers(1, 3000)))
            b[s:e] = bytes(b[s:e]).lower()
        for _ in range(int(rng.integers(0, 3))):
            s = int(rng.integers(0, L)); e = min(L, s + int(rng.integers(1, 200)))
            b[s:e] = b"N" * (e - s)
        for _ in range(int(rng.integers(0, 30))):
            b[int(rng.integers(0, L))] = IUPAC[int(rng.integers(0, len(IUPAC)))]
        seqs.append(bytes(b))
    return names, seqs


def write_fasta(path, names, seqs):
    with open(path, "wb") as f:
        for n, s in zip(names, seqs):
            f.write(b">" + n.encode() + b"\n")
            for i in range(0, len(s), 60):
                f.write(s[i:i + 60] + b"\n")


# ---- alignments -----------------------------------------------------------------------------------------------------
def read_at(rng, ref, pos, L, strand, conv, snps):
    """SEQ as printed for a hit of L bases at pos: the reference (random bases past its end and for non-ACGT), the
    planted C/T SNPs on the opposite strand, bisulfite conversion on the hit's strand, then substitutions, N, '=' and
    lowercase"""
    if L == 0:
        return "*"
    seg = np.frombuffer(ref[pos:pos + L], dtype=np.uint8).copy()
    a = np.concatenate([seg, ACGT[rng.integers(0, 4, L - len(seg))]]) if len(seg) < L else seg
    bad = ~np.isin(a, ACGT)
    a[bad] = ACGT[rng.integers(0, 4, int(bad.sum()))]
    for q in snps:
        if pos <= q < pos + L and rng.random() < 0.7:
            j = q - pos
            if strand[0] == "+" and a[j] == G:
                a[j] = A
            elif strand[0] == "-" and a[j] == C:
                a[j] = T
    hit = a == (C if strand[0] == "+" else G)
    a[hit & (rng.random(L) < conv)] = T if strand[0] == "+" else A
    sub = rng.random(L) < 0.01
    a[sub] = np.frombuffer(b"ACGTN", dtype=np.uint8)[rng.integers(0, 5, int(sub.sum()))]
    if rng.random() < 0.05:
        a[rng.random(L) < 0.05] = ord("=")
    if rng.random() < 0.05:
        s = int(rng.integers(0, L)); e = min(L, s + int(rng.integers(1, 40)))
        a[s:e] = np.frombuffer(bytes(a[s:e]).lower(), dtype=np.uint8)
    return bytes(a).decode()


def read_length(rng, size):
    u = rng.random()
    if size < 16 and u < 0.7:
        return int(rng.integers(1, size + 1))
    if u < 0.03:
        return 0                                                        # SEQ '*'
    if u < 0.08:
        return int(rng.integers(1, 13))                                 # shorter than some -t
    if u < 0.12:
        return int(rng.integers(151, 701))                              # past BSX_MBIAS_CYCLES
    return int(rng.integers(30, 151))


def make_records(rng, names, seqs, n, rm_dup=False, dup_frac=0.15, conv=0.75):
    """-> list of alignments {qname, flag (SAM FLAG), chrom, pos (0-based), strand, insert, pnext (1-based, 0 = none),
    seq}.  With rm_dup, no alignment on a FASTA sequence has its -r fragment end outside [0, size): the script raises
    IndexError there."""
    up = [s.upper() for s in seqs]
    hot = [rng.integers(0, len(s), size=3).tolist() for s in seqs]    # most reads pile up near these, for depth
    snps = [[min(len(s) - 1, h + int(d)) for h in hs for d in rng.integers(0, 300, 4)] for s, hs in zip(seqs, hot)]
    out = []
    for i in range(n):
        if out and rng.random() < dup_frac:                              # -r: exact duplicates, and shared fragment ends
            r = dict(out[int(rng.integers(0, len(out)))])
            r["qname"] = "d%d" % i
            if rng.random() < 0.5:
                k = names.index(r["chrom"]) if r["chrom"] in names else 0
                L = max(1, read_length(rng, len(seqs[k])))
                if r["strand"] in ("+-", "-+"):                          # the same end: pos + len stays
                    end = r["pos"] + len(r["seq"]) if r["seq"] != "*" else r["pos"] + 1
                    if end - L < 0:
                        L = end
                    r["pos"] = end - L
                r["seq"] = read_at(rng, up[k], r["pos"], L, r["strand"], conv, snps[k]) if L else "*"
                r["flag"] = int(r["flag"]) ^ (0x80 if rng.random() < 0.5 else 0)
            out.append(r)
            continue
        k = int(rng.integers(0, len(names)))
        size = len(seqs[k])
        L = read_length(rng, size)
        span = max(L, 1)
        u = rng.random()
        if u < 0.1 and size - 1 - span >= 0:                              # pos + len in {size - 1, size, size + 1}
            pos = size + int(rng.integers(-1, 2)) - span
        elif u < 0.14:
            pos = int(rng.integers(0, size + 1))
        elif u < 0.7:
            pos = min(max(0, size - span), max(0, hot[k][int(rng.integers(0, 3))] + int(rng.integers(-300, 300))))
        else:
            pos = int(rng.integers(0, max(1, size - span + 1)))
        strand = STRANDS[int(rng.integers(0, 4))]
        c = conv if rng.random() < 0.9 else float(rng.choice([0.0, 0.5]))
        seq = read_at(rng, up[k], pos, L, strand, c, snps[k])
        u = rng.random()
        if u < 0.35:
            ins = 0
        elif u < 0.55:
            ins = int(rng.integers(1, max(2, span)))                      # |insert| < len
        else:
            ins = int(rng.integers(span, span + 500))
        ins = -ins if rng.random() < 0.5 else ins
        u = rng.random()
        if u < 0.15:
            pnext = 0
        elif u < 0.4:
            pnext = max(0, pos - int(rng.integers(1, 400))) + 1          # before the read
        elif u < 0.7:
            pnext = pos + int(rng.integers(0, span)) + 1                 # inside
        else:
            pnext = pos + span + int(rng.integers(0, 400)) + 1           # after
        flag = 0
        for bit, p in ((0x1, 0.5), (0x2, 0.6), (0x4, 0.03), (0x10, 0.5), (0x40, 0.3), (0x80, 0.4), (0x100, 0.15)):
            flag |= bit if rng.random() < p else 0
        out.append(dict(qname="r%d" % i, flag=flag, chrom=UNKNOWN if rng.random() < 0.03 else names[k], pos=pos, strand=strand,
                        insert=ins, pnext=pnext, seq=seq))
    if rm_dup:
        size = dict(zip(names, (len(s) for s in seqs)))

        def end_ok(r):
            if r["chrom"] not in size:
                return True
            fe = r["pos"] + len(r["seq"]) if r["strand"] in ("+-", "-+") else r["pos"]
            return fe < size[r["chrom"]]
        out = [r for r in out if end_ok(r)]
    return out


def flag_text(flag, letters):
    """FLAG as a number, or as letters; letters that are all digits ("1", "2", "12": 0x40 / 0x80 alone) read as a
    number, so those stay numeric"""
    text = "".join(FLAG_LETTERS[b] for b in range(11) if flag >> b & 1)
    return text if letters and not text.isdigit() and text else str(flag)


def sam_text(recs, names, seqs, letters=None):
    """SAM with @SQ lines; letters: per record, print FLAG as samtools view -X letters"""
    lines = ["@HD\tVN:1.0\n"] + ["@SQ\tSN:%s\tLN:%d\n" % (n, len(s)) for n, s in zip(names, seqs)]
    for i, r in enumerate(recs):
        seq = r["seq"]
        lines.append("\t".join([r["qname"], flag_text(r["flag"], letters is not None and letters[i]), r["chrom"], str(r["pos"] + 1), "255",
                                "%dM" % len(seq) if seq != "*" else "*", "=" if r["pnext"] else "*", str(r["pnext"]), str(r["insert"]),
                                seq, "I" * len(seq) if seq != "*" else "*", "NM:i:0", "ZS:Z:" + r["strand"]]) + "\n")
    return "".join(lines)


def bsp_text(recs):
    """BSP: 0x4 -> NM, 0x100 -> MA, else UM; the pair filter reads the insert column (0 = not paired)"""
    lines = []
    for r in recs:
        f = "NM" if r["flag"] & 0x4 else ("MA" if r["flag"] & 0x100 else "UM")
        lines.append("\t".join([r["qname"], r["seq"], "I" * len(r["seq"]), f, r["chrom"], str(r["pos"] + 1), r["strand"], str(r["insert"]),
                                "ACGT", "0:0"]) + "\n")
    return "".join(lines)


# ---- options --------------------------------------------------------------------------------------------------------
def draw_options(rng, names, seqs, sam):
    """one combination the command line accepts (M-bias and exclusion need SAM or BAM)"""
    o = dict(unique=rng.random() < 0.3, pair=rng.random() < 0.25, meth0=rng.random() < 0.4, combine_cpg=rng.random() < 0.3,
             rm_dup=rng.random() < 0.4, trim_fillin=int(rng.integers(0, 11)), min_depth=int(rng.integers(1, 5)))
    o["chroms"] = sorted(str(x) for x in rng.choice(names, int(rng.integers(1, len(names))), replace=False)) \
        if len(names) > 1 and rng.random() < 0.25 else None
    o["mbias"] = bool(sam and rng.random() < 0.35)
    o["ignore"] = tuple(int(x) for x in rng.integers(0, 7, 4)) if sam and rng.random() < 0.35 else None
    o["ct_snp"] = [None, "no-action", "correct", "skip"][int(rng.integers(0, 4))]
    u = rng.random()
    o["conv"] = None if u < 0.4 else (0 if u < 0.55 else int(rng.integers(1, 6)))
    u = rng.random()
    sel = {n: len(s) for n, s in zip(names, seqs) if not o["chroms"] or n in o["chroms"]}
    if u < 0.3:
        o["regions"] = None
    elif u < 0.65:
        o["regions"] = ("bed", random_regions(sel, int(rng.integers(1, 300)), seed=int(rng.integers(0, 1 << 30))))
    else:
        w = max(int(rng.integers(1, 5001)), sum(sel.values()) // 40_000)   # at most ~40k tiles: the oracle loops in Python
        o["regions"] = ("tiles", w)
    return o


def region_list(o, names, seqs):
    if o["regions"] is None:
        return None
    kind, v = o["regions"]
    if kind == "bed":
        return v
    return RO.tiles({n: len(s) for n, s in zip(names, seqs) if not o["chroms"] or n in o["chroms"]}, v)


def summary_line(valid, nc, nd):
    return "total %d valid mappings, %d covered cytosines, average coverage: %.2f fold." % (valid, nc, nd / nc if nc else 0.0)


def expected(names, seqs, files, o, sam_rules=None):
    """the composed oracle: counters, valid, M-bias, conversion bins, region sums and the texts"""
    res = CV.conversion(names, seqs, files, threshold=o["conv"] or 0, chroms=o["chroms"], unique=o["unique"], pair=o["pair"],
                        trim_fillin=o["trim_fillin"], combine_cpg=o["combine_cpg"], rm_dup=o["rm_dup"], ignore=o["ignore"] or (0, 0, 0, 0),
                        sam_rules=sam_rules)
    table, (nc, nd) = CV.table(res, meth0=o["meth0"], min_depth=o["min_depth"], ct_snp=o["ct_snp"])
    e = dict(res=res, table=table, summary=summary_line(res["valid"], nc, nd), stats=(nc, nd))
    if o["mbias"]:
        e["mbias_text"] = MB.mbias_text(res["mbias"])
    if o["conv"] is not None:
        e["conv_text"] = CV.report_text(res["bins"], o["conv"])
        e["conv_line"] = CV.stderr_line(res, o["conv"])
    regs = region_list(o, names, seqs)
    if regs is not None:
        e["regs"] = regs
        e["sums"] = RO.regions(res["counters"], res["ref"], regs, combine_cpg=o["combine_cpg"], min_depth=o["min_depth"], ct_snp=o["ct_snp"])
        e["region_text"] = RO.report_text(regs, e["sums"])
    return e


# ---- the device through the Python API --------------------------------------------------------------------------------
def new_meth(B, ix, o):
    mh = B.Meth(ix, B.meth_opts(unique=o["unique"], pair=o["pair"], meth0=o["meth0"], trim_fillin=o["trim_fillin"],
                                combine_cpg=o["combine_cpg"], min_depth=o["min_depth"], rm_dup=o["rm_dup"]))
    if o["conv"] is not None:
        mh.enable_conversion_filter(o["conv"])
    if o["mbias"]:
        mh.enable_mbias()
    if o["ignore"]:
        mh.set_ignore(*o["ignore"])
    if o["ct_snp"]:
        mh.enable_ct_snp(o["ct_snp"])
    return mh


def batch_cuts(rng, n):
    """1-6 batches at random cut points: empty and one-alignment batches included"""
    pts = [int(x) for x in rng.integers(0, n + 1, int(rng.integers(0, 4)))]
    if pts and rng.random() < 0.5:
        pts += [pts[0], min(n, pts[0] + 1)]                              # an empty and a one-alignment batch
    return [0] + sorted(pts) + [n]


def read_fd(fn):
    """run fn(fd) on a temporary file -> (its return value, the file's text)"""
    with tempfile.TemporaryFile() as f:
        r = fn(f.fileno())
        f.seek(0)
        return r, f.read().decode()


def first_diff(what, got, exp):
    if isinstance(exp, str):
        if got == exp:
            return None
        gl, el = got.splitlines(), exp.splitlines()
        for i, (x, y) in enumerate(zip(gl, el)):
            if x != y:
                return "%s line %d: got %r, expected %r" % (what, i, x[:200], y[:200])
        return "%s: %d lines, expected %d" % (what, len(gl), len(el))
    got, exp = np.asarray(got, dtype=np.int64), np.asarray(exp, dtype=np.int64)
    if got.shape == exp.shape and np.array_equal(got, exp):
        return None
    if got.shape != exp.shape:
        return "%s: shape %s, expected %s" % (what, got.shape, exp.shape)
    i = tuple(int(x) for x in np.argwhere(got != exp)[0])
    return "%s at %s: got %d, expected %d (%d differences)" % (what, i, got[i], exp[i], int((got != exp).sum()))


def compare_counters(mh, names, o, res):
    """valid count, counters and evidence of the selected sequences, M-bias bins and overflow, conversion bins and
    dropped count of mh against conversion_oracle's res -> first difference or None"""
    bad = first_diff("valid", mh.valid(), res["valid"])
    for k, name in enumerate(names):
        if bad or name not in res["counters"]:
            continue
        m, d = mh.counters(k)
        ex = res["counters"][name]
        bad = first_diff("meth of " + name, m, ex[0]) or first_diff("depth of " + name, d, ex[1])
        if not bad and o.get("ct_snp"):
            c, s = mh.ct_snp_counters(k)
            bad = first_diff("confirm of " + name, c, ex[2]) or first_diff("snp of " + name, s, ex[3])
    if not bad and o.get("mbias"):
        h, over = mh.mbias()
        bad = first_diff("M-bias", h, res["mbias"]) or first_diff("M-bias overflow", over, res["mbias_overflow"])
    if not bad and o.get("conv") is not None:
        h, dropped = mh.conversion()
        bad = first_diff("conversion bins", h, res["bins"]) or first_diff("dropped", dropped, res["dropped"])
    return bad


def device_check(B, names, seqs, files, o, e, rng=None, cuts=None):
    """pile up `files` through Meth.add (batches at `cuts`, or drawn), then every check of the module doc against e
    -> first difference or None"""
    sel = [not o["chroms"] or n in o["chroms"] for n in names]
    cols = api_arrays(files, names) or [[] for _ in range(8)]
    keep = [i for i, k in enumerate(cols[1]) if sel[k]]                  # -c: the command line drops the others at parse
    cols = [[c[i] for i in keep] for c in cols]
    n = len(cols[0])
    cuts = cuts or batch_cuts(rng, n)
    regs = e.get("regs")
    idx = {x: i for i, x in enumerate(names)}
    ci, st, en = ([idx[c] for c, _, _ in regs], [s for _, s, _ in regs], [x for _, _, x in regs]) if regs is not None else (None, None, None)
    ix = B.Index.packed(names, seqs)
    mh = new_meth(B, ix, o)
    try:
        for b, x in zip(cuts, cuts[1:]):
            mh.add(*[c[b:x] for c in cols[:7]], read2=cols[7][b:x])
            if regs is not None and not o["combine_cpg"] and x < n and rng is not None and rng.random() < 0.5:
                mh.regions(ci, st, en)                                   # a look in between changes nothing
        bad = compare_counters(mh, names, o, e["res"])
        if not bad and o["mbias"]:
            bad = first_diff("M-bias report", read_fd(mh.write_mbias)[1], e["mbias_text"])
        if not bad and o["conv"] is not None:
            bad = first_diff("conversion report", read_fd(mh.write_conversion)[1], e["conv_text"])
        if not bad and regs is not None:
            bad = first_diff("region sums", mh.regions(ci, st, en), e["sums"]) \
                or first_diff("region report", read_fd(lambda fd: mh.write_regions(fd, ci, st, en))[1], e["region_text"])
        if not bad:
            (w, stats), text = read_fd(lambda fd: mh.write(seqs, fd, chroms=sel))
            bad = first_diff("table", text, e["table"]) or first_diff("summary", summary_line(mh.valid(), *stats), e["summary"])
        return bad
    finally:
        mh.close(); ix.close()


def one_round(rng, k):
    """-> (description, first difference or None)"""
    import bsmap_b200 as B
    names, seqs = make_reference(rng)
    sam = rng.random() < 0.7
    o = draw_options(rng, names, seqs, sam)
    n = int(rng.choice([1, 60, 400, 2000]))
    recs = make_records(rng, names, seqs, n, rm_dup=o["rm_dup"])
    desc = dict(round=k, lengths=[len(s) for s in seqs], alignments=len(recs), fmt="sam" if sam else "bsp",
                opts={x: v for x, v in o.items() if v and x != "regions"},
                regions=None if o["regions"] is None else (o["regions"][0], o["regions"][1] if o["regions"][0] == "tiles" else len(o["regions"][1])))
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "a.sam" if sam else "a.bsp")
        with open(path, "w") as f:
            f.write(sam_text(recs, names, seqs) if sam else bsp_text(recs))
        e = expected(names, seqs, [path], o)
        bad = device_check(B, names, seqs, [path], o, e, rng=rng)
    return desc, bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=40)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    rng = np.random.default_rng(a.seed)
    fails = 0
    for k in range(a.rounds):
        desc, bad = one_round(rng, k)
        print(("FAIL " if bad else "ok   ") + str(desc) + ("  -> " + bad if bad else ""), flush=True)
        fails += bad is not None
    print(f"{a.rounds - fails}/{a.rounds} rounds identical")
    sys.exit(1 if fails else 0)


if __name__ == "__main__":
    main()
