"""The conversion filter: the numpy restatement (oracle/conversion_oracle.py) tied to mbias_oracle and the reference
script's own tables at threshold 0, checked against deleting the dropped records from the text, and hand-computed
known answers on a small genome."""
from __future__ import annotations

import gzip
import os
import sys

import numpy as np
import pytest

import cases as CS
from test_methratio_cpu import GOLD, MANIFEST, opts_kwargs
from test_mbias_cpu import NAMES, SEQS, mbias_kwargs, oracle_files, sam_line

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import conversion_oracle as CV  # noqa: E402
import mbias_oracle as MB  # noqa: E402
import methratio_oracle as MO  # noqa: E402

# the golden runs the M-bias tests take (their marginals are the table only at -m 1)
MBIAS_KEYS = sorted(k for k in MANIFEST if "-m" not in MANIFEST[k]["opts"] or MANIFEST[k]["opts"][MANIFEST[k]["opts"].index("-m") + 1] == "1")


@pytest.mark.parametrize("key", MBIAS_KEYS)
def test_threshold_0_reproduces_the_goldens(tmp_path, key):
    """threshold 0: the counters and M-bias are mbias_oracle's, the table is the reference script's, and the score
    histogram sums to the valid mappings"""
    ent = MANIFEST[key]
    case = CS.BY_NAME[ent["case"]]
    d = case.data()
    files = oracle_files(ent, case, str(tmp_path))
    kw = mbias_kwargs(ent["opts"])
    res = CV.conversion(d["gnames"], d["gseqs"], files, threshold=0, **kw)
    hist, overflow, mb, nmap = MB.mbias(d["gnames"], d["gseqs"], files, **kw)
    assert res["valid"] == nmap and res["dropped"] == 0 and int(res["bins"].sum()) == nmap
    assert np.array_equal(res["mbias"], hist) and res["mbias_overflow"] == overflow
    for c, (m, dp, _, _) in res["counters"].items():
        assert np.array_equal(m, mb[c][0]) and np.array_equal(dp, mb[c][1]), c
    tk = opts_kwargs(ent["opts"])
    txt, _ = CV.table(res, meth0=tk.get("meth0", False), min_depth=tk.get("min_depth", 1))
    assert txt == gzip.open(os.path.join(GOLD, key + ".txt.gz"), "rt").read()
    assert sum(len(s) for s in res["scores"]) == sum(len(MO.parse_alignments(f, set(res["ref"]), kw.get("unique", False), kw.get("pair", False))) for f in files)


def delete_records(files, res, threshold, td, unique=False, pair=False):
    """copies of the alignment files without the records scoring threshold or more"""
    out = []
    for k, (path, sc) in enumerate(zip(files, res["scores"])):
        sam = path[-4:].upper() == ".SAM"
        lines = open(path).read().splitlines(keepends=True)
        kept = CV.records(path, set(res["ref"]), unique, pair)
        assert len(kept) == len(sc)
        drop = {ln for (ln, _), s in zip(kept, sc) if s is not None and s >= threshold}
        p = os.path.join(td, "kept%d%s" % (k, ".sam" if sam else ".bsp"))
        open(p, "w").write("".join(x for i, x in enumerate(lines) if i not in drop))
        out.append(p)
    return out


NO_RMDUP_KEYS = [k for k in MBIAS_KEYS if "-r" not in MANIFEST[k]["opts"]]


@pytest.mark.parametrize("threshold", [1, 3])
def test_dropping_is_deleting(tmp_path, threshold):
    """without -r, the filtered counters and table are methratio_oracle's on the text without the dropped records;
    the valid mappings are the unfiltered ones"""
    total_dropped = 0
    for key in NO_RMDUP_KEYS:
        ent = MANIFEST[key]
        case = CS.BY_NAME[ent["case"]]
        d = case.data()
        td = tmp_path / key
        td.mkdir()
        files = oracle_files(ent, case, str(td))
        kw = opts_kwargs(ent["opts"])
        ckw = {k: v for k, v in kw.items() if k not in ("meth0", "min_depth")}
        res = CV.conversion(d["gnames"], d["gseqs"], files, threshold=threshold, **ckw)
        exp_txt, (nmap, nc, nd) = MO.methratio(d["gnames"], d["gseqs"], delete_records(files, res, threshold, str(td), kw.get("unique", False), kw.get("pair", False)), **kw)
        txt, (gc, gd) = CV.table(res, meth0=kw.get("meth0", False), min_depth=kw.get("min_depth", 1))
        assert txt == exp_txt and (gc, gd) == (nc, nd), key
        assert nmap == res["valid"] - res["dropped"] and res["dropped"] == int(res["bins"][threshold:].sum())
        total_dropped += res["dropped"]
    assert total_dropped > 0


# ---- known answers -------------------------------------------------------------------------------------------------
# chr1  0 G  1 C  2 A  3 C  4 G  5 T  6 T  7 C  8 A  9 G  10 C  11 T  12 C  13 N  14 A  15 C  16 C
#   '+' C: 1 CHH, 3 CpG, 7 CHG, 10 CHH, 12 CHH (next to N), 15 CHH, 16 CHH (last base)
#   '-' G: 0 CHH (position 0), 4 CpG, 9 CHG
# chr2  0 G  1 G  2 T  3 N  4 G  5 A  6 C  7 G        '+' C: 6 CpG      '-' G: 0 CHH, 1 CHH, 4 CHH (next to N), 7 CpG
REF10 = "GCACGTTCAG"
END7 = "CTCNACC"                                         # chr1[10:17], every C methylated: four CHH calls
PE = 0x1 | 0x2 | 0x40


def kat_file(tmp_path, lines, name="kat.sam"):
    p = tmp_path / name
    p.write_text("@HD\tVN:1.0\n" + "".join(lines))
    return str(p)


def run(tmp_path, lines, names=NAMES, seqs=SEQS, **kw):
    return CV.conversion(names, seqs, [kat_file(tmp_path, lines)], **kw)


# name -> (lines, kwargs, scores in file order)
KATS = {
    # '+': methylated C at 1 (CHH), 3 (CpG), 7 (CHG); the CpG does not count
    "plus": ([sam_line(0, "chr1", 1, REF10, "++")], {}, [2]),
    "plus_converted": ([sam_line(0, "chr1", 1, "GTATGTTTAG", "++")], {}, [0]),
    # '-': methylated G at 0 (CHH, off the sequence start), 4 (CpG), 9 (CHG)
    "minus": ([sam_line(16, "chr1", 1, REF10, "-+")], {}, [2]),
    "minus_partly": ([sam_line(16, "chr1", 1, "ACACGTTCAG", "-+")], {}, [1]),
    # CHH at the sequence end and next to N (read N makes no call)
    "chr1_end": ([sam_line(0, "chr1", 11, END7, "++")], {}, [4]),
    # '-' at chr2's start: G 0 (CHH, nothing before it), 1 unmethylated, 4 (CHH next to N)
    "chr2_start": ([sam_line(16, "chr2", 1, "GATNGA", "-+")], {}, [2]),
    # the CpG on both strands of chr2 6/7 does not count; the '-' G at 4 (CHH next to N) does
    "chr2_cpg": ([sam_line(0, "chr2", 5, "GACG", "++"), sam_line(16, "chr2", 5, "GACG", "--")], {"trim_fillin": 0}, [0, 1]),
    # -t: '+-' loses its last 2 printed bases, the CHH at 15 and 16 with them
    "fillin": ([sam_line(16, "chr1", 11, END7, "+-")], {"threshold": 3}, [2]),
    "fillin_off": ([sam_line(16, "chr1", 11, END7, "+-")], {"threshold": 3, "trim_fillin": 0}, [4]),
    # mate overlap: mate at 0-based 15 -> seq[:5]
    "overlap": ([sam_line(PE, "chr1", 11, END7, "++", tlen=7, pnext=16, rnext="=")], {"threshold": 3, "trim_fillin": 0}, [2]),
    "overlap_bsp_rules": ([sam_line(PE, "chr1", 11, END7, "++", tlen=7, pnext=16, rnext="=")], {"threshold": 3, "trim_fillin": 0, "sam_rules": False}, [4]),
    # exclusion: read 1's last two cycles hold the CHH at 15 and 16
    "ignore": ([sam_line(0, "chr1", 11, END7, "++")], {"threshold": 3, "ignore": (0, 2, 0, 0)}, [2]),
    "ignore_read2": ([sam_line(0x81, "chr1", 11, END7, "++")], {"threshold": 3, "ignore": (0, 2, 0, 0)}, [4]),
    # -r: the holder is dropped and keeps its key, so the converted duplicate still loses
    "rm_dup": ([sam_line(0, "chr1", 11, END7, "++"), sam_line(0, "chr1", 11, "TTTNATT", "++")], {"threshold": 3, "rm_dup": True}, [4, None]),
    # -g with a dropped '+' hit at the CpG 3/4 and a kept '-' one
    "combine_cpg": ([sam_line(0, "chr1", 1, "GCACGTTCAGCTC", "++"), sam_line(16, "chr1", 1, REF10, "-+")], {"threshold": 3, "combine_cpg": True}, [4, 2]),
    # threshold 1 drops any score; 255 only the last bin
    "threshold_1": ([sam_line(0, "chr1", 1, REF10, "++"), sam_line(16, "chr1", 1, "ACACGTTCAG", "-+"), sam_line(0, "chr1", 1, "GTATGTTTAG", "++")],
                    {"threshold": 1}, [2, 1, 0]),
    "threshold_255": ([sam_line(0, "chr1", 11, END7, "++")], {"threshold": 255}, [4]),
}


@pytest.mark.parametrize("name", sorted(KATS))
def test_known_scores(tmp_path, name):
    """the scores, the histogram and dropped; the kept counters are mbias_oracle's on the kept records alone"""
    lines, kw, exp = KATS[name]
    res = run(tmp_path, lines, **kw)
    assert res["scores"] == [exp]
    n = kw.get("threshold", 0)
    valid = [s for s in exp if s is not None]
    assert res["valid"] == len(valid) and int(res["bins"].sum()) == len(valid)
    assert res["dropped"] == sum(1 for s in valid if n and s >= n) == int(res["bins"][n:].sum() if n else 0)
    for s in valid:
        assert res["bins"][s] >= 1
    mkw = {k: v for k, v in kw.items() if k != "threshold"}
    if kw.get("rm_dup"):
        kept = []                                       # the holder's key is not released: its duplicate loses too
    else:
        kept = [x for x, s in zip(lines, exp) if not (n and s is not None and s >= n)]
    _, _, mb, _ = MB.mbias(NAMES, SEQS, [kat_file(tmp_path, kept, "kept.sam")], **mkw)
    for c, (m, dp, _, _) in res["counters"].items():
        assert np.array_equal(m, mb[c][0]) and np.array_equal(dp, mb[c][1]), c


def test_dropped_alignment_adds_nothing(tmp_path):
    """a dropped alignment leaves no call, no M-bias bin and no C/T SNP evidence, but stays a valid mapping"""
    res = run(tmp_path, [sam_line(0, "chr1", 1, REF10 + "CTC", "++")], threshold=3)
    assert res["scores"] == [[4]] and res["dropped"] == 1 and res["valid"] == 1
    assert all(int(a.sum()) == 0 for v in res["counters"].values() for a in v) and int(res["mbias"].sum()) == 0
    kept = run(tmp_path, [sam_line(0, "chr1", 1, REF10 + "CTC", "++")], threshold=5)
    assert kept["dropped"] == 0 and int(kept["counters"]["chr1"][2].sum()) == 3 and int(kept["mbias"].sum()) == 5


def test_lower_case_reference(tmp_path):
    """a lower-case reference reads as upper case"""
    lines = [sam_line(0, "chr1", 11, END7, "++"), sam_line(16, "chr2", 1, "GATNGA", "-+")]
    up = run(tmp_path, lines, threshold=3)
    low = run(tmp_path, lines, seqs=[s.lower() for s in SEQS], threshold=3)
    assert up["scores"] == low["scores"] == [[4, 2]] and np.array_equal(up["bins"], low["bins"])


def test_last_bin_holds_255_and_more(tmp_path):
    """300 methylated CHH calls land in bin 255, labelled 255+; threshold 255 drops them"""
    names, seqs = ["c"], [b"C" * 300 + b"A" * 20]
    lines = [sam_line(0, "c", 1, "C" * 300, "++"), sam_line(0, "c", 1, "C" * 255, "++"), sam_line(0, "c", 1, "C" * 254 + "T", "++")]
    res = CV.conversion(names, seqs, [kat_file(tmp_path, lines)], threshold=255)
    assert res["scores"] == [[300, 255, 254]]
    assert res["bins"][255] == 2 and res["bins"][254] == 1 and res["dropped"] == 2
    assert CV.report_text(res["bins"], 255) == CV.HEADER + "254\t1\t0\n255+\t2\t1\n"
    assert CV.stderr_line(res, 255) == "conversion filter: 2 of 3 valid mappings dropped (>= 255 methylated non-CpG calls)"


def test_report_text(tmp_path):
    res = run(tmp_path, KATS["threshold_1"][0], threshold=2)
    assert CV.report_text(res["bins"], 2) == CV.HEADER + "0\t1\t0\n1\t1\t0\n2\t1\t1\n"
    assert CV.report_text(res["bins"], 0) == CV.HEADER + "0\t1\t0\n1\t1\t0\n2\t1\t0\n"
    assert CV.stderr_line(res, 0) == "conversion filter: 0 of 3 valid mappings dropped (report only)"


def test_records(tmp_path):
    lines = [sam_line(0, "chr1", 1, REF10, "++").replace("r\t", "a\t", 1), sam_line(4, "chr1", 1, REF10, "++").replace("r\t", "u\t", 1),
             sam_line(0, "chr2", 1, "GGTN", "++").replace("r\t", "b\t", 1)]
    p = kat_file(tmp_path, lines)
    assert CV.records(p, set(NAMES)) == [(1, "a"), (3, "b")]
