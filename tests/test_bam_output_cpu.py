"""`-o out.bam`: bsx_sam_to_sorted_bam against the vendored samtools 0.1.7 (what the reference's sam2bam.sh runs):
`samtools view -bS | samtools sort | samtools index` on the reference's own SAM output.  The BAM must decompress to the
same bytes; the .bai must hold what `samtools index` computes for our file (bins, chunks, linear index).  Without
oracle/_ref/samtools (make -C oracle samtools) both are checked against committed digests of samtools' output
(bam_output_sha256.json, bam_index_sha256.json; tests/golden/make_reference_digests.py)."""
from __future__ import annotations

import gzip
import hashlib
import json
import os
import struct
import subprocess

import pytest

import cases as CS
import runners as R

import bsmap_b200 as B
from bsmap_b200 import lib as BL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAMTOOLS = os.path.join(ROOT, "oracle", "_ref", "samtools")
DIGESTS = os.path.join(ROOT, "tests", "golden", "bam_output_sha256.json")
BAI_DIGESTS = os.path.join(ROOT, "tests", "golden", "bam_index_sha256.json")
NAMES = ["se_cfg2_r0_uR", "pe_sam", "pe_sam_v5_R", "pe_readthrough", "rrbs_pe", "rrbs_se_A", "se_n1", "se_cfg1", "se_mixed_A", "se_cfg5"]
pytestmark = pytest.mark.skipif(not os.path.exists(BL.LIB_PATH), reason="library not built")


def parse_bai(path):
    d = open(path, "rb").read()
    assert d[:4] == b"BAI\1"
    o = 4
    n, = struct.unpack_from("<i", d, o); o += 4
    out = []
    for _ in range(n):
        nb, = struct.unpack_from("<i", d, o); o += 4
        bins = {}
        for _ in range(nb):
            b, nc = struct.unpack_from("<Ii", d, o); o += 8
            bins[b] = [struct.unpack_from("<QQ", d, o + 16 * i) for i in range(nc)]; o += 16 * nc
        nl, = struct.unpack_from("<i", d, o); o += 4
        out.append((bins, list(struct.unpack_from("<%dQ" % nl, d, o)))); o += 8 * nl
    assert o == len(d)
    return out


def bai_digest(path):
    """sha256 of the index parse_bai reads (per reference: bins in key order with their chunks, then the linear index).
    samtools writes the bins of a reference in hash-table order and this library in key order, so two .bai files that
    hold the same index need not be the same bytes."""
    canon = [[sorted((b, [list(c) for c in ch]) for b, ch in bins.items()), list(lin)] for bins, lin in parse_bai(path)]
    return hashlib.sha256(json.dumps(canon).encode()).hexdigest()


@pytest.mark.parametrize("name", NAMES)
def test_sorted_bam_equals_samtools(tmp_path, name):
    case = CS.BY_NAME[name]
    sam = str(tmp_path / "in.sam")
    open(sam, "wb").write(R.golden_load(case)[0])
    ours = str(tmp_path / "ours.bam")
    B.sam_to_sorted_bam(sam, ours, threads=3)
    raw = gzip.open(ours, "rb").read()
    assert raw[:4] == b"BAM\1" and open(ours, "rb").read()[-28:] == bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
    assert hashlib.sha256(raw).hexdigest() == json.load(open(DIGESTS))[name], "decompressed BAM differs from samtools' (committed digest)"
    if not os.path.exists(SAMTOOLS):
        assert bai_digest(ours + ".bai") == json.load(open(BAI_DIGESTS))[name], \
            "index differs from what `samtools index` computes for this file (committed digest of its bins, chunks and linear index)"
        return
    ref = str(tmp_path / "ref")
    subprocess.run(f"{SAMTOOLS} view -bS {sam} > {tmp_path}/tmp.bam 2>/dev/null && {SAMTOOLS} sort {tmp_path}/tmp.bam {ref}", shell=True, check=True)
    assert gzip.open(ref + ".bam", "rb").read() == raw
    mine = parse_bai(ours + ".bai")
    os.remove(ours + ".bai")
    subprocess.run([SAMTOOLS, "index", ours], check=True)
    assert parse_bai(ours + ".bai") == mine


@pytest.mark.parametrize("name", ["pe_sam", "se_cfg5", "rrbs_se_A"])
def test_bounded_memory_path_writes_the_same_files(tmp_path, monkeypatch, name):
    """text taken in 20 KB chunks (sorted runs on disk + merge) and BGZF windows of two blocks (the index trails the
    writer): same .bam and .bai bytes as the one-chunk, one-window conversion"""
    case = CS.BY_NAME[name]
    sam = str(tmp_path / "in.sam")
    open(sam, "wb").write(R.golden_load(case)[0])
    assert os.path.getsize(sam) > 200_000
    B.sam_to_sorted_bam(sam, str(tmp_path / "a.bam"), threads=3)
    monkeypatch.setenv("BSX_BAM_CHUNK_MB", "0.02"); monkeypatch.setenv("BSX_BAM_WINDOW_BLOCKS", "2")
    B.sam_to_sorted_bam(sam, str(tmp_path / "b.bam"), threads=3)
    assert open(tmp_path / "a.bam", "rb").read() == open(tmp_path / "b.bam", "rb").read()
    assert open(tmp_path / "a.bam.bai", "rb").read() == open(tmp_path / "b.bam.bai", "rb").read()
    assert not [f for f in os.listdir(tmp_path) if f.endswith(".tmp")], "run files must be removed"


def test_bam_writer_errors(tmp_path):
    with pytest.raises(B.BsxError, match="cannot open"):
        B.sam_to_sorted_bam(str(tmp_path / "missing.sam"), str(tmp_path / "x.bam"))
    empty = tmp_path / "empty.sam"
    empty.write_bytes(b"@HD\tVN:1.0\n@SQ\tSN:chr1\tLN:100\n")
    B.sam_to_sorted_bam(str(empty), str(tmp_path / "e.bam"))
    raw = gzip.open(tmp_path / "e.bam", "rb").read()
    assert raw.startswith(b"BAM\1") and raw.endswith(b"chr1\0" + struct.pack("<i", 100))
    assert parse_bai(str(tmp_path / "e.bam.bai")) == [({}, [])]
