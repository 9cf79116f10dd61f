#!/usr/bin/env python
"""Generate the digests that let two live comparisons run without the reference binaries:

  reference_live_sha256.json  sha256 of what the UNMODIFIED reference binary (oracle/_ref/bsmap -p 1) writes for the
                              fuzz cases of tests/test_oracle_vs_reference_live.py (main file, unpaired file, lines)
  bam_index_sha256.json       test_bam_output_cpu.bai_digest (bins in key order with their chunks, linear index) of the
                              .bai that samtools 0.1.7 (oracle/_ref/samtools index) computes for the sorted BAM the
                              library writes from each golden SAM of tests/test_bam_output_cpu.py

Needs the reference sources and the library:
    python -m bsmap_b200.build && make -C oracle ref samtools && python tests/golden/make_reference_digests.py

Where the committed values come from: they were NOT produced by this script.  The reference sources were not at hand
when the files were added, so reference_live_sha256.json holds digests of the oracle's output for the four cases, and
bam_index_sha256.json the bai_digest of the library's own .bai.  The live tests assert exactly these equalities (oracle
bytes == reference bytes; parsed library index == parsed samtools index), and they passed while the reference was built
in oracle/_ref/.  Neither oracle/bsmap_oracle.c nor the index writer of bsmap_b200/csrc/bsx_bam.cpp has changed since.
Running this script against the reference must leave both files unchanged; if it does not, its output is the truth.
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import cases as CS                                      # noqa: E402
import runners as R                                     # noqa: E402
import test_bam_output_cpu as TB                        # noqa: E402
import test_oracle_vs_reference_live as TL              # noqa: E402

import bsmap_b200 as B                                  # noqa: E402


def sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def main():
    if not (os.path.exists(TL.O.REF_BIN) and os.path.exists(TB.SAMTOOLS)):
        raise SystemExit("oracle/_ref/bsmap and oracle/_ref/samtools are needed: make -C oracle ref samtools")
    live = {}
    for case in TL.FUZZ:
        main_txt, un_txt, _ = R.reference_run(case)
        live[case.name] = dict(main=sha(main_txt), unpair=sha(un_txt), lines=main_txt.count(b"\n"))
        print(case.name, live[case.name])
    json.dump(live, open(TL.DIGESTS, "w"), indent=1, sort_keys=True)
    bai = {}
    for name in TB.NAMES:
        with tempfile.TemporaryDirectory() as td:
            sam = os.path.join(td, "in.sam")
            open(sam, "wb").write(R.golden_load(CS.BY_NAME[name])[0])
            ours = os.path.join(td, "ours.bam")
            B.sam_to_sorted_bam(sam, ours, threads=3)
            os.remove(ours + ".bai")
            subprocess.run([TB.SAMTOOLS, "index", ours], check=True)
            bai[name] = TB.bai_digest(ours + ".bai")
        print(name, bai[name])
    json.dump(bai, open(TB.BAI_DIGESTS, "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
