#!/usr/bin/env python
"""Generates the expectations of the two full-size comparisons of tests/test_gpu.py with the reference binary:
  config2_raw_digest.json        BASELINE config 2 in full (2 Mb, 400 segments): size, line count and MD5 of the raw TSV
                                 (0.9 MB, too large to store), a seeded sample of its lines, and the stderr lines
  config5_1000_monomers_raw.tsv  config 5's 1,000 monomers against 3,700 bp of one of its arrays: the whole raw TSV
Usage:   python tests/golden/make_golden_full_runs.py <dp-compatible binary>
The binary is the unmodified reference (oracle/_ref/dp, built by oracle/Makefile) or one shown byte-identical to it on
these inputs.  The committed files were written by the oracle port (oracle/_build/oracle_dp).  On these inputs its output
is byte-identical to that of the project's dp at commit fa14fa1, which both tests, run against the reference binary
itself, had found byte-identical to the reference."""
import hashlib
import json
import os
import random
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import cases  # noqa: E402
import sd_oracle  # noqa: E402

CONFIG2 = os.path.join(HERE, "config2_raw_digest.json")
CONFIG5 = os.path.join(HERE, "config5_1000_monomers_raw.tsv")
SAMPLE_LINES = 400


def main():
    binary = os.path.abspath(sys.argv[1])
    with tempfile.TemporaryDirectory() as td:
        rp, mp = cases.write_config2(td)
        p = subprocess.run([binary, rp, mp, str(os.cpu_count() or 1), "5000", "500"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                           check=True)
    lines = p.stdout.decode().splitlines(True)
    sample = sorted(random.Random(2).sample(range(len(lines)), SAMPLE_LINES))
    with open(CONFIG2, "w") as f:
        json.dump({"generator": "tests/golden/make_golden_full_runs.py", "argv_tail": ["<threads>", "5000", "500"],
                   "bytes": len(p.stdout), "lines": len(lines), "md5": hashlib.md5(p.stdout).hexdigest(),
                   "stderr": [ln for ln in p.stderr.decode().splitlines() if not ln.startswith("[sd_b200]")],
                   "sample": [[i, lines[i]] for i in sample]}, f, indent=0)
    rn, reads, mn, mons = cases.config5_sample()
    out = sd_oracle.decompose_reads(rn, reads, mn, mons, part_size=1700, overlap=300, binary=binary, threads=2)
    with open(CONFIG5, "w", newline="") as f:
        f.write(out)
    print("config 2: %d lines, md5 %s; config 5 sample: %d lines" % (len(lines), hashlib.md5(p.stdout).hexdigest(), out.count("\n")))


if __name__ == "__main__":
    main()
