#!/usr/bin/env python
"""Cost of streaming the segment symbols through the sweep kernels, and what one-segment-per-read decomposition costs.

    python tools/long_segment_probe.py [--out profiles/r03_long_segments.txt] [--reps 5]

(a) Staged vs streamed symbols at the same geometry (SD_GEOM pins it, SD_STREAM_SYMBOLS=1 selects the streamed variant),
    the two handles alternating within this one process: config 2 (400 x 5,500 columns, classic (19,10)), a 50-segment
    cluster shape (12,16) and the saturated classic shape C=24, T=8, NS=4 (4,000 segments).  Kernel times are CUDA-event
    times through sd_stage / sd_run_staged; "cycles/column" is the sweep time in SM cycles at the clock read below over
    the columns of one segment (5,500), i.e. the per-column latency when every CTA of the launch runs at once.
(b) One 400 kb and one 990 kb DXZ1 array as single segments against the 12 DXZ1 monomers: classic vs cluster sweep
    (both streamed: they do not fit shared memory), with the traceback time.
(c) A file of long reads decomposed with -b 5000 and with one segment per read (sd_run_files): wall time and the number
    of raw-TSV records that differ.
Needs a CUDA device; the card's name, clocks and power limit are read at the start."""
import argparse
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np

from stringdecomposer_b200 import _lib, synth, Decomposer
from stringdecomposer_b200.hostpipe import segment_reads

LOG = []


def say(s=""):
    print(s, flush=True)
    LOG.append(s)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem",
                        "--format=csv,noheader", "-i", "0"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"
    say("card: %s   (name, power limit, SM clock, max SM clock, memory clock)" % line)
    try:
        return float(line.split(",")[3].split()[0]) * 1e6
    except (IndexError, ValueError):
        return 1.965e9


def pack(segs):
    blob = "".join(segs).encode()
    off = np.zeros(len(segs) + 1, dtype=np.int64)
    np.cumsum([len(s) for s in segs], out=off[1:])
    return blob, off


def handle(mons, data, env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        d = Decomposer(mons, devices=[0])
        d.stage(data)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    d.run_staged()
    return d


def timed(d):
    d.reset_stats()
    d.run_staged()
    st = d.stats()
    return st["sweep_ms"], st["traceback_ms"]


def compare(title, mons, segs, variants, reps, clk, cols):
    """variants: [(label, env)]; all handles alternate, min and median of `reps` rounds"""
    data = pack(segs)
    hs = [(lab, handle(mons, data, env)) for lab, env in variants]
    times = {lab: [] for lab, _ in hs}
    tbs = {lab: [] for lab, _ in hs}
    for _ in range(reps):
        for lab, d in hs:
            sw, tb = timed(d)
            times[lab].append(sw)
            tbs[lab].append(tb)
    ref = hs[0][1].fetch_staged()
    say(title)
    base = None
    for lab, d in hs:
        st = d.stats()
        r, o = d.fetch_staged()
        same = bool(len(r) == len(ref[0]) and (r == ref[0]).all() and (o == ref[1]).all())
        med = float(np.median(times[lab]))
        base = base or med
        say("  %-28s lat=%d C=%d T=%d NS=%d NT=%d NG=%d stream=%d  sweep min %.3f med %.3f ms (%+.1f %%)  %.0f cycles/column"
            "  traceback med %.3f ms  same records=%s" % (lab, st["lat"], st["C"], st["T"], st["NS"], st["NT"], st["NG"], st["stream"],
                                                            min(times[lab]), med, 100 * (med / base - 1), med * 1e-3 * clk / cols,
                                                            float(np.median(tbs[lab])), same))
        d.close()


def part_a(reps, clk):
    rn, reads, mn, mons = synth.config2()
    segs, _ = segment_reads(reads, 5000, 500)
    for title, segs_, env in (
            ("(a) config 2, 400 x 5,500 columns, classic (19,10)", segs, {"SD_LAT": "0", "SD_GEOM": "19,10,1"}),
            ("(a) 50 segments of config 2, cluster (12,16)", segs[:50], {"SD_LAT": "1", "SD_GEOM": "12,16,1"}),
    ):
        compare(title, mons, segs_, [("staged", env), ("streamed", dict(env, SD_STREAM_SYMBOLS="1"))], reps, clk, 5500)
    rn, reads, mn, mons = synth.config2(length=20_000_000, seed=12)
    segs, _ = segment_reads(reads, 5000, 500)
    env = {"SD_LAT": "0", "SD_GEOM": "24,8,4"}
    compare("(a) saturated classic C=24 T=8 NS=4, %d x 5,500 columns" % len(segs), mons, segs,
            [("staged", env), ("streamed", dict(env, SD_STREAM_SYMBOLS="1"))], reps, clk, 5500)


def part_b(reps, clk):
    names, mons = synth.load_dxz1()
    for n in (400_000, 990_000):
        seg = synth.hor_array(mons, n, 0.02, seed=7)
        compare("(b) one %d bp DXZ1 array as one segment, 12 monomers" % n, mons, [seg],
                [("cluster (planner's choice)", {}), ("classic", {"SD_LAT": "0"})], reps, clk, n)


def part_c(tmp):
    rn, reads, mn, mons = synth.sample_reads(24, 150_000, 0.02, 0.04, 0.04, seed=31, array_len=2_000_000)
    rp, mp = os.path.join(tmp, "reads.fa"), os.path.join(tmp, "mons.fa")
    synth.write_fasta(rp, rn, reads, width=80)
    synth.write_fasta(mp, mn, mons)
    longest = max(len(r) for r in reads)
    outs = {}
    for part in (5000, 5000, longest, longest, 5000, longest):          # first call of each warms up; alternate
        with open(os.path.join(tmp, "out"), "w+b") as fo, open(os.devnull, "w") as fe:
            t0 = time.perf_counter()
            st = _lib.run_files(rp, mp, 1, part, 500, (-1, -1, -1, 1), -1, out_fd=fo.fileno(), err_fd=fe.fileno())
            dt = time.perf_counter() - t0
            fo.seek(0)
            outs.setdefault(part, []).append((dt, st, fo.read().decode().splitlines()))
    say("(c) %d reads of %d bp (ONT-like errors) against the 12 DXZ1 monomers, sd_run_files" % (len(reads), len(reads[0])))
    for part in (5000, longest):
        walls = [o[0] for o in outs[part][1:]]
        say("  -b %-7d wall %.3f s (runs after the first: %s)  status %d  %d records" % (
            part, min(walls), ", ".join("%.3f" % w for w in walls), outs[part][-1][1], len(outs[part][-1][2])))
    a, b = set(outs[5000][-1][2]), set(outs[longest][-1][2])
    say("  records only with -b 5000: %d   only with one segment per read: %d   common: %d" % (len(a - b), len(b - a), len(a & b)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles", "r03_long_segments.txt"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parts", default="abc")
    args = ap.parse_args()
    if _lib.device_count() < 1:
        sys.exit("long_segment_probe: needs a CUDA device")
    clk = card()
    with tempfile.TemporaryDirectory() as tmp:
        if "a" in args.parts:
            part_a(args.reps, clk)
        if "b" in args.parts:
            part_b(args.reps, clk)
        if "c" in args.parts:
            part_c(tmp)
    card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(LOG) + "\n")


if __name__ == "__main__":
    main()
