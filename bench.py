#!/usr/bin/env python
"""bench.py -- DP GCUPS of the string-decomposition sweep on the BASELINE.json config-2 workload.

One "step" = one pass of the hot path (forward sweep + traceback kernels) over one batch: the synthetic 2 Mb
cenX-like DXZ1 HOR array cut into 400 segments (part 5000, overlap 500) against the 12 DXZ1 monomers and their
reverse complements.  `value` is measured with the segments already resident in HBM (CUDA events on the library's
stream); `e2e` goes through the public C ABI (sd_decompose) with host buffers, H2D and D2H inside the timed region.
N > 1 (north_star: strong scaling of ONE 2 Mb array): rank 0 of the torchrun launch drives all N GPUs through the
library's own partitioning (Engine::split: contiguous segment ranges, one host thread + stream per GPU, records
gathered on the host; no collective on the data path -- segments are independent, SURVEY 8e); the other ranks only
join the barriers.  The round-1 replica measurement (one array per GPU, one process per GPU) is kept under "replicas".

--impl reference times the unmodified reference binary (oracle/_ref/dp, built from /root/reference by
oracle/Makefile) on the same workload with -t <host cores>.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PART, OVERLAP = 5000, 500
SCORING = (-1, -1, -1, 1)
WORKLOAD = "config2: synthetic 2 Mb cenX-like DXZ1 HOR array, 12 monomers (+RC), part 5000 overlap 500"
METRIC = "dp_gcups"
UNIT = "GCUPS"
# ALU-pipe instructions the sweep needs per DP cell in the packed s16x2 kernel (DESIGN.md section 3): per register
# (2 cells) 3 VIADDMNMX + 0.5 VIMNMX3 + 1 LOP3 = 4.5 -> 2.25 per cell (the 2 IMAD per register run on the FMA pipe)
OPS_PER_CELL = {1: 2.25, 0: 4.5}
SURVEY_OPS_PER_CELL = {1: 5.5, 0: 11.0}      # SURVEY.md section 8d planning figures (s16x2 / s32)


def dist_setup(n_gpus):
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if ws > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl" if torch.cuda.is_available() else "gloo")
        global CPU_GROUP
        CPU_GROUP = dist.new_group(backend="gloo")
    return ws, rank, local


CPU_GROUP = None


def barrier_sync(ws):
    """Barrier + device synchronisation on both sides.  The ranks meet on the CPU (gloo) first: a rank that waits for
    rank 0 inside an NCCL barrier keeps a spinning kernel on its GPU, and in the strong-scaling leg rank 0 is running the
    sweep on that very GPU -- the NCCL barrier proper is entered only once everybody has arrived."""
    import torch
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    if ws > 1:
        import torch.distributed as dist
        dist.barrier(group=CPU_GROUP)
        dist.barrier()
        if torch.cuda.is_available():
            torch.cuda.synchronize()


def max_over_ranks(x, ws):
    if ws == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda" if torch.cuda.is_available() else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x, ws):
    if ws == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda" if torch.cuda.is_available() else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region: NVML from a thread (10 ms period, no extra
    process), falling back to the nvidia-smi recipe of B200_PROFILING.md."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.proc, self.lines, self.samples, self.stop_flag = gpu, None, [], [], False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu)
        except Exception:
            self.nvml = None

    def start(self):
        if self.nvml:
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
                mx = n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)
                try:
                    r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((sm, mx, r))
            except Exception:
                pass
            time.sleep(0.01)

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln)

    def stop(self):
        if self.nvml:
            self.stop_flag = True
            self.th.join(timeout=1)
            n = self.nvml
            names = {"hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8), "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            sm = [s[0] for s in self.samples]
            reasons = sorted({k for s in self.samples for k, bit in names.items() if s[2] & bit})
            busy = [x for x in sm if x > 0.5 * max(sm)] if sm else []
            return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": float(max(s[1] for s in self.samples)) if self.samples else None,
                    "reasons": reasons, "samples": len(sm), "source": "nvml, 10 ms period during the timed region"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [x for x in sm if x > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100"}


def workload(rank):
    from stringdecomposer_b200 import synth
    from stringdecomposer_b200.hostpipe import segment_reads
    rnames, reads, mnames, mons = synth.config2(seed=2 + rank)
    segs, where = segment_reads(reads, PART, OVERLAP)
    return rnames, reads, mnames, mons, segs


def cells_of(segs, mons):
    return sum(len(s) for s in segs) * 2 * sum(len(m) for m in mons)


def headline_cells(reads, mons):
    # north_star: "read bp x total monomer bp" (fwd + RC rows)
    return sum(len(r) for r in reads) * 2 * sum(len(m) for m in mons)


def run_reference_arm(args, ws, rank):
    """The reference's own CPU implementation (oracle/_ref/dp) on the same workload, all host cores."""
    if rank != 0:
        return
    from stringdecomposer_b200 import synth
    ref = os.path.join(ROOT, "oracle", "_ref", "dp")
    kind = "reference"
    if not os.path.exists(ref):
        ref = os.path.join(ROOT, "oracle", "_build", "oracle_dp")
        kind = "port"
    if not os.path.exists(ref):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "port"], check=False)
    cores = os.cpu_count() or 1
    rnames, reads, mnames, mons = synth.config2(seed=2)
    with tempfile.TemporaryDirectory() as td:
        rp, mp = os.path.join(td, "reads.fa"), os.path.join(td, "monomers.fa")
        synth.write_fasta(rp, rnames, reads)
        synth.write_fasta(mp, mnames, mons)
        cmd = [ref, rp, mp, str(cores), str(PART), str(OVERLAP)]
        times = []
        for it in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            with open(os.path.join(td, "out.tsv"), "wb") as out:
                subprocess.run(cmd, stdout=out, stderr=subprocess.DEVNULL, check=True)
            dt = time.perf_counter() - t0
            if it >= args.warmup:
                times.append(dt)
    T = sum(times)
    cells = headline_cells(reads, mons) * len(times)
    val = cells / T / 1e9
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * T / len(times), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "segments": 400, "scoring": "-1,-1,-1,1"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": "full config-2 contig (2,000,000 bp) per step, dp -t %d, wall time of the process" % cores},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "decomposed_mbp_per_s": sum(len(r) for r in reads) * len(times) / T / 1e6, "gpu_launches": 0}
    emit(line)


def timed_resident(dec, packed, args, ws, flushes, sampler_gpu):
    """`value` leg: segments resident in HBM, sweep + traceback kernels, CUDA events on the library's streams."""
    import torch
    dec.stage(packed)
    for _ in range(args.warmup):
        dec.run_staged()
    sampler = ClockSampler(sampler_gpu)
    barrier_sync(ws)
    sampler.start()
    dec.reset_stats()
    dev_ms = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for f in flushes:
            f.zero_()                         # 256 MiB > 126 MB L2, on every device that takes part
        for d in range(len(flushes)):
            torch.cuda.synchronize(flushes[d].device)
        dev_ms += dec.run_staged()            # max over devices of (sweep + traceback), CUDA events per device
    barrier_sync(ws)
    wall = time.perf_counter() - t0
    return dev_ms, wall, sampler.stop(), dec.stats()


def timed_e2e(dec, packed, args, ws):
    """`e2e` leg: host buffers through the C-ABI call sd_decompose, H2D + kernels + D2H inside the timed region.  The K
    calls are issued back to back from native code (libsd_bench.so), as a C/C++ host application would; the same loop
    from Python (ctypes + numpy copies of the result per call) is reported next to it."""
    from stringdecomposer_b200._lib import HostBuffer
    pinned = HostBuffer.pack(packed)                    # the step's inputs in page-locked host memory (sd_host_alloc)
    for _ in range(args.warmup):
        dec.decompose(pinned)
    barrier_sync(ws)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r2, o2 = dec.decompose(pinned)
    py_s = time.perf_counter() - t0
    dec.reset_stats()
    sec, nrec = dec.decompose_timed(pinned, 0, args.steps)
    barrier_sync(ws)
    assert nrec == len(r2)
    return sec, dec.stats(), r2, o2, py_s


def pack_segments(segs):
    blob = "".join(segs).encode()
    off = np.zeros(len(segs) + 1, dtype=np.int64)
    np.cumsum([len(s) for s in segs], out=off[1:])
    return blob, off


def dump_outputs(out_dir, recs, roff):
    """What the last timed step returned to its caller (sd_fetch_staged): every record field and the per-segment record
    offsets, as float64 (exact for these int32 / int64 values), so that two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name in recs.dtype.names:
        np.save(os.path.join(out_dir, "records_%s.npy" % name), recs[name].astype(np.float64))
    np.save(os.path.join(out_dir, "record_offsets.npy"), roff.astype(np.float64))


_OUT = None


def emit(line):
    out = _OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the rescoring / process / replica extras")
    ap.add_argument("--geom", default=None, help="override launch geometry C,T,NS (exploration)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the records of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the outputs of --impl ours")
    # stdout carries the one JSON line and nothing else: native libraries that write to file descriptor 1 (NCCL prints
    # its version banner there when NCCL_DEBUG is set) are sent to stderr, the line goes to the saved descriptor
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.geom:
        os.environ["SD_GEOM"] = args.geom
    if args.impl == "reference":
        # CPU only: rank 0 of a torchrun launch runs it, the other ranks exit at once (no process group, no GPU touched)
        run_reference_arm(args, int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")))
        return
    ws, rank, local = dist_setup(args.gpus)

    import torch
    from stringdecomposer_b200 import Decomposer, int_peak
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)

    # ---- strong scaling (north_star): ONE 2 Mb array, its 400 segments split over the N GPUs of the box by the
    # library (Engine::split, one host thread + stream per GPU, records gathered on the host in segment order --
    # the AlignReadsSet gather of main.cpp:84-121).  Rank 0 drives all N devices; the other ranks of the torchrun
    # launch only take part in the barriers.
    rnames, reads, mnames, mons, segs = workload(0)
    packed = pack_segments(segs)
    cells_hl = float(headline_cells(reads, mons))
    cells_act = float(cells_of(segs, mons))
    line = None
    if rank == 0:
        dec = Decomposer(mons, *SCORING, devices=list(range(ws)))
        flushes = [torch.empty(256 << 20, dtype=torch.uint8, device="cuda:%d" % d) for d in range(ws)]
        dev_ms, wall, clocks, st = timed_resident(dec, packed, args, ws, flushes, local)
        recs, roff = dec.fetch_staged()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, recs, roff)
        e2e_s, st2, r2, o2, e2e_py_s = timed_e2e(dec, packed, args, ws)
        same = bool(len(r2) == len(recs) and (r2 == recs).all() and (o2 == roff).all())
        value = cells_hl * args.steps / (dev_ms * 1e-3) / 1e9
        sweep_ms = st["sweep_ms"] / args.steps
        tb_ms = st["traceback_ms"] / args.steps
        # ---- roofline of the dominant kernel (sweep): integer issue rate, aggregated over the N devices ----
        alu, both, mhz = int_peak(local)
        opc = OPS_PER_CELL[1 if st["packed"] else 0]
        ach = cells_act / (sweep_ms * 1e-3) * opc / 1e12
        peak = ws * alu / 1e12
        in_bytes = float(sum(len(s) for s in segs))
        roof = {"bound": "int_alu", "achieved": ach, "peak": peak, "unit": "Tlane-op/s", "frac": ach / peak,
                "traffic": float(st["sweep_store_bytes"]) + in_bytes,
                "traffic_source": "computed at run time from the launch layout (sd_get_stats: 2-bit backpointer words incl. slot "
                                  "padding + 8 B per column + 1 B per column read); the ncu dram__bytes of the same launch are in profiles/",
                "traffic_algorithmic": 0.25 * cells_act + 9.0 * in_bytes,
                "peak_source": "measured in this run by sd_int_peak: independent VIADDMNMX.S16x2 streams on all SMs "
                               "(the integer ALU pipe, 64 lanes/clk/SM), times %d GPUs; with the FMA pipe (IMAD) in parallel: %.2f per GPU" % (ws, both / 1e12),
                "ops_per_cell": opc, "kernel": "sweep_lat_kernel" if st["lat"] else "sweep_kernel", "kernel_ms": sweep_ms, "traceback_ms": tb_ms,
                "frac_with_survey_ops_per_cell": cells_act / (sweep_ms * 1e-3) * SURVEY_OPS_PER_CELL[1 if st["packed"] else 0] / (ws * alu),
                "hbm": {"achieved_gbs": (float(st["sweep_store_bytes"]) + in_bytes) / (sweep_ms * 1e-3) / 1e9,
                        "peak_gbs": _hbm_peak() * ws, "note": "2-bit backpointers, 0.25 B/cell; not the limiter"}}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ws, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "s16x2" if st["packed"] else "s32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "segments": len(segs), "segments_per_gpu": st["dev_segments"], "scoring": "-1,-1,-1,1",
                           "partition": "one array; contiguous column-balanced segment ranges, one per GPU, driven by one host process "
                                        "(Engine::split); no collective on the data path",
                           "l2": "256 MiB memset on every GPU between timed steps",
                           "geometry": {k: st[k] for k in ("C", "T", "NS", "NT", "NG", "lat", "scanw")}},
                "cells_actual_gcups": cells_act * args.steps / (dev_ms * 1e-3) / 1e9,
                "decomposed_mbp_per_s": sum_len(reads) * args.steps / (dev_ms * 1e-3) / 1e6,
                "wall_ms_per_step": 1e3 * wall / args.steps,
                "e2e": {"value": cells_hl * args.steps / e2e_s / 1e9, "unit": UNIT, "h2d_bytes_per_step": st2["h2d_bytes"] // args.steps,
                        "d2h_bytes_per_step": st2["d2h_bytes"] // args.steps, "ms_per_step": 1e3 * e2e_s / args.steps,
                        "python_caller_ms_per_step": 1e3 * e2e_py_s / args.steps,
                        "caller": "sd_decompose called K times back to back from native code (libsd_bench.so) on segment text in "
                                  "page-locked host memory (sd_host_alloc); python_caller_ms_per_step is the same loop through ctypes",
                        "matches_resident_run": same},
                "gpu_launches": int(st["launches"]), "clocks": clocks, "roofline": roof}
        if ws == 1 and not args.no_extras:
            line["rescoring"] = rescoring(segs, mons, recs, roff, local, alu)
            line["process"] = process_boundary(rnames, reads, mnames, mons)
            line["ed_thr"] = ed_thr_leg(dec, packed, cells_hl, args)
            line["config3_waves"] = config3_waves(local)
        if not args.no_cpu_baseline and ws == 1:          # reported at N=1 only
            line["cpu_baseline"] = cpu_baseline(reads, rnames, mnames, mons)
        dec.close()
        del flushes
    else:
        # same sequence of barriers as rank 0 (timed_resident: 2, timed_e2e: 2)
        for _ in range(4):
            barrier_sync(ws)

    # ---- replicas (extra key): every GPU decomposes its own 2 Mb array, one process per GPU (weak scaling) ----
    if ws > 1 and not args.no_extras:
        rn_r, reads_r, mn_r, mons_r, segs_r = workload(rank)
        dec = Decomposer(mons_r, *SCORING, devices=[local])
        flush = [torch.empty(256 << 20, dtype=torch.uint8, device="cuda:%d" % local)]
        dev_ms_r, wall_r, _, st_r = timed_resident(dec, pack_segments(segs_r), args, ws, flush, local)
        dev_ms_r = max_over_ranks(dev_ms_r, ws)
        cells_r = sum_over_ranks(float(headline_cells(reads_r, mons_r)), ws)
        if rank == 0:
            line["replicas"] = {"what": "one 2 Mb array per GPU, one process per GPU (round-1 measurement, weak scaling)",
                                "value": cells_r * args.steps / (dev_ms_r * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": dev_ms_r / args.steps}
        dec.close()
    if rank == 0:
        emit(line)
    if ws > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def ed_thr_leg(dec, packed, cells_hl, args):
    """SURVEY 8 row f2: the same batch through sd_decompose with the --ed_thr pre-filter on (FilterMonomersForRead,
    main.cpp:135-149): distances + ranks on the device, then the sweep on the re-ordered subset."""
    out = {}
    for thr in (40, 10 ** 6):
        dec.set_ed_thr(thr)
        for _ in range(2):
            dec.decompose(packed)
        dec.reset_stats()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            dec.decompose(packed)
        dt = (time.perf_counter() - t0) / args.steps
        st = dec.stats()
        out["ed_thr_%s" % ("all" if thr > 10 ** 5 else thr)] = {"e2e_ms_per_step": 1e3 * dt, "e2e_gcups": cells_hl / dt / 1e9,
                                                                  "copy_in_plus_filter_ms": st["h2d_ms"] / args.steps,
                                                                  "sweep_ms": st["sweep_ms"] / args.steps}
    dec.set_ed_thr(-1)
    out["what"] = ("sd_decompose with the --ed_thr pre-filter: hw_distance_rows_kernel + filter_rank_kernel run on the copy-in stream "
                   "(their time is inside copy_in_plus_filter_ms); ed_thr=40 keeps the closest rows, 'all' keeps every row re-ordered")
    return out


def config3_waves(device):
    """BASELINE config 3 (ONT-like 100 kb reads) on a 600-read sample through sd_decompose: 12,000 segments, more than one
    wave of backpointers, so that copy-in / kernels / copy-out of successive waves overlap (two wave slots)."""
    from stringdecomposer_b200 import Decomposer, synth
    from stringdecomposer_b200.hostpipe import segment_reads
    rn, reads, mn, mons = synth.config3(n_reads=600, read_len=100_000)
    segs, _ = segment_reads(reads, PART, OVERLAP)
    packed = pack_segments(segs)
    dec = Decomposer(mons, *SCORING, devices=[device])
    dec.decompose(packed)
    dec.reset_stats()
    t0 = time.perf_counter()
    dec.decompose(packed)
    dt = time.perf_counter() - t0
    st = dec.stats()
    dec.close()
    cells = float(cells_of(segs, mons))
    return {"what": "config 3 sample: 600 reads x 100 kb (60 Mb), one sd_decompose call with host buffers; the sweeps of the "
                    "waves alternate between two streams (the next wave fills the tail of the previous one; overlap counted once), the "
                    "traceback of a wave runs on a third stream under the next sweep",
            "segments": len(segs), "cells": cells, "sweep_ms": st["sweep_ms"], "traceback_ms_overlapped": st["traceback_ms"],
            "e2e_ms": 1e3 * dt, "e2e_over_sweep": 1e3 * dt / st["sweep_ms"],
            "sweep_gcups_actual_cells": cells / st["sweep_ms"] / 1e6, "e2e_gcups_actual_cells": cells / dt / 1e9,
            "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"],
            "geometry": {k: st[k] for k in ("C", "T", "NS", "NT", "NG", "lat")}}


def process_boundary(rnames, reads, mnames, mons):
    """The boundary main.py:194 actually crosses is a process: wall time of `dp` on the config-2 contig, cold (CUDA
    context creation, module load, FASTA ingest, TSV) -- not the warm-handle number `e2e` reports."""
    from stringdecomposer_b200 import synth
    dp = os.path.join(ROOT, "stringdecomposer_b200", "build", "bin", "dp")
    with tempfile.TemporaryDirectory() as td:
        rp, mp = os.path.join(td, "reads.fa"), os.path.join(td, "monomers.fa")
        synth.write_fasta(rp, rnames, reads)
        synth.write_fasta(mp, mnames, mons)
        walls = []
        for _ in range(3):
            t0 = time.perf_counter()
            with open(os.path.join(td, "out.tsv"), "wb") as out:
                subprocess.run([dp, rp, mp, "1", str(PART), str(OVERLAP)], stdout=out, stderr=subprocess.DEVNULL, check=True)
            walls.append(time.perf_counter() - t0)
    ctx = None
    probe = os.path.join(ROOT, "tools", "probes", "ctx_time")
    if os.path.exists(probe):
        try:
            outp = subprocess.run([probe], stdout=subprocess.PIPE, timeout=60).stdout.decode()
            ctx = float(outp.split("context")[1].split("ms")[0]) / 1e3
        except Exception:
            ctx = None
    return {"what": "wall time of the drop-in `dp` process on the config-2 contig (2 Mb), including CUDA start-up; "
                    "cuda_context_s is what an empty CUDA program needs on this box for cudaFree(0) (tools/probes/ctx_time.cu)",
            "dp_process_s": min(walls), "dp_process_s_all": walls, "cuda_context_s": ctx,
            "gcups": headline_cells(reads, mons) / min(walls) / 1e9}


# ALU-pipe instructions per cell of identity_kernel (2 VIADDMNMX + 2 VIADD + 1 LOP3; the ISETP issues elsewhere):
# 4.96 measured from sm__inst_executed_pipe_alu in profiles/r01_identity_r1.md
IDENTITY_ALU_OPS_PER_CELL = 5


def rescoring(segs, mons, recs, roff, device, alu_peak):
    """Extra, outside the timed step: the reference's next stage (main.py:29-60, one edlib global alignment per
    interval/monomer pair) on the intervals this very decomposition produced, against all 24 monomer rows."""
    from stringdecomposer_b200 import nw_identity, synth
    rows = list(mons) + [synth.revcomp(m) for m in mons]
    qs = [segs[s][int(r["start"]):int(r["end"]) + 1] for s in range(len(segs)) for r in recs[roff[s]:roff[s + 1]]]
    cells = float(sum(len(q) for q in qs)) * float(sum(len(t) for t in rows))
    best_k, best_w = 1e30, 1e30
    for _ in range(4):
        t0 = time.perf_counter()
        res = nw_identity(qs, rows, device=device)
        best_w = min(best_w, time.perf_counter() - t0)
        best_k = min(best_k, res["kernel_ms"])
    return {"what": "identity_kernel: NW identity of every decomposed interval x %d monomer rows (main.py aai)" % len(rows),
            "pairs": len(res["matches"]), "cells": cells, "kernel_ms": best_k, "kernel_gcups": cells / best_k / 1e6,
            "call_ms_host_buffers": best_w * 1e3, "alignments_per_s_host_buffers": len(res["matches"]) / best_w,
            "alu_ops_per_cell": IDENTITY_ALU_OPS_PER_CELL,
            "int_alu_roofline_frac": cells / (best_k * 1e-3) * IDENTITY_ALU_OPS_PER_CELL / alu_peak}


def sum_len(reads):
    return sum(len(r) for r in reads)


def _hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"]
    except Exception:
        return 6650.0


def cpu_baseline(reads, rnames, mnames, mons):
    """Reference binary (or the oracle port) on a bounded sample of the same workload, all host cores."""
    from stringdecomposer_b200 import synth
    ref = os.path.join(ROOT, "oracle", "_ref", "dp")
    kind = "reference"
    if not os.path.exists(ref):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "port"], check=False)
        ref, kind = os.path.join(ROOT, "oracle", "_build", "oracle_dp"), "port"
    if not os.path.exists(ref):
        return {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": "oracle not built"}
    cores = os.cpu_count() or 1
    sample = reads[0]
    with tempfile.TemporaryDirectory() as td:
        rp, mp = os.path.join(td, "reads.fa"), os.path.join(td, "monomers.fa")
        synth.write_fasta(rp, rnames[:1], [sample])
        synth.write_fasta(mp, mnames, mons)
        t0 = time.perf_counter()
        with open(os.path.join(td, "out.tsv"), "wb") as out:
            subprocess.run([ref, rp, mp, str(cores), str(PART), str(OVERLAP)], stdout=out, stderr=subprocess.DEVNULL, check=True)
        dt = time.perf_counter() - t0
    cells = len(sample) * 2 * sum(len(m) for m in mons)
    return {"value": cells / dt / 1e9, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": "the full config-2 contig (2,000,000 bp, 400 segments), dp -t %d, process wall time %.2f s" % (cores, dt),
            "process_wall_s": dt}


if __name__ == "__main__":
    main()
