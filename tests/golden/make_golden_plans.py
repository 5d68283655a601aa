"""Writes tests/golden/plans.json: the launch geometry the planner picks for a grid of shapes.

The grid is every monomer-set shape of test_host.py's planner test (1 to 2,047 monomers, rows of 1 to 1,536 bp), plus
the 12 DXZ1 monomers, crossed with segment lengths of 40, 5,500, 20,500 and 100,000 bp and 19, 400 and 40,000 segments
on one device.  The table was written from the planner of the commit before segments could be streamed through the
sweep kernels; test_long_segments.py checks that every shape that planned then still gets the same geometry and reads
its symbols from shared memory (stream == 0).

    python tests/golden/make_golden_plans.py [path/to/stringdecomposer_b200/csrc]

The planner comes from the given csrc directory (default: this checkout's): its plan.cpp is compiled with
tests/emu/plan_probe.cpp into a temporary library.
"""
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
FIELDS = ("packed", "C", "T", "NS", "NT", "NG", "lat", "scanw", "SG")
SEG_LENS = (40, 5500, 20500, 100000)
SEG_COUNTS = (19, 400, 40000)


def monomer_sets():
    """-> [(name, monomers)]: test_host.py's planner shapes (same generator, same seeds) and the DXZ1 set."""
    out = []
    al = np.frombuffer(b"ACGT", dtype=np.uint8)
    for N in (1, 5, 13, 32, 33, 100, 256, 1000, 2047):
        rng = np.random.default_rng(N)

        def rs(n):
            return al[rng.integers(0, 4, n)].tobytes().decode()
        for L in (1, 7, 48, 171, 340, 700, 1536):
            if N * L > 200000:
                continue
            mons = [rs(int(rng.integers(max(1, L // 2), L + 1))) for _ in range(N)]
            mons[0] = rs(L)
            rs(40)                           # the test's segment: keeps the generator in step with test_host.py
            out.append(("N%d_L%d" % (N, L), mons))
    seqs, cur = [], None
    for ln in open(os.path.join(HERE, "DXZ1_star_monomers.fa")):
        if ln.startswith(">"):
            cur = []
            seqs.append(cur)
        elif cur is not None:
            cur.append(ln.strip().upper())
    out.append(("DXZ1", ["".join(s) for s in seqs]))
    return out


def plan(lib, mons, seg_len, nseg, scoring=(-1, -1, -1, 1)):
    """-> dict of the geometry fields (plus "stream"), or {"error": message}."""
    blob = "".join(mons).encode()
    off = np.zeros(len(mons) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(m) for m in mons])
    out = (C.c_int32 * 10)()
    msg = C.create_string_buffer(512)
    st = lib.sd_plan_probe(blob, off.ctypes.data_as(C.POINTER(C.c_int64)), len(mons), *scoring, seg_len, nseg, out, msg, 512)
    if st:
        return {"error": msg.value.decode()}
    d = dict(zip(FIELDS, (int(v) for v in out[:9])))
    d["stream"] = int(out[9])
    return d


def build(out_dir, csrc=None):
    """Compile plan_probe.cpp + csrc/plan.cpp (host code only, as the emulator build does) -> path of the library."""
    csrc = os.path.abspath(csrc or os.path.join(HERE, "..", "..", "stringdecomposer_b200", "csrc"))
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    lib = os.path.join(out_dir, "libsd_plan_probe.so")
    subprocess.run([cxx, "-std=c++17", "-O1", "-fPIC", "-shared", "-DSD_EMULATOR_BUILD", "-I" + csrc, "-o", lib,
                    os.path.join(HERE, "..", "emu", "plan_probe.cpp"), os.path.join(csrc, "plan.cpp")], check=True)
    return lib


def load(path):
    lib = C.CDLL(path)
    lib.sd_plan_probe.argtypes = [C.c_char_p, C.POINTER(C.c_int64), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_int32, C.c_int64, C.POINTER(C.c_int32), C.c_char_p, C.c_int32]
    lib.sd_plan_probe.restype = C.c_int
    return lib


def main():
    with tempfile.TemporaryDirectory() as td:
        lib = load(build(td, sys.argv[1] if len(sys.argv) > 1 else None))
        write_table(lib)


def write_table(lib):
    rows = []
    for name, mons in monomer_sets():
        for n in SEG_LENS:
            for nseg in SEG_COUNTS:
                d = plan(lib, mons, n, nseg)
                d.pop("stream", None)
                rows.append(dict(set=name, seg_len=n, nseg=nseg, **d))
    with open(os.path.join(HERE, "plans.json"), "w") as f:
        json.dump({"fields": list(FIELDS), "plans": rows}, f, indent=0)
        f.write("\n")
    print("%d shapes, %d refused" % (len(rows), sum("error" in r for r in rows)))


if __name__ == "__main__":
    main()
