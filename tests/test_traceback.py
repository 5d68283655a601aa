"""The traceback kernel on its own, against a walker written from the reference.

On the GPU the traceback only ever sees the paths real sweeps produce: nearly diagonal, with short indels.  Here
tests/cuda/traceback_probe.cu runs traceback_kernel and gather_kernel (traceback_kernels.cuh) on tables the test
writes, and tests/emu/traceback_twin.cpp runs the emulator's walker (sweep_core.cuh: traceback_segment + fetch_code) on
the same file.  Geometry and layout come from an SD_DUMP_TABLES dump of a real run, so the walk reads exactly the layouts
the backend uses; the codes and J in it are replaced by
(a) the oracle's tables, encoded into that layout, with random bits in every cell the walk must never read (pad cells,
    the stored k == 0 codes, columns past a segment's end): expected sd_oracle.align_segment;
(b) constructed move fields -- long insertion and deletion runs, diagonal runs at the 32-column window and the 8-window
    ring, diagonal/deletion alternation (the walk drifts out of its cached words on every step), jumps at word and lane
    boundaries, k == 0 insertion runs and the i == 1 row-0 case, reverse-complement rows, rows of slot groups >= 1,
    --ed_thr rank permutations with dropped ranks, random mixes: expected the walker of test_oracle.py, written from
    main.cpp:217-267 and not from the kernel;
(c) a jump to a row outside the monomer set, or to a dropped rank, in one segment of several: expected error word 1,
    count 0 for that segment and the other segments' records unchanged.
Constructed fields are valid by construction and checked before a file is written: column 0 holds only the codes 0
and 3 and every jump row is in range (except where (c) wants it otherwise), so the walk cannot leave its tables."""
import os
import subprocess

import numpy as np
import pytest

import cases
import sd_oracle
from test_dp_tables import cell_words, dxz1_inputs, read_dump, slot_inputs, word_bias
from test_oracle import walk_tables
from test_score_domain import decompose

CSRC = os.path.join(cases.ROOT, "stringdecomposer_b200", "csrc")
DEFAULT = (-1, -1, -1, 1)


@pytest.fixture(scope="module")
def twin(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("traceback_twin") / "traceback_twin")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"       # the same choice as tests/emu/Makefile
    subprocess.run([cxx, "-std=c++17", "-O2", "-Wall", "-Wno-unknown-pragmas", "-I", CSRC, "-o", out,
                    os.path.join(cases.HERE, "emu", "traceback_twin.cpp")], check=True)
    return out


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("traceback_probe") / "traceback_probe")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")          # the same override as csrc/Makefile
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-I", CSRC,
                    "-o", out, os.path.join(cases.HERE, "cuda", "traceback_probe.cu")], check=True)
    return out


# ---- a real run's layout -------------------------------------------------------------------------------------------------

def layout(flavour, mons, segs, env, tmp_path, ed_thr=-1):
    """the wave of a real run (one wave: the inputs are small) -> its dump"""
    d = tmp_path / "dump"
    d.mkdir(exist_ok=True)
    for f in os.listdir(d):
        os.remove(d / f)
    decompose(flavour, mons, segs, DEFAULT, dict(env, SD_DUMP_TABLES=str(d)), ed_thr)
    (f,) = os.listdir(d)
    w = read_dump(str(d / f))
    assert w["first"] == 0 and w["nseg"] == len(segs)
    return w


class Tables:
    """the codes and JR of a wave in decoded form: every word starts random, live cells are set one row at a time"""

    def __init__(self, w, rng):
        self.w = w
        self.dec = rng.integers(0, 1 << 32, w["codes"].size, dtype=np.uint64)
        self.jr = rng.integers(-1000, 1000, w["jr"].shape).astype(np.int32)

    def set_row(self, s, row, codes):
        """codes [n][L-1] of cells k >= 1 of full-set row `row` of segment s"""
        n, L1 = codes.shape
        if L1 == 0:
            return
        idx, shift, _ = cell_words(self.w, s, row, L1 + 1, n)
        c = codes.astype(np.uint64) << shift[None, :]
        m = np.uint64(3) << shift[None, :]
        # cells of one row never share a word bit range, so the updates of one word may be applied one after the other
        for j in range(L1):
            self.dec[idx[:, j]] = (self.dec[idx[:, j]] & ~m[:, j]) | c[:, j]

    def set_j(self, s, J, argJ):
        o = int(self.w["seg_j_off"][s])
        n = len(J) - 1
        self.jr[o + 1:o + n + 1, 0] = J[1:]
        self.jr[o + 1:o + n + 1, 1] = argJ[1:]

    def raw(self):
        """the words as the sweep stores them: decoded minus the bias of each word"""
        g = self.w["g"]
        return ((self.dec - word_bias(g, np.arange(self.dec.size) % g["CW"])) & 0xFFFFFFFF).astype(np.uint32)


def write_file(path, w, tabs, segs, rows, scoring, r2r=None):
    g = w["g"]
    nseg, R = len(segs), len(rows)
    assert R == 2 * g["M"]
    so = np.zeros(nseg + 1, np.int64)
    so[1:] = np.cumsum([len(s) for s in segs])
    ro = np.zeros(R + 1, np.int32)
    ro[1:] = np.cumsum([len(r) for r in rows])
    hdr = [g[k] for k in ("packed", "C", "T", "nslots", "M", "NS", "NT", "CW", "NG", "SG", "lat", "scanw", "stream")]
    hdr += list(scoring) + [nseg, len(w["cta_code_off"]) - 1, r2r is not None]
    with open(path, "wb") as f:
        f.write(np.array(hdr, np.int32).tobytes() + so.tobytes() + ro.tobytes())
        f.write("".join(segs).encode() + "".join(rows).encode())
        f.write(np.asarray(w["cta_code_off"], np.int64).tobytes() + tabs.raw().tobytes())
        f.write(np.asarray(w["seg_j_off"], np.int64).tobytes() + tabs.jr.tobytes())
        if r2r is not None:
            f.write(np.asarray(r2r, np.int32).tobytes())


def run_files(binary, paths):
    """one process for many files: the probe pays for its CUDA context once"""
    subprocess.run([binary] + [str(p) for p in paths], check=True)


def read_result(path, nseg):
    v = np.fromfile(str(path) + ".out", np.int32)
    error, total, counts = int(v[0]), int(v[1]), v[2:2 + nseg]
    recs = v[2 + nseg:].reshape(-1, 4)
    assert len(recs) == max(total, 0)
    per, pos = [], 0
    for c in counts:
        per.append([tuple(int(x) for x in r) for r in recs[pos:pos + max(c, 0)]])
        pos += max(c, 0)
    return error, total, [int(c) for c in counts], per


def run_file(binary, path, nseg):
    run_files(binary, [path])
    return read_result(path, nseg)


def as_int(recs):
    return [(r, a, b, int(sc)) for r, a, b, sc in recs]


# ---- (a) the oracle's tables -----------------------------------------------------------------------------------------------

def run_oracle_tables(binary, flavour, tmp_path, mons, segs, env, scoring=DEFAULT, ed_thr=-1, seed=0):
    w = layout(flavour, mons, segs, env, tmp_path, ed_thr)
    rows = sd_oracle.rows_of(mons)
    tabs = Tables(w, np.random.default_rng(seed))
    r2r = np.full((len(segs), len(rows)), -1, np.int32) if ed_thr >= 0 else None
    want = []
    for s, seg in enumerate(segs):
        t = sd_oracle.dp_tables(seg, mons, scoring, ed_thr)
        ro = t["row_off"]
        for x, row in enumerate(t["keep"]):
            tabs.set_row(s, row, t["code"][:, ro[x] + 1:ro[x + 1]])
        tabs.set_j(s, t["J"], t["argJ"])
        if r2r is not None:
            r2r[s, :len(t["keep"])] = t["keep"]
        want.append(as_int(sd_oracle.align_segment(seg, mons, scoring, ed_thr)))
    path = tmp_path / "oracle.bin"
    write_file(path, w, tabs, segs, rows, scoring, r2r)
    error, total, counts, got = run_file(binary, path, len(segs))
    for s in range(len(segs)):
        assert got[s] == want[s], ("segment %d (%d bp)" % (s, len(segs[s])), w["g"], env, ed_thr, first_difference(got[s], want[s]))
    assert error == 0 and total == sum(len(x) for x in want)


ORACLE_CASES = [("classic 19,10,3", {"SD_LAT": "0", "SD_GEOM": "19,10,3"}, "dxz1", -1),
                ("classic s32 8,4,3", {"SD_LAT": "0", "SD_GEOM": "8,4,3", "SD_FORCE_S32": "1"}, "slots", -1),
                ("deferred 6,32", {"SD_LAT": "1", "SD_GEOM": "6,32,1", "SD_LAT_WARPS": "2"}, "dxz1", -1),
                ("group 4 slots", {"SD_GROUP_SLOTS": "4"}, "dxz1", -1),
                ("ed_thr", {"SD_LAT": "0"}, "dxz1", 12)]


def oracle_case_inputs(kind):
    return dxz1_inputs(5) if kind == "dxz1" else slot_inputs(8 * 4 + 3, 32)


# ---- (b) constructed move fields -------------------------------------------------------------------------------------------

def k0_codes(seg, rows, J, scoring):
    """the k == 0 move of every row and column from J (main.cpp:245 with H[i][r][0] = J[i] + s, :191-193, and
    H[0][r][0] = s, :173-177): 1 when the insertion equality holds, else 3"""
    ins, _, mm, ma = scoring
    n = len(seg)
    out = np.full((n, len(rows)), 3, np.int8)
    for x, r in enumerate(rows):
        s = np.array([ma if c == r[0] else mm for c in seg], np.int64)
        h = np.concatenate([[s[0]], J[1:n] + s[1:]])
        out[1:, x] = np.where(h[1:] == h[:-1] + ins, 1, 3)
    return out


def construct(rng, seg, rows, keep, scoring, mix, pick=None, pick_row=None, J=None):
    """a move field over the kept rows (in rank order) of one segment -> the table dict walk_tables reads.
    mix: probabilities of the codes 0..3 in cells the walk does not visit; pick(i, rank, k) -> the code of a cell the
    walk visits (k >= 1), pick_row(i) -> the rank a jump at column i names.  Checked: column 0 holds only 0 and 3 at
    k >= 1, every jump rank is in range."""
    n = len(seg)
    kr = [rows[r] for r in keep]
    ro = np.zeros(len(kr) + 1, np.int32)
    ro[1:] = np.cumsum([len(r) for r in kr])
    code = rng.choice(4, size=(n, int(ro[-1])), p=mix).astype(np.int8)
    code[0][np.isin(code[0], (1, 2))] = 0
    if J is None:
        J = rng.integers(-60, 60, n + 1).astype(np.int64)
    argJ = rng.integers(0, len(kr), n + 1).astype(np.int32)
    k0 = k0_codes(seg, kr, J, scoring)
    for x in range(len(kr)):
        code[:, ro[x]] = k0[:, x]
    # the walk, assigning the cells it visits (each cell and each argJ[i] is visited at most once: i and k only fall)
    i, x = n - 1, int(argJ[n]) if pick_row is None else pick_row(n)
    argJ[n] = x
    k = int(ro[x + 1] - ro[x]) - 1
    while True:
        if k >= 1 and pick is not None:
            c = pick(i, x, k)
            if i == 0 and c in (1, 2):
                c = 0
            code[i, ro[x] + k] = c
        c = int(code[i, ro[x] + k])
        if c == 0:
            k -= 1
        elif c == 1:
            i -= 1
        elif c == 2:
            i, k = i - 1, k - 1
        elif i == 0:
            break
        else:
            if pick_row is not None:
                argJ[i] = pick_row(i)
            x = int(argJ[i])
            i -= 1
            k = int(ro[x + 1] - ro[x]) - 1
    assert not np.isin(code[0], (1, 2)).any() and (0 <= argJ[1:]).all() and (argJ[1:] < len(kr)).all()
    return {"code": code, "J": J, "argJ": argJ, "row_off": ro, "keep": list(keep)}


def pattern(moves):
    """pick() that plays `moves` over and over"""
    state = {"n": 0}

    def pick(i, x, k):
        c = moves[state["n"] % len(moves)]
        state["n"] += 1
        return c
    return pick


def fields(rng, seg, rows, keep, scoring, C, T):
    """(name, table) of every family of constructed fields for one segment"""
    L = max(len(rows[r]) for r in keep)
    nk = len(keep)
    long_ranks = [x for x, r in enumerate(keep) if len(rows[r]) == L]
    mostly_diag = (0.05, 0.05, 0.85, 0.05)
    out = []
    for run in (40, 100, 300):
        out.append(("insertion run %d" % run, construct(rng, seg, rows, keep, scoring, mostly_diag, pattern([1] * run + [2, 2, 0]))))
    out.append(("deletion runs across rows", construct(rng, seg, rows, keep, scoring, mostly_diag, pattern([0]),
                                                        pick_row=lambda i: long_ranks[i % len(long_ranks)])))
    for d in (31, 32, 33, 63, 64, 65, 255, 256, 257):
        for odd in (0, 1, 3):
            out.append(("diagonal run %d then %d" % (d, odd),
                        construct(rng, seg, rows, keep, scoring, mostly_diag, pattern([2] * d + [odd]),
                                  pick_row=lambda i: long_ranks[i % len(long_ranks)])))
    out.append(("diagonal/deletion alternation", construct(rng, seg, rows, keep, scoring, mostly_diag, pattern([2, 0]))))
    out.append(("diagonal/insertion alternation", construct(rng, seg, rows, keep, scoring, mostly_diag, pattern([2, 1]))))
    for ks in ((7, 8, 9), (15, 16, 17), (C - 1, C, C + 1), (C * T - 1, C * T - 2), (1, 2)):
        out.append(("jumps at k %s" % (ks,),
                    construct(rng, seg, rows, keep, scoring, mostly_diag, lambda i, x, k, ks=ks: 3 if k in ks else 2,
                              pick_row=lambda i: int(rng.integers(0, nk)))))
    # k == 0 insertion runs: J chosen so that main.cpp:245's equality holds for every row whose first symbol is A
    ins, _, mm, ma = scoring
    s = np.array([ma if c == "A" else mm for c in seg], np.int64)
    J = np.zeros(len(seg) + 1, np.int64)
    J[1] = s[0] + ins - s[1] if len(seg) > 1 else 0       # i == 1: the row-0 cell H[0][r][0] = s (main.cpp:173-177)
    for i in range(2, len(seg)):
        J[i] = J[i - 1] + s[i - 1] + ins - s[i] if rng.random() < 0.9 else J[i - 1] + 5
    J[len(seg)] = J[len(seg) - 1] + 3
    out.append(("k == 0 insertion runs", construct(rng, seg, rows, keep, scoring, mostly_diag, pattern([0] * 5 + [2]), J=J)))
    for mix in ((0.25, 0.25, 0.25, 0.25), (0.6, 0.1, 0.28, 0.02), (0.1, 0.6, 0.28, 0.02), (0.02, 0.02, 0.95, 0.01)):
        out.append(("random mix %s" % (mix,), construct(rng, seg, rows, keep, scoring, mix, pick_row=lambda i: int(rng.integers(0, nk)))))
    return out


def run_fields(binary, flavour, tmp_path, mons, segs, env, scoring=DEFAULT, permute=False, seed=1):
    """every family on every segment of a real run's layout, one file per family, all segments at once"""
    rng = np.random.default_rng(seed)
    w = layout(flavour, mons, segs, env, tmp_path)
    g = w["g"]
    rows = list(sd_oracle.rows_of(mons))
    # rows starting with A (the k == 0 insertion runs); the layout only depends on their lengths
    rows = ["A" + r[1:] if rng.random() < 0.7 else r for r in rows]
    R = len(rows)
    keeps = []
    for s in range(len(segs)):
        if permute:                # --ed_thr: a permutation of a subset of the rows; the dropped ranks map to -1
            keeps.append([int(r) for r in rng.permutation(R)[:max(1, R - int(rng.integers(0, R)))]])
        else:
            keeps.append(list(range(R)))
    per_seg = [fields(rng, seg, rows, keeps[s], scoring, g["C"], g["T"]) for s, seg in enumerate(segs)]
    r2r = None
    if permute:
        r2r = np.full((len(segs), R), -1, np.int32)
        for s in range(len(segs)):
            r2r[s, :len(keeps[s])] = keeps[s]
    paths, wants = [], []
    for f in range(len(per_seg[0])):
        tabs = Tables(w, rng)
        want = []
        for s, seg in enumerate(segs):
            t = per_seg[s][f][1]
            ro = t["row_off"]
            for x, row in enumerate(t["keep"]):
                tabs.set_row(s, row, t["code"][:, ro[x] + 1:ro[x + 1]])
            tabs.set_j(s, t["J"], t["argJ"])
            want.append(as_int(walk_tables(t, len(seg))))
        paths.append(tmp_path / ("field%02d.bin" % f))
        write_file(paths[-1], w, tabs, segs, rows, scoring, r2r)
        wants.append(want)
    run_files(binary, paths)
    for f, (path, want) in enumerate(zip(paths, wants)):
        error, total, counts, got = read_result(path, len(segs))
        for s in range(len(segs)):
            assert got[s] == want[s], ("%s, segment %d (%d bp)" % (per_seg[s][f][0], s, len(segs[s])), g, env,
                                       first_difference(got[s], want[s]))
        assert error == 0 and total == sum(len(x) for x in want), (per_seg[0][f][0], error, total)
    return w


def first_difference(got, want):
    for j, (a, b) in enumerate(zip(got, want)):
        if a != b:
            return "record %d: %s, want %s" % (j, a, b)
    return "%d records, want %d" % (len(got), len(want))


def field_inputs(C, T):
    """monomers up to the longest row the geometry takes (capped at 600 bp), a length-1 row, and segments of 1, 2, 31, 32,
    33 and 700 columns"""
    rng = np.random.default_rng(C * T)
    L = min(C * T, 600)
    mons = ["".join("ACGT"[x] for x in rng.integers(0, 4, n)) for n in (L, L - 1, max(2, L // 3), 1, 17)]
    segs = ["".join("ACGTN"[x] for x in rng.integers(0, 5, n)) for n in (700, 1, 2, 31, 32, 33)]
    return mons, segs


FIELD_GEOMS = [("classic 19,10,2", {"SD_LAT": "0", "SD_GEOM": "19,10,2"}),
               ("classic s32 24,8,3", {"SD_LAT": "0", "SD_GEOM": "24,8,3", "SD_FORCE_S32": "1"}),
               ("classic 48,32,1", {"SD_LAT": "0", "SD_GEOM": "48,32,1"}),
               ("classic 8,4,3", {"SD_LAT": "0", "SD_GEOM": "8,4,3"}),
               ("deferred 12,16", {"SD_LAT": "1", "SD_GEOM": "12,16,1", "SD_LAT_WARPS": "3"}),
               ("group 2 slots", {"SD_GROUP_SLOTS": "2", "SD_GEOM": "24,8,2"})]


def geom_of(env):
    C, T = 24, 8
    if "SD_GEOM" in env:
        C, T, _ = map(int, env["SD_GEOM"].split(","))
    return C, T


# ---- (c) the error path ----------------------------------------------------------------------------------------------------

def run_bad_rows(binary, flavour, tmp_path):
    mons, segs = slot_inputs(77, 40, nseg=5)
    w = layout(flavour, mons, segs, {"SD_LAT": "0", "SD_GEOM": "8,8,2"}, tmp_path)
    rows = sd_oracle.rows_of(mons)
    R = len(rows)
    for case in ("final row", "inner row", "dropped rank"):
        rng = np.random.default_rng(len(case))
        tabs = Tables(w, rng)
        want = []
        r2r = np.tile(np.arange(R, dtype=np.int32), (len(segs), 1)) if case == "dropped rank" else None
        for s, seg in enumerate(segs):
            t = sd_oracle.dp_tables(seg, mons)
            ro = t["row_off"]
            for x in range(R):
                tabs.set_row(s, x, t["code"][:, ro[x] + 1:ro[x + 1]])
            tabs.set_j(s, t["J"], t["argJ"])
            want.append(as_int(sd_oracle.align_segment(seg, mons)))
        bad = 4                                                  # 1,300 bp: several jumps
        o = int(w["seg_j_off"][bad])
        n = len(segs[bad])
        if case == "final row":
            tabs.jr[o + n, 1] = 2 * w["g"]["M"] + 5
        else:
            starts = [a for _, a, _, _ in want[bad] if a > 0]
            tabs.jr[o + starts[len(starts) // 2], 1] = R if case == "inner row" else R - 1
            if r2r is not None:
                r2r[bad, R - 1] = -1
        path = tmp_path / "bad.bin"
        write_file(path, w, tabs, segs, rows, DEFAULT, r2r)
        error, total, counts, got = run_file(binary, path, len(segs))
        assert error == 1 and counts[bad] == 0, (case, error, counts)
        for s in range(len(segs)):
            if s != bad:
                assert got[s] == want[s], (case, s)


# ---- CPU: the emulator's walker on the same files ----------------------------------------------------------------------------

def test_twin_on_oracle_tables(twin, tmp_path):
    for name, env, kind, thr in ORACLE_CASES:
        mons, segs = oracle_case_inputs(kind)
        run_oracle_tables(twin, cases.EMU_LIB, tmp_path, mons, segs, env, ed_thr=thr)


@pytest.mark.parametrize("name,env", FIELD_GEOMS[:2] + FIELD_GEOMS[4:5])
def test_twin_on_constructed_fields(twin, tmp_path, name, env):
    mons, segs = field_inputs(*geom_of(env))
    run_fields(twin, cases.EMU_LIB, tmp_path, mons, segs, env, permute="s32" in name)


def test_twin_error_path(twin, tmp_path):
    run_bad_rows(twin, cases.EMU_LIB, tmp_path)


# ---- GPU: traceback_kernel ---------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name,env,kind,thr", ORACLE_CASES, ids=[c[0] for c in ORACLE_CASES])
def test_gpu_traceback_on_oracle_tables(probe, tmp_path, name, env, kind, thr):
    mons, segs = oracle_case_inputs(kind)
    run_oracle_tables(probe, "cuda", tmp_path, mons, segs, env, ed_thr=thr)


@pytest.mark.gpu
@pytest.mark.parametrize("permute", [False, True])
@pytest.mark.parametrize("name,env", FIELD_GEOMS, ids=[g[0] for g in FIELD_GEOMS])
def test_gpu_traceback_on_constructed_fields(probe, tmp_path, name, env, permute):
    mons, segs = field_inputs(*geom_of(env))
    run_fields(probe, "cuda", tmp_path, mons, segs, env, permute=permute)


@pytest.mark.gpu
def test_gpu_traceback_error_path(probe, tmp_path):
    run_bad_rows(probe, "cuda", tmp_path)
