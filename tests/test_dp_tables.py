"""Every backpointer and every J of the sweeps against the oracle's DP table, cell by cell.

The record tests only see the cells a traceback walks through: on a config-2 segment about one backpointer in 4,000.
A sweep that writes a wrong code or a wrong J[i] anywhere else passes them until some input routes a path through that
cell.  Here SD_DUMP_TABLES makes the backend (or the emulator) write every wave's backpointer words and its {J, row}
array, and the test decodes them with its own restatement of the layout (DESIGN.md section 4, sweep_core.cuh:
place_row, lane_tid, fetch_code, decode_code) and compares them with sd_oracle.dp_tables:
- the code of every live cell (i, r, k >= 1): the move the reference's traceback takes there (main.cpp:242-253), which
  the tag order must reproduce in every cell (DESIGN section 3.2), in the classic and in the deferred form (3.8);
- J[i] and its lowest row for i = 1..n (J[n] is the final maximum).

Cells that are not compared, and why:
- pad cells (k >= the row's length) and the lanes of a slot past its row: no DP cell lives there;
- the stored k == 0 codes: the sweep never takes the insertion move at k == 0 (main.cpp:194) while the reference's
  traceback tests it there (:245); the traceback derives that move from J and the symbols and never reads the code;
- columns past a segment's end inside its CTA: a CTA sweeps as many columns as its longest segment, and nothing is
  stored or read past the end of the shorter ones;
- rows the --ed_thr filter dropped: they are swept but their row ends do not take part in J (their key is excluded),
  and no jump names them, so the traceback never enters them.  The kept rows are compared in rank order, which is also
  the tie-break order of J's row.

The CPU variants run the emulator on one case of each sweep kind and width; the gpu variants run the CUDA library on
the whole matrix."""
import os
import tempfile

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings

import cases
import sd_oracle
from stringdecomposer_b200 import synth
from test_properties import problem_env, problems
from test_score_domain import copies, decompose, deletion_for, random_monomers, row_limit_inputs

GEOM_FIELDS = ("packed", "C", "T", "nslots", "M", "NS", "NT", "CW", "NG", "SG", "lat", "scanw", "stream")
DEFAULT = (-1, -1, -1, 1)


# ---- the dump and its decoder --------------------------------------------------------------------------------------------

def read_dump(path):
    """one SD_DUMP_TABLES file (format: stringdecomposer_b200/csrc/common.h, dump_wave_tables)"""
    raw = open(path, "rb").read()
    hdr = np.frombuffer(raw, np.int32, 16)
    w = {"g": dict(zip(GEOM_FIELDS, (int(x) for x in hdr[:13]))), "first": int(hdr[13]), "nseg": int(hdr[14])}
    nctas, pos = int(hdr[15]), 64
    w["cta_code_off"] = np.frombuffer(raw, np.int64, nctas + 1, pos)
    pos += 8 * (nctas + 1)
    w["seg_j_off"] = np.frombuffer(raw, np.int64, w["nseg"] + 1, pos)
    pos += 8 * (w["nseg"] + 1)
    w["codes"] = np.frombuffer(raw, np.uint32, int(w["cta_code_off"][-1]), pos)
    pos += 4 * int(w["cta_code_off"][-1])
    w["jr"] = np.frombuffer(raw, np.int32, 2 * int(w["seg_j_off"][-1]), pos).reshape(-1, 2)
    assert pos + w["jr"].nbytes == len(raw), path
    return w


def cell_words(w, s, row, L, n):
    """where cells k = 1..L-1 of DP row `row` (an index into the full row set) of segment s of the wave live, columns
    0..n-1: -> word index [n][L-1], bit shift [L-1], bias of each word [L-1].  Restated from DESIGN section 4 and
    sweep_core.cuh:
      slot: packed, the forward row and its reverse complement share a slot (the reverse complement in bits 16..31)
      slot group grp = slot / SG; its CTA is s*NG + grp when NG > 1 (its slot instance slot - grp*SG), else the CTA
        s / NS holds NS segments of nslots slot instances each
      lane t = k / C of the slot instance holds cells [t*C, t*C + C); thread lane_tid = (ginst / spw)*32 +
        (ginst % spw)*T + t with spw = 32 / T slots per warp
      word wi = kk / cpw (cpw = 8 packed, 16 s32) of the CW words the thread stores per column, at
        cta_code_off[cta] + i*NT*CW + tid*CW + wi; cell c = kk % cpw at bits 2*(ncell-1-c) + half after adding the
        bias (4^ncell - 1)/3 per half (the sweep stores the raw digits)"""
    g = w["g"]
    packed, C, T = g["packed"], g["C"], g["T"]
    slot = (row if row < g["M"] else row - g["M"]) if packed else row
    half = 16 if packed and row >= g["M"] else 0
    grp = slot // g["SG"]
    if g["NG"] > 1:
        cta, ginst = s * g["NG"] + grp, slot - grp * g["SG"]
    else:
        cta, ginst = s // g["NS"], (s % g["NS"]) * g["nslots"] + slot
    k = np.arange(1, L)
    t, kk = k // C, k % C
    cpw = 8 if packed else 16
    wi, c = kk // cpw, kk % cpw
    spw = 32 // T
    tid = (ginst // spw) * 32 + (ginst % spw) * T + t
    col = int(w["cta_code_off"][cta]) + np.arange(n, dtype=np.int64)[:, None] * (g["NT"] * g["CW"])
    ncell = np.minimum(cpw, C - wi * cpw)
    return col + (tid * g["CW"] + wi)[None, :], (2 * (ncell - 1 - c) + half).astype(np.uint64), word_bias(g, wi)


def word_bias(g, wi):
    """the bias of word wi of a thread's CW words: (4^ncell - 1)/3 in each half"""
    cpw = 8 if g["packed"] else 16
    ncell = np.minimum(cpw, g["C"] - np.asarray(wi) * cpw)
    return (((0x55555555 >> (32 - 2 * ncell)) * (0x10001 if g["packed"] else 1)) & 0xFFFFFFFF).astype(np.uint64)


def decode_row(w, s, row, L, n):
    """codes [n][L-1] of DP row `row`, cells k = 1..L-1, of segment s of the wave (cell_words)"""
    idx, shift, bias = cell_words(w, s, row, L, n)
    words = w["codes"][idx].astype(np.uint64)
    return ((((words + bias[None, :]) & 0xFFFFFFFF) >> shift[None, :]) & 3).astype(np.int8)


def compare_segment(w, s, seg, mons, scoring, ed_thr):
    """the first difference of segment s of wave w from the oracle's table, or None"""
    n = len(seg)
    t = sd_oracle.dp_tables(seg, mons, scoring, ed_thr)
    jr = w["jr"][int(w["seg_j_off"][s]):int(w["seg_j_off"][s]) + n + 1]
    for i in range(1, n + 1):
        if (jr[i, 0], jr[i, 1]) != (t["J"][i], t["argJ"][i]):
            return "J[%d] = %s, want %s" % (i, tuple(jr[i]), (t["J"][i], t["argJ"][i]))
    ro = t["row_off"]
    for x, row in enumerate(t["keep"]):
        L = int(ro[x + 1] - ro[x])
        if L < 2:
            continue
        got = decode_row(w, s, row, L, n)
        want = t["code"][:, ro[x] + 1:ro[x + 1]]
        if not np.array_equal(got, want):
            i, kk = (int(v[0]) for v in np.nonzero(got != want))
            return "column %d, row %d (rank %d), k %d: code %d, want %d" % (i, row, x, kk + 1, got[i, kk], want[i, kk])
    return None


def check_tables(flavour, mons, segs, scoring=DEFAULT, env=None, ed_thr=-1):
    """decompose with SD_DUMP_TABLES and compare every segment's tables with the oracle -> stats"""
    with tempfile.TemporaryDirectory() as td:
        _, stats = decompose(flavour, mons, segs, scoring, dict(env or {}, SD_DUMP_TABLES=td), ed_thr)
        waves = [read_dump(os.path.join(td, f)) for f in sorted(os.listdir(td))]
    assert sum(w["nseg"] for w in waves) == len(segs) and waves
    for w in waves:
        g = w["g"]
        assert (g["C"], g["T"], g["NS"], g["NG"], g["lat"], g["packed"], g["stream"]) == \
            tuple(stats[key] for key in ("C", "T", "NS", "NG", "lat", "packed", "stream")), (g, stats)
        for s in range(w["nseg"]):
            seg = segs[w["first"] + s]
            bad = compare_segment(w, s, seg, mons, scoring, ed_thr)
            assert bad is None, "segment %d (%d bp): %s; geometry %s, scoring %s, env %s, ed_thr %d" % (
                w["first"] + s, len(seg), bad, g, scoring, env, ed_thr)
    return stats


# ---- inputs ----------------------------------------------------------------------------------------------------------------

def slot_inputs(seed, longest, nseg=7):
    """monomers of 1 .. longest bp (a length-1 row among them) and nseg segments of mixed lengths, 1 bp included"""
    rng = np.random.default_rng(seed)
    lens = sorted({1, 2, longest} | {int(x) for x in rng.integers(1, longest + 1, 3)})
    mons = random_monomers(rng, lens)
    seg_lens = [1, 2, 900, 37, 1300, 5, 640][:nseg]
    return mons, [copies(rng, mons, n, rate=0.05) for n in seg_lens]


def dxz1_inputs(seed, lens=(1, 300, 1200, 61, 2)):
    names, mons = synth.load_dxz1()
    arr = synth.hor_array(mons, sum(lens) + 10, 0.04, seed=seed)
    segs, pos = [], 0
    for n in lens:
        segs.append(arr[pos:pos + n])
        pos += n
    return mons, segs


def one_rows_distance(segs, mons):
    rows = sd_oracle.rows_of(mons)
    d = sorted(sd_oracle.lib().sdo_hw_distance(r.encode(), len(r), segs[-1].encode(), len(segs[-1])) for r in rows)
    return d[len(d) // 2]


CLASSIC_GEOMS = ("8,32,1", "16,16,1", "24,8,1", "24,8,2", "32,8,1", "48,4,2", "48,4,3", "12,16,1", "20,10,1", "20,10,2",
                 "19,10,1", "19,10,3", "8,1,4", "8,2,2", "16,1,1", "24,1,2", "32,2,1", "48,1,1", "8,4,3", "48,32,1")
DEFERRED_GEOMS = (("6,32,1", "4"), ("6,32,1", "1"), ("6,32,1", "2"), ("12,16,1", "3"), ("12,16,1", "1"), ("24,8,1", "0"),
                  ("24,8,1", "1"), ("12,32,1", "2"), ("24,16,1", "1"), ("24,32,1", "2"), ("48,32,1", "1"))


def run_classic(flavour, geom, force32):
    C, T, NS = map(int, geom.split(","))
    mons, segs = slot_inputs(C * T + NS, min(C * T, 171))
    stats = check_tables(flavour, mons, segs, DEFAULT, {"SD_LAT": "0", "SD_GEOM": geom, "SD_FORCE_S32": force32})
    assert (stats["C"], stats["T"], stats["NS"], stats["lat"]) == (C, T, NS, 0), stats
    assert stats["packed"] == (force32 == "0"), stats


def run_deferred(flavour, geom, warps, force32):
    C, T, _ = map(int, geom.split(","))
    mons, segs = slot_inputs(C * T + 1000, min(C * T, 171), nseg=4)
    stats = check_tables(flavour, mons, segs, (-2, -2, -3, 1),
                         {"SD_LAT": "1", "SD_GEOM": geom, "SD_LAT_WARPS": warps, "SD_FORCE_S32": force32})
    assert (stats["C"], stats["T"], stats["lat"]) == (C, T, 1), stats


GROUP_ENVS = ({"SD_GROUP_SLOTS": "1"}, {"SD_GROUP_SLOTS": "4"}, {"SD_GROUP_SLOTS": "8"},
              {"SD_GROUP_SLOTS": "4", "SD_GROUP_GSLOTS": "2"}, {"SD_GROUP_SLOTS": "1", "SD_FORCE_S32": "1"})


def run_group(flavour, env):
    mons, segs = dxz1_inputs(9)
    stats = check_tables(flavour, mons, segs, DEFAULT, env)
    assert stats["NG"] > 1 and stats["lat"] == 0, stats


SWEEP_ENVS = (("classic", {"SD_LAT": "0"}), ("deferred", {"SD_LAT": "1"}), ("group", {"SD_GROUP_SLOTS": "4"}))


def run_streamed(flavour, env):
    mons, segs = dxz1_inputs(17)
    stats = check_tables(flavour, mons, segs, DEFAULT, dict(env, SD_STREAM_SYMBOLS="1"))
    assert stats["stream"] == 1 or stats["NG"] > 1, stats


def run_ed_thr(flavour, env):
    mons, segs = dxz1_inputs(23)
    for thr in (0, one_rows_distance(segs, mons), 10_000):
        check_tables(flavour, mons, segs, DEFAULT, env, thr)


SCORINGS = ((-2, -2, -3, 1), (2, -1, -3, 1), (-1, 2, -2, 1), (3, 3, -2, 4), (-30, -1, -1, 1), (-300, -1, -1, 1))


def run_scoring(flavour, scoring):
    rng = np.random.default_rng(abs(scoring[0]) * 100 + abs(scoring[1]))
    mons = random_monomers(rng, [171, 160, 120, 1])
    segs = [copies(rng, mons, n) for n in (1500, 700, 1)]
    for _, env in SWEEP_ENVS:
        check_tables(flavour, mons, segs, scoring, env)


def run_key_domain(flavour, L, target):
    rng = np.random.default_rng(L * 7 + 11)
    mons = random_monomers(rng, [L, L])
    scoring = (-1, deletion_for(L, target), -1, 1)
    segs = [copies(rng, mons, 3000)]
    for _, env in SWEEP_ENVS:
        if env.get("SD_LAT") == "1":
            env = dict(env, SD_LAT_WARPS="1")          # the deferred sweep's profile slices of 1,536 bp rows: one warp
        assert check_tables(flavour, mons, segs, scoring, env)["packed"] == 0


def run_n_symbols(flavour, env):
    rng = np.random.default_rng(41)
    mons = [synth_n(rng, n) for n in (40, 7, 1, 90)] + ["N"]
    segs = [synth_n(rng, n) for n in (500, 1, 120)]
    check_tables(flavour, mons, segs, DEFAULT, env)


def synth_n(rng, n):
    return np.frombuffer(b"ACGTN", np.uint8)[rng.integers(0, 5, n)].tobytes().decode()


# ---- CPU: the emulator, one case of each sweep kind and width -------------------------------------------------------------

def test_emulated_tables_against_oracle():
    run_classic(cases.EMU_LIB, "19,10,3", "0")
    run_classic(cases.EMU_LIB, "8,4,3", "1")
    run_deferred(cases.EMU_LIB, "6,32,1", "2", "0")
    run_deferred(cases.EMU_LIB, "12,16,1", "1", "1")
    run_group(cases.EMU_LIB, {"SD_GROUP_SLOTS": "4"})
    run_streamed(cases.EMU_LIB, {"SD_LAT": "0"})
    run_ed_thr(cases.EMU_LIB, {"SD_LAT": "1"})
    run_n_symbols(cases.EMU_LIB, {})


def test_decoder_sees_a_single_wrong_code(tmp_path):
    # the comparison must find one wrong code among all cells: change one cell of a real dump and expect that cell
    mons, segs = slot_inputs(3, 40, nseg=3)
    decompose(cases.EMU_LIB, mons, segs, DEFAULT, {"SD_LAT": "0", "SD_GEOM": "8,8,2", "SD_DUMP_TABLES": str(tmp_path)})
    (f,) = os.listdir(tmp_path)
    w = read_dump(os.path.join(tmp_path, f))
    g = w["g"]
    assert g["packed"] == 1 and g["NS"] == 2 and compare_segment(w, 2, segs[2], mons, DEFAULT, -1) is None
    slot = len(mons) - 1                                   # the longest row's reverse complement: the upper half of its words
    row, n, L = slot + g["M"], len(segs[2]), len(mons[slot])
    before = decode_row(w, 2, row, L, n)
    k, i = L - 1, 500
    kk, spw = k % g["C"], 32 // g["T"]
    ginst = (2 % g["NS"]) * g["nslots"] + slot
    tid = (ginst // spw) * 32 + (ginst % spw) * g["T"] + k // g["C"]
    at = int(w["cta_code_off"][2 // g["NS"]]) + i * g["NT"] * g["CW"] + tid * g["CW"] + kk // 8
    ncell = min(8, g["C"] - kk // 8 * 8)
    bias = ((0x55555555 >> (32 - 2 * ncell)) * 0x10001) & 0xFFFFFFFF
    codes = w["codes"].copy()
    codes[at] = np.uint32((((int(codes[at]) + bias) ^ (1 << (16 + 2 * (ncell - 1 - kk % 8)))) - bias) & 0xFFFFFFFF)
    w["codes"] = codes
    after = decode_row(w, 2, row, L, n)
    assert np.count_nonzero(before != after) == 1 and after[i, k - 1] != before[i, k - 1]
    assert compare_segment(w, 2, segs[2], mons, DEFAULT, -1).startswith("column %d, row %d (rank %d), k %d:" % (i, row, row, k))


# ---- GPU: the whole matrix ---------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("geom", CLASSIC_GEOMS)
@pytest.mark.parametrize("force32", ["0", "1"])
def test_gpu_classic_tables(geom, force32):
    run_classic("cuda", geom, force32)


@pytest.mark.gpu
@pytest.mark.parametrize("geom,warps", DEFERRED_GEOMS)
@pytest.mark.parametrize("force32", ["0", "1"])
def test_gpu_deferred_tables(geom, warps, force32):
    run_deferred("cuda", geom, warps, force32)


@pytest.mark.gpu
@pytest.mark.parametrize("env", GROUP_ENVS, ids=str)
def test_gpu_group_tables(env):
    run_group("cuda", env)


@pytest.mark.gpu
@pytest.mark.parametrize("name,env", SWEEP_ENVS)
def test_gpu_streamed_and_ed_thr_tables(name, env):
    run_streamed("cuda", env)
    run_ed_thr("cuda", env)
    run_n_symbols("cuda", env)


@pytest.mark.gpu
@pytest.mark.parametrize("scoring", SCORINGS, ids=str)
def test_gpu_scoring_tables(scoring):
    run_scoring("cuda", scoring)


@pytest.mark.gpu
@pytest.mark.parametrize("target", ("3*2^17", "max"))
@pytest.mark.parametrize("L", (300, 600, 1000, 1536))
def test_gpu_key_domain_tables(L, target):
    run_key_domain("cuda", L, target)


@pytest.mark.gpu
def test_gpu_row_limit_tables():
    for dup in (0, 1):
        mons, segs = row_limit_inputs(dup)
        assert check_tables("cuda", mons, segs)["NG"] > 1


@pytest.mark.gpu
@settings(max_examples=40, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(problems())
def test_gpu_tables_property(problem):
    monomers, segments, scoring = problem[:3]
    check_tables("cuda", monomers, segments, scoring, {k: v for k, v in problem_env(problem).items() if v})
