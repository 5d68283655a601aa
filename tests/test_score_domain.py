"""Edges of the score domain against the int64 oracle.

The planner accepts any scoring whose scores stay clear of the reference's INF sentinel and inside the exact float
range of its output.  These tests walk the edges of that domain: 32-bit sweeps with long monomers and large deletion
penalties (where rel * 4096 of an interior cell no longer fits the column key's 32 bits), the last packed and the
first 32-bit monomer length of a scoring, rebases of the reference base in nearly every column, the row bits of the
key at 4,096 rows, and record scores near 2^23.

Every case runs on the CPU through the host emulator, which also forms the kernels' per-lane column key
(sweep_core.cuh: lane_key) next to its own select-based key and fails on any difference (key_violation), and, marked
`gpu`, through the CUDA library.  Segments are mutated copies of the monomers (2 % substitutions), so that interior
lanes carry nearly the row end's value."""
import contextlib
import os

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

import cases
import sd_oracle
from stringdecomposer_b200 import Decomposer, SdError

SD_ERR_UNSUPPORTED, SD_ERR_INTERNAL = 3, 5
ENV_KEYS = ("SD_LAT", "SD_LAT_WARPS", "SD_GROUP_SLOTS", "SD_GROUP_GSLOTS", "SD_STREAM_SYMBOLS", "SD_FORCE_S32", "SD_GEOM",
            "SD_EMU_BAD_JUMP_ROW", "SD_WAVE_BYTES", "SD_PROFILE", "SD_DUMP_TABLES")
_AL = np.frombuffer(b"ACGT", dtype=np.uint8)


@contextlib.contextmanager
def environ(env):
    old = {k: os.environ.get(k) for k in ENV_KEYS}
    for k in ENV_KEYS:
        os.environ.pop(k, None)
    os.environ.update(env)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def random_monomers(rng, lengths):
    return [_AL[rng.integers(0, 4, n)].tobytes().decode() for n in lengths]


def mutate(rng, s, rate):
    a = np.frombuffer(s.encode(), dtype=np.uint8).copy()
    hit = rng.random(len(a)) < rate
    a[hit] = _AL[rng.integers(0, 4, int(hit.sum()))]
    return a.tobytes().decode()


def copies(rng, mons, n, rate=0.02):
    """n bp of substituted copies of randomly picked monomers, a quarter of them reverse-complemented"""
    out, total = [], 0
    while total < n:
        m = mons[int(rng.integers(0, len(mons)))]
        if rng.random() < 0.25:
            m = sd_oracle.rows_of([m])[1]
        out.append(mutate(rng, m, rate))
        total += len(m)
    return "".join(out)[:n]


def decompose(flavour, mons, segs, scoring, env=None, ed_thr=-1):
    """-> (records of each segment as oracle tuples, stats)"""
    with environ(env or {}):
        d = Decomposer(mons, *scoring, devices=[0] if flavour == "cuda" else None, flavour=flavour)
        try:
            if ed_thr >= 0:
                d.set_ed_thr(ed_thr)
            recs, off = d.decompose(segs)
            stats = d.stats()
        finally:
            d.close()
    got = [[(int(r["row"]), int(r["start"]), int(r["end"]), float(r["score"])) for r in recs[off[j]:off[j + 1]]]
           for j in range(len(segs))]
    return got, stats


def check(flavour, mons, segs, scoring, env=None, ed_thr=-1):
    got, stats = decompose(flavour, mons, segs, scoring, env, ed_thr)
    for j, s in enumerate(segs):
        want = sd_oracle.align_segment(s, mons, scoring, ed_thr)
        assert got[j] == want, (len(mons), [len(m) for m in mons], scoring, env, ed_thr, j)
    return stats


def refused(flavour, mons, segs, scoring, env=None):
    with pytest.raises(SdError) as e:
        decompose(flavour, mons, segs, scoring, env)
    return e.value


def inf_ok(n, lmax, scoring):
    """plan.cpp: the INF-sentinel check and the exact-float check of make_plan"""
    ins, dl, mm, ma = scoring
    lo = n * max(abs(ins), abs(mm)) + 2 * lmax * abs(dl) + 2 * abs(mm) + abs(ma)
    hi = (n + lmax) * max(abs(ma), abs(mm), abs(ins), abs(dl))
    return lo < 999_000 and hi < (1 << 23)


def packed_ok(lmax, scoring):
    """plan.cpp: packed_range_ok (the s16x2 range proof)"""
    ins, dl, mm, ma = scoring
    if ins > 0 or dl > 0:
        return False
    D, I = -dl, -ins
    smax, smin = max(ma, mm), min(ma, mm)
    s2max, s2min = smax + I + D, smin + I + D
    L = max(lmax, 2)
    relmax = D * (L + 2) + I + max(smax, 0) + 2 * max(abs(s2min), abs(s2max)) + 4
    dmax = D * (L + 1) + I + max(abs(smax), abs(smin)) + 1
    pad = relmax + abs(s2min) + 4096 // 4 + 2
    return 4 * (pad + relmax + 2 * dmax) + 2 * 4096 + 64 <= 32767


# ---- the 32-bit column key: (L-1)*|del| across 2^18 up to the INF check's limit ---------------------------------------

SEG = 3000
LENGTHS = (300, 600, 1000, 1536)
# (L-1)*|del| targets: 2^17, 2^18 -/+ 2,000, 3 * 2^17, and the largest the INF check accepts (about 499,000).
# 3 * 2^18 lies beyond that limit for every L: it is checked to be refused.
TARGETS = ("2^17", "2^18-2000", "2^18+2000", "3*2^17", "max")


def deletion_for(L, target, n=SEG):
    if target == "max":
        d = 1
        while inf_ok(n, L, (-1, -(d + 1), -1, 1)):
            d += 1
        return -d
    v = {"2^17": 1 << 17, "2^18-2000": (1 << 18) - 2000, "2^18+2000": (1 << 18) + 2000, "3*2^17": 3 << 17}[target]
    return -max(1, round(v / (L - 1)))


def domain_inputs(L, target):
    rng = np.random.default_rng(L * 7 + TARGETS.index(target))
    mons = random_monomers(rng, [L, L])
    return mons, [copies(rng, mons, SEG)], (-1, deletion_for(L, target), -1, 1)


def sweeps(L):
    """(name, env, ed_thr) of every sweep that takes an L bp monomer pair in 32-bit lanes"""
    thr = max(4, L // 20)          # keeps the forward rows (2 % substitutions), drops the reverse complements
    out = [("planner", {}, -1), ("classic", {"SD_LAT": "0"}, -1), ("deferred", {"SD_LAT": "1"}, -1),
           ("group", {"SD_GROUP_SLOTS": "1"}, -1), ("streamed", {"SD_STREAM_SYMBOLS": "1"}, -1),
           ("ed_thr", {}, thr), ("ed_thr classic", {"SD_LAT": "0"}, thr), ("ed_thr deferred", {"SD_LAT": "1"}, thr)]
    return out


def run_domain(flavour, L, target):
    mons, segs, scoring = domain_inputs(L, target)
    assert inf_ok(SEG, L, scoring)
    ran = set()
    for name, env, thr in sweeps(L):
        if env.get("SD_LAT") == "1":
            # the deferred sweep's profile slices must fit shared memory: one warp per CTA where four do not
            try:
                decompose(flavour, mons, segs[:1], scoring, env)
            except SdError as e:
                assert e.status == SD_ERR_UNSUPPORTED and "deferred-jump" in str(e), e
                env = dict(env, SD_LAT_WARPS="1")
        stats = check(flavour, mons, segs, scoring, env, thr)
        assert stats["packed"] == 0, (name, stats)
        if env.get("SD_LAT") == "1":
            assert stats["lat"] == 1, (name, stats)
        if env.get("SD_LAT") == "0" or "SD_GROUP_SLOTS" in env:
            assert stats["lat"] == 0, (name, stats)
        if "SD_STREAM_SYMBOLS" in env:
            assert stats["stream"] == 1, (name, stats)
        ran.add((stats["lat"], stats["NG"] > 1 and stats["lat"] == 0))
    assert {(1, False), (0, False), (0, True)} <= ran, ran          # deferred, classic and group sweeps all ran


@pytest.mark.parametrize("target", TARGETS)
@pytest.mark.parametrize("L", LENGTHS)
def test_s32_column_key_against_oracle(L, target):
    run_domain(cases.EMU_LIB, L, target)


@pytest.mark.gpu
@pytest.mark.parametrize("target", TARGETS)
@pytest.mark.parametrize("L", LENGTHS)
def test_gpu_s32_column_key_against_oracle(L, target):
    run_domain("cuda", L, target)


@pytest.mark.parametrize("L", LENGTHS)
def test_deletion_beyond_the_inf_limit_is_refused(L):
    mons, segs, _ = domain_inputs(L, "max")
    dl = -round((3 << 18) / (L - 1))
    e = refused(cases.EMU_LIB, mons, segs, (-1, dl, -1, 1))
    assert e.status == SD_ERR_UNSUPPORTED and "INF sentinel" in str(e)
    e = refused(cases.EMU_LIB, mons, segs, (-1, deletion_for(L, "max") - 1, -1, 1))
    assert e.status == SD_ERR_UNSUPPORTED and "INF sentinel" in str(e)


# ---- the packed / 32-bit boundary -------------------------------------------------------------------------------------

BOUNDARY_SCORINGS = ((-1, -1, -1, 1), (-2, -2, -3, 1), (-1, -3, -1, 2))


def last_packed(scoring):
    L = 2
    while packed_ok(L + 1, scoring):
        L += 1
    return L


def boundary_inputs(scoring, L):
    rng = np.random.default_rng(L)
    mons = random_monomers(rng, [L, L - 1, max(1, L // 3)])
    return mons, [copies(rng, mons, SEG), copies(rng, mons, 1200)]


def run_boundary(flavour, scoring):
    L = last_packed(scoring)
    assert L + 1 <= 1536, L
    for length, packed in ((L, 1), (L + 1, 0)):
        mons, segs = boundary_inputs(scoring, length)
        for env in ({}, {"SD_LAT": "0"}, {"SD_LAT": "1", "SD_LAT_WARPS": "1"}):
            assert check(flavour, mons, segs, scoring, env)["packed"] == packed, (length, env)
        if packed:
            assert check(flavour, mons, segs, scoring, {"SD_FORCE_S32": "1"})["packed"] == 0


@pytest.mark.parametrize("scoring", BOUNDARY_SCORINGS, ids=str)
def test_packed_boundary_against_oracle(scoring):
    # the emulator traps any 16-bit overflow: the last packed length is where the range proof is tight
    run_boundary(cases.EMU_LIB, scoring)


@pytest.mark.gpu
@pytest.mark.parametrize("scoring", BOUNDARY_SCORINGS, ids=str)
def test_gpu_packed_boundary_against_oracle(scoring):
    run_boundary("cuda", scoring)


def test_packed_boundary_formula_matches_the_planner():
    for scoring in BOUNDARY_SCORINGS:
        L = last_packed(scoring)
        for length, packed in ((L, 1), (L + 1, 0)):
            _, stats = decompose(cases.EMU_LIB, ["A" * length], ["A" * 50], scoring)
            assert stats["packed"] == packed, (scoring, length)


# ---- rebases: the reference base Bref moves hundreds of times per segment ----------------------------------------------

REBASE_CASES = [
    ((-30, -1, -1, 1), 10),          # 4*30 per column: a rebase every ~34 columns, ten 3 kb segments
    ((-300, -1, -1, 1), 1),          # a rebase every ~3 columns
    ((2, -1, -3, 1), 3),             # positive insertion score: 32-bit lanes
    ((-1, 2, -2, 1), 3),             # positive deletion score: 32-bit lanes, endadd > 0
    ((3, 3, -2, 4), 3),
]


def run_rebases(flavour, scoring, nseg):
    rng = np.random.default_rng(abs(scoring[0]) * 100 + abs(scoring[1]))
    mons = random_monomers(rng, [171, 160, 120])
    segs = [copies(rng, mons, SEG) for _ in range(nseg)]
    assert inf_ok(SEG, 171, scoring)
    for env in ({}, {"SD_LAT": "0"}, {"SD_LAT": "1"}, {"SD_GROUP_SLOTS": "1"}):
        stats = check(flavour, mons, segs, scoring, env)
        if scoring[0] > 0 or scoring[1] > 0:
            assert stats["packed"] == 0


@pytest.mark.parametrize("scoring,nseg", REBASE_CASES, ids=str)
def test_rebases_against_oracle(scoring, nseg):
    run_rebases(cases.EMU_LIB, scoring, nseg)


@pytest.mark.gpu
@pytest.mark.parametrize("scoring,nseg", REBASE_CASES, ids=str)
def test_gpu_rebases_against_oracle(scoring, nseg):
    run_rebases("cuda", scoring, nseg)


# ---- the row bits of the key: 2,048 monomers, 4,096 rows --------------------------------------------------------------

def row_limit_inputs(dup):
    """2,048 distinct 9 bp monomers; dup: the last one repeats the one before it (rows 2046/2047 and 4094/4095 tie,
    the lower row wins).  The segment is made of copies of the reverse complements of the last three monomers."""
    rng = np.random.default_rng(2048 + dup)
    seen, mons = set(), []
    while len(mons) < 2048:
        m = random_monomers(rng, [9])[0]
        if m not in seen and sd_oracle.rows_of([m])[1] not in seen:
            seen.update((m, sd_oracle.rows_of([m])[1]))
            mons.append(m)
    if dup:
        mons[-1] = mons[-2]
    rcs = sd_oracle.rows_of(mons[-3:])[3:]
    seg = "".join(rcs[int(rng.integers(0, 3))] for _ in range(70))
    return mons, [seg]


def run_row_limit(flavour):
    for dup in (0, 1):
        mons, segs = row_limit_inputs(dup)
        got, stats = decompose(flavour, mons, segs, (-1, -1, -1, 1))
        assert got[0] == sd_oracle.align_segment(segs[0], mons)
        assert stats["NG"] > 1 and stats["lat"] == 0, stats            # the group sweep
        rows = {r[0] for r in got[0]}
        assert (4095 in rows) != bool(dup) and 4094 in rows, rows          # key row bits 0 and 1
    e = refused(flavour, mons + ["ACGTACGTA"], segs, (-1, -1, -1, 1))
    assert e.status == SD_ERR_UNSUPPORTED and "2048 monomers" in str(e)


def test_row_limit_against_oracle():
    run_row_limit(cases.EMU_LIB)


@pytest.mark.gpu
def test_gpu_row_limit_against_oracle():
    run_row_limit("cuda")


# ---- record scores near the exact float bound (2^23) ------------------------------------------------------------------

def float_bound_inputs():
    rng = np.random.default_rng(23)
    mons = random_monomers(rng, [171, 171])
    n = 2800
    match = (1 << 23) // (n + 171)                  # (n + Lmax) * match just under 2^23
    assert (n + 171) * match < (1 << 23) <= (n + 172) * match
    seg = copies(rng, mons, n + 1)
    return mons, seg, (-1, -1, -1, match)


def run_float_bound(flavour):
    mons, seg, scoring = float_bound_inputs()
    for env in ({}, {"SD_LAT": "0"}, {"SD_LAT": "1"}):
        got, stats = decompose(flavour, mons, [seg[:-1]], scoring, env)
        want = sd_oracle.align_segment(seg[:-1], mons, scoring)
        assert got[0] == want and stats["packed"] == 0, env
        assert all(r[3] == int(r[3]) for r in got[0])
        assert sum(int(r[3]) for r in got[0]) > (1 << 22)              # the segment's total score is near the bound
    e = refused(flavour, mons, [seg], scoring)
    assert e.status == SD_ERR_UNSUPPORTED and "exact float range" in str(e)


def test_float_bound_against_oracle():
    run_float_bound(cases.EMU_LIB)


@pytest.mark.gpu
def test_gpu_float_bound_against_oracle():
    run_float_bound("cuda")


# ---- the traceback refuses a jump row outside the monomer set ---------------------------------------------------------

def test_traceback_reports_a_bad_jump_row():
    # the emulator corrupts the row of the last jump of the first segment; the traceback must report it as an internal
    # error instead of indexing the row table with it
    rng = np.random.default_rng(5)
    mons = random_monomers(rng, [171, 150])
    segs = [copies(rng, mons, 1000)]
    e = refused(cases.EMU_LIB, mons, segs, (-1, -1, -1, 1), {"SD_EMU_BAD_JUMP_ROW": "1"})
    assert e.status == SD_ERR_INTERNAL and "row outside the monomer set" in str(e)
    assert check(cases.EMU_LIB, mons, segs, (-1, -1, -1, 1))["segments"] == 1


# ---- property: long monomers and large deletion penalties -------------------------------------------------------------

@st.composite
def domain_problems(draw, max_len):
    seed = draw(st.integers(0, 2**32 - 1))
    lengths = draw(st.lists(st.integers(1, max_len), min_size=1, max_size=3))
    n = draw(st.integers(1, 1500))
    ins = draw(st.integers(-20, 2))
    mm = draw(st.integers(-20, 0))
    match = draw(st.integers(0, 20))
    dl = -draw(st.integers(-3, 500))
    scoring = (ins, dl, mm, match)
    if not inf_ok(n, max(lengths), scoring):          # the largest |del| the INF check accepts
        room = 999_000 - 1 - n * max(abs(ins), abs(mm)) - 2 * abs(mm) - abs(match)
        scoring = (ins, -min(-dl, room // (2 * max(lengths))), mm, match)
    env = draw(st.sampled_from([{}, {"SD_LAT": "0"}, {"SD_LAT": "1", "SD_LAT_WARPS": "1"}, {"SD_GROUP_SLOTS": "1"},
                                {"SD_STREAM_SYMBOLS": "1"}]))
    ed_thr = draw(st.sampled_from([-1, -1, -1, 10, 60]))
    return seed, lengths, n, scoring, env, ed_thr


def run_problem(flavour, problem):
    seed, lengths, n, scoring, env, ed_thr = problem
    assert inf_ok(n, max(lengths), scoring)
    rng = np.random.default_rng(seed)
    mons = random_monomers(rng, lengths)
    segs = [copies(rng, mons, n), copies(rng, mons, max(1, n // 3), rate=0.05)]
    check(flavour, mons, segs, scoring, env, ed_thr)


@settings(max_examples=40, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(domain_problems(1000))
def test_emulated_score_domain_property(problem):
    run_problem(cases.EMU_LIB, problem)


@pytest.mark.gpu
@settings(max_examples=25, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(domain_problems(600))
def test_cuda_score_domain_property(problem):
    run_problem("cuda", problem)
