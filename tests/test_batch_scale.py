"""The CUDA backend at batch scale, and the --ed_thr filter kernels, against the int64 oracle.

Several paths of the backend only run beyond the sizes of the other tests:
- the gather kernel's chunk loop, for waves of more than 1,024 segments;
- ramped waves (a device share of at least 4,096 segments starts with a small wave and doubles), whose classic sweeps
  alternate between two streams;
- group-sweep slot groups that sweep several segment blocks one after the other (SD_GROUP_GSLOTS caps their number);
- the --ed_thr filter with more than 128 rows (a second row block of hw_distance_rows_kernel) and more than 256 rows
  (the strided loop of filter_rank_kernel), every word count NB of the Myers/Hyyro kernel and the generic kernel.

Every case compares the records of every segment with sd_oracle.align_segment, and checks through stats() or the
SD_PROFILE line that it reached its path.  The CPU variants run the emulator on the smallest instance of each case
(it has one wave slot and runs one unit per segment, so it neither ramps nor loops over blocks).  The filter kernels
are also run on their own (tests/cuda/filter_probe.cu) and their tables compared with the oracle's textbook DP."""
import concurrent.futures
import multiprocessing
import os
import re
import subprocess

import numpy as np
import pytest

import cases
import sd_oracle
from stringdecomposer_b200 import SdError, synth
from test_score_domain import copies, decompose, random_monomers

DEFAULT = (-1, -1, -1, 1)
SD_ERR_UNSUPPORTED = 3
CSRC = os.path.join(cases.ROOT, "stringdecomposer_b200", "csrc")


# ---- the oracle, in a process pool -------------------------------------------------------------------------------------

def _align(args):
    return sd_oracle.align_segment(*args)


def _hw(args):
    return [sd_oracle.lib().sdo_hw_distance(r.encode(), len(r), args[1].encode(), len(args[1])) for r in args[0]]


def _filter(args):
    return sd_oracle.filter_rows(*args)


@pytest.fixture(scope="module")
def oracle():
    sd_oracle.lib()
    with concurrent.futures.ProcessPoolExecutor(os.cpu_count() or 1, mp_context=multiprocessing.get_context("fork")) as pool:
        yield pool


def want(pool, segs, mons, scoring=DEFAULT, ed_thr=-1):
    # longest first, so that a long segment does not start last
    order = sorted(range(len(segs)), key=lambda j: -len(segs[j]))
    res = pool.map(_align, [(segs[j], mons, scoring, ed_thr) for j in order], chunksize=1 if len(segs) < 100 else 8)
    out = [None] * len(segs)
    for j, r in zip(order, res):
        out[j] = r
    return out


def check(flavour, mons, segs, expect, env=None, ed_thr=-1, scoring=DEFAULT):
    got, stats = decompose(flavour, mons, segs, scoring, env, ed_thr)
    bad = [j for j in range(len(segs)) if got[j] != expect[j]]
    assert not bad, ("%d of %d segments differ from the oracle, first %d (%d bp)" % (len(bad), len(segs), bad[0], len(segs[bad[0]])),
                     env, ed_thr, stats)
    return stats


def mixed_segments(rng, mons, nseg, longest):
    """nseg mutated copies of the monomers, lengths 1 .. longest (both present), shuffled"""
    lens = [1, longest] + [int(x) for x in rng.integers(1, longest + 1, nseg - 2)]
    rng.shuffle(lens)
    return [copies(rng, mons, n) for n in lens]


def launches_per_wave(ed_thr):
    # sweep, traceback, gather; the filter adds hw_distance and filter_rank.  The emulator counts sweep and traceback.
    return 3 + (2 if ed_thr >= 0 else 0)


# ---- one wave of 1,025 to 4,095 segments: the gather kernel's chunk loop ------------------------------------------------

def one_wave_inputs(nseg):
    rng = np.random.default_rng(nseg)
    mons = random_monomers(rng, [int(x) for x in rng.integers(20, 191, 12)])     # C*T >= 190 for SD_GEOM=19,10,3
    return mons, mixed_segments(rng, mons, nseg, 600)


ONE_WAVE_ENVS = [("planner", {}, None), ("classic 24,8,4", {"SD_LAT": "0", "SD_GEOM": "24,8,4"}, (24, 8, 4)),
                 ("classic 19,10,3", {"SD_LAT": "0", "SD_GEOM": "19,10,3"}, (19, 10, 3)), ("deferred", {"SD_LAT": "1"}, None),
                 ("streamed", {"SD_STREAM_SYMBOLS": "1"}, None), ("s32", {"SD_FORCE_S32": "1"}, None)]


def run_one_wave(flavour, pool, nseg, envs):
    mons, segs = one_wave_inputs(nseg)
    expect = want(pool, segs, mons)
    for name, env, geom in envs:
        stats = check(flavour, mons, segs, expect, env)
        if flavour == "cuda":
            assert stats["launches"] == 3, (name, stats)            # one wave of nseg > 1024 segments
        if geom:
            assert (stats["C"], stats["T"], stats["NS"], stats["NG"], stats["lat"]) == geom + (1, 0), (name, stats)
        if name == "deferred":
            assert stats["lat"] == 1, stats
        if name == "streamed":
            assert stats["stream"] == 1, stats
        if name == "s32":
            assert stats["packed"] == 0, stats


def test_one_wave_against_oracle(oracle):
    run_one_wave(cases.EMU_LIB, oracle, 1025, ONE_WAVE_ENVS[1:2])


@pytest.mark.gpu
@pytest.mark.parametrize("nseg", [1500, 3000])
def test_gpu_one_wave_against_oracle(oracle, nseg):
    run_one_wave("cuda", oracle, nseg, ONE_WAVE_ENVS)


# ---- ramped waves (CUDA only: two wave slots) ---------------------------------------------------------------------------

def ramp_waves(share, NS):
    """pipeline.cpp: Engine::decompose's wave loop for a share of one device, without a memory budget"""
    ramp = max(1024, share // 16) // NS * NS if share >= 4096 else share
    s0, n = 0, 0
    while s0 < share:
        hi = min(share, s0 + max(ramp, NS))
        if share - hi < ramp // 2:
            hi = share
        n, s0 = n + 1, hi
        if ramp < share:
            ramp *= 2
    return n


def ramp_inputs(nseg):
    rng = np.random.default_rng(nseg + 1)
    mons = random_monomers(rng, [int(x) for x in rng.integers(20, 61, 4)])
    return mons, mixed_segments(rng, mons, nseg, 200)


@pytest.mark.gpu
@pytest.mark.parametrize("nseg", [4096, 9001])
def test_gpu_ramped_waves_against_oracle(oracle, nseg):
    mons, segs = ramp_inputs(nseg)
    thr = 6
    for ed_thr in (-1, thr):
        expect = want(oracle, segs, mons, ed_thr=ed_thr)
        stats = check("cuda", mons, segs, expect, {}, ed_thr)
        assert stats["NG"] == 1 and stats["lat"] == 0, stats             # classic sweeps: two streams
        waves = ramp_waves(nseg, stats["NS"])
        assert waves >= 3 and stats["launches"] == waves * launches_per_wave(ed_thr), (waves, stats)
        if nseg < 5000:
            continue
        # A budget of about a third of the batch per wave slot (SD_WAVE_BYTES is shared by the two slots) cuts the last
        # ramped wave.  The batch's device bytes are estimated as sweep_kernels.cu: wave_bytes counts them: backpointers
        # and J (sweep_store_bytes), a 32-byte record and one symbol byte per column, and with the filter 12 bytes per
        # segment and row.  Only the intent is asserted: more waves than the ramp alone, but not a flood of small ones.
        total = stats["sweep_store_bytes"] + 33 * stats["columns"] + (12 * nseg * 2 * len(mons) if ed_thr >= 0 else 0)
        stats = check("cuda", mons, segs, expect, {"SD_WAVE_BYTES": str(2 * total // 3)}, ed_thr)
        assert waves < stats["launches"] // launches_per_wave(ed_thr) <= 2 * waves, (waves, stats)


# ---- group sweep: slot groups that sweep several segment blocks ---------------------------------------------------------

def group_inputs(natural):
    """25 segments (13 blocks at NS = 2, the last one with a missing segment) of 1 .. 600 bp; blocks pair a 1 bp segment
    with a 600 bp one.  natural: 65 monomers of 128/129 bp, which need three CTAs per segment without an override."""
    rng = np.random.default_rng(25 + natural)
    mons = random_monomers(rng, [128 + (j & 1) for j in range(65)] if natural else [int(x) for x in rng.integers(20, 121, 8)])
    lens = [int(x) for x in rng.integers(1, 601, 25)]
    lens[0:4] = [1, 600, 600, 1]
    lens[-1] = 1
    return mons, [copies(rng, mons, n) for n in lens]


GSLOTS = (1, 2, 3)


def run_group_blocks(flavour, pool, capfd, natural, gslots):
    mons, segs = group_inputs(natural)
    thr = 40 if natural else 10
    for ed_thr in (-1, thr):
        expect = want(pool, segs, mons, ed_thr=ed_thr)
        for s32 in (0, 1):
            env = {} if natural else {"SD_GROUP_SLOTS": "1"}
            env = dict(env, SD_PROFILE="1", SD_LAT="0")
            if s32:
                env["SD_FORCE_S32"] = "1"
            for n in gslots:
                capfd.readouterr()
                stats = check(flavour, mons, segs, expect, dict(env, SD_GROUP_GSLOTS=str(n)), ed_thr)
                assert stats["NG"] > 1 and stats["lat"] == 0 and stats["NS"] == 2 and stats["packed"] == 1 - s32, stats
                if flavour == "cuda":
                    got = [int(x) for x in re.findall(r"(\d+) group slot\(s\)", capfd.readouterr().err)]
                    assert got == [n], (n, got)                  # 13 blocks over n slot groups


def test_group_blocks_against_oracle(oracle, capfd):
    run_group_blocks(cases.EMU_LIB, oracle, capfd, 0, GSLOTS[:1])


@pytest.mark.gpu
@pytest.mark.parametrize("natural", [0, 1])
def test_gpu_group_blocks_against_oracle(oracle, capfd, natural):
    run_group_blocks("cuda", oracle, capfd, natural, GSLOTS)


@pytest.mark.gpu
def test_gpu_group_blocks_without_override(oracle, capfd):
    # 160 config-5 monomers with SD_GROUP_SLOTS=1: 40 CTAs per segment.  600 segments are 300 blocks at NS = 2, more
    # than the 4,736 CTAs (32 per SM) a B200 can hold at once make slot groups of 40.
    _, _, _, mons = synth.config5(n_monomers=160, total=5000)
    rng = np.random.default_rng(160)
    segs = mixed_segments(rng, mons, 600, 100)
    expect = want(oracle, segs, mons)
    capfd.readouterr()
    stats = check("cuda", mons, segs, expect, {"SD_GROUP_SLOTS": "1", "SD_PROFILE": "1"})
    assert stats["NG"] == 40 and stats["lat"] == 0 and stats["launches"] == 3, stats
    got = [int(x) for x in re.findall(r"(\d+) group slot\(s\)", capfd.readouterr().err)]
    nblocks = -(-len(segs) // stats["NS"])
    assert len(got) == 1 and 0 < got[0] < nblocks, (got, nblocks, stats)


# ---- --ed_thr with many rows --------------------------------------------------------------------------------------------

def many_rows_sets(full):
    """(name, monomers, segments): word edges of the Myers/Hyyro kernel (NB = 1..4 and the generic kernel) and 130 to 4,094
    rows; the tile edges of the segment text (4,095 / 4,096 / 4,097 / 8,193 bp) go with the cheaper sets"""
    rng = np.random.default_rng(4094)
    tiles = [4095, 4096, 4097, 8193] if full else []
    out = []
    for M, lens, seglens in ((65, (64, 65), [1, 300] + tiles), (65, (128, 129), [700] + tiles[:2]), (130, (192, 193), [1, 500]),
                             (65, (256, 257), [600, 257]), (300, (20, 64), [1, 64, 600])):
        mons = random_monomers(rng, [lens[j % 2] for j in range(M)] if lens[1] - lens[0] == 1 else
                               [int(x) for x in rng.integers(lens[0], lens[1] + 1, M)])
        out.append(("%d x %s" % (M, lens), mons, [copies(rng, mons, n) for n in seglens]))
    seen, m9 = set(), []
    while len(m9) < 2047:
        m = random_monomers(rng, [9])[0]
        if m not in seen:
            seen.add(m)
            m9.append(m)
    out.append(("2047 x 9", m9, [copies(rng, m9[:40], n) for n in (1, 9, 630)]))
    return out if full else out[:1]


def thresholds(seg, mons):
    """0, large, and exactly the distance of one row (the median one): off by one, that row moves in or out"""
    d = _hw((sd_oracle.rows_of(mons), seg))
    return (0, max(d), sorted(d)[len(d) // 2])


def run_many_rows(flavour, pool, full):
    ran = set()
    for name, mons, segs in many_rows_sets(full):
        for thr in thresholds(segs[-1], mons):
            expect = want(pool, segs, mons, ed_thr=thr)
            for env in ({"SD_LAT": "0"}, {"SD_LAT": "1"}, {"SD_GROUP_SLOTS": "1"}):
                try:
                    stats = check(flavour, mons, segs, expect, env, thr)
                except SdError as e:
                    # the deferred sweep holds at most 32 warps per segment
                    assert env.get("SD_LAT") == "1" and e.status == SD_ERR_UNSUPPORTED and "deferred-jump" in str(e), (name, e)
                    continue
                if flavour == "cuda":
                    assert stats["launches"] == launches_per_wave(thr), stats
                ran.add("deferred" if stats["lat"] else "group" if stats["NG"] > 1 else "classic")
    assert ran == {"classic", "deferred", "group"}, ran


def test_many_rows_against_oracle(oracle):
    run_many_rows(cases.EMU_LIB, oracle, False)


@pytest.mark.gpu
def test_gpu_many_rows_against_oracle(oracle):
    run_many_rows("cuda", oracle, True)


# ---- the filter kernels on their own ------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def filter_probe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("filter_probe") / "filter_probe")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")          # the same override as csrc/Makefile
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-I", CSRC,
                    "-o", out, os.path.join(cases.HERE, "cuda", "filter_probe.cu")], check=True)
    return out


def run_probe(probe, tmp_path, segs, rows, ed_thr, kjbase):
    nseg, R = len(segs), len(rows)
    so = np.zeros(nseg + 1, np.int64)
    so[1:] = np.cumsum([len(s) for s in segs])
    ro = np.zeros(R + 1, np.int32)
    ro[1:] = np.cumsum([len(r) for r in rows])
    src, dst = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    with open(src, "wb") as f:
        f.write(np.array([nseg, R, ed_thr, kjbase is not None], np.int32).tobytes() + so.tobytes() + ro.tobytes())
        f.write("".join(segs).encode() + "".join(rows).encode())
        if kjbase is not None:
            f.write(np.ascontiguousarray(kjbase, np.int32).tobytes())
    subprocess.run([probe, src, dst], check=True)
    out = np.fromfile(dst, np.int32)
    np_ = nseg * R
    assert out.size == 3 * np_ + 5 * nseg
    return (out[:np_].reshape(nseg, R), out[np_:2 * np_].reshape(nseg, R), out[2 * np_:3 * np_].reshape(nseg, R),
            out[3 * np_:].reshape(nseg, 5))


def _rand(rng, n, alphabet=b"ACGT"):
    return np.frombuffer(alphabet, np.uint8)[rng.integers(0, len(alphabet), n)].tobytes().decode()


EDGE_LENGTHS = (1, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 256, 257)


def filter_cases():
    """(name, rows, segments, kjbase or None); every case is run with ed_thr 0, a large one and one row's distance"""
    rng = np.random.default_rng(7)
    out = []
    for nb, top in ((1, 64), (2, 128), (3, 192), (4, 256), ("generic", 257)):
        # rows of every edge length up to 64*NB (the longest sets NB), several of each
        lens = [n for n in EDGE_LENGTHS if n <= top] * 3
        rows = [_rand(rng, n) for n in lens]
        segs = [_rand(rng, 1), _rand(rng, 63), copies(rng, rows, 4095), copies(rng, rows, 4097, rate=0.1)]
        out.append(("NB %s" % nb, rows, segs, rng.integers(-1 << 20, 1 << 20, (len(rows), 5))))
    for R in (1, 127, 128, 129, 256, 257):
        rows = [_rand(rng, int(n)) for n in rng.integers(1, 65, R)]
        segs = [copies(rng, rows, n) for n in (1, 63, 600, 4096)]
        out.append(("R %d" % R, rows, segs, rng.integers(-1 << 20, 1 << 20, (R, 5))))
    rows = [_rand(rng, int(n)) for n in rng.integers(1, 13, 4094)]
    out.append(("R 4094", rows, [copies(rng, rows[:50], n) for n in (1, 300)], rng.integers(-1 << 20, 1 << 20, (4094, 5))))
    rows = [_rand(rng, int(n)) for n in rng.integers(20, 41, 129)]
    out.append(("8193 and 100 kb", rows, [copies(rng, rows, 8193, rate=0.05), copies(rng, rows, 100_000, rate=0.05)], None))
    # N in rows and segments (N matches N only)
    rows = [_rand(rng, int(n), b"ACGTN") for n in rng.integers(1, 130, 140)]
    out.append(("N", rows, [_rand(rng, 2000, b"ACGTN"), _rand(rng, 5, b"NNNNA"), copies(rng, rows, 700)],
                rng.integers(-1 << 20, 1 << 20, (140, 5))))
    # ties: every row is at the same distance (no C in the rows, none but C in the segments), ranks follow the row index
    rows = [_rand(rng, 70, b"AGT") for _ in range(300)]
    out.append(("ties", rows, ["C" * 500, "C" * 4097], rng.integers(-1 << 20, 1 << 20, (300, 5))))
    return out


def expected_tables(dist, ed_thr, kjbase):
    """-> rank_of_row, row_of_rank, seg_kj of one segment from its oracle distances (main.cpp:141-147)"""
    R = len(dist)
    order = [r for _, r in sorted((d, r) for r, d in enumerate(dist))]
    rank = [-1] * R
    r2r = [-1] * R
    for pos, r in enumerate(order):
        if pos == 0 or dist[r] <= ed_thr:
            rank[r], r2r[pos] = pos, r
    kj = [-(1 << 31)] * 5
    if kjbase is not None:
        kj = [max(int(kjbase[r][sym]) - rank[r] for r in range(R) if rank[r] >= 0) for sym in range(5)]
    return rank, r2r, kj


@pytest.mark.gpu
def test_gpu_filter_kernels_against_oracle(oracle, filter_probe, tmp_path):
    for name, rows, segs, kjbase in filter_cases():
        dist = np.array(list(oracle.map(_hw, [(rows, s) for s in segs])), np.int32)
        for thr in (0, int(dist.max()), int(np.sort(dist[-1])[len(rows) // 2])):
            d, rank, r2r, kj = run_probe(filter_probe, tmp_path, segs, rows, thr, kjbase)
            assert (d == dist).all(), (name, [(s, r) for s, r in zip(*np.nonzero(d != dist))][:5])
            kept = list(oracle.map(_filter, [(s, rows, thr) for s in segs]))
            for s in range(len(segs)):
                want_rank, want_r2r, want_kj = expected_tables(list(dist[s]), thr, kjbase)
                assert list(rank[s]) == want_rank, (name, thr, s)
                assert list(r2r[s]) == want_r2r, (name, thr, s)
                assert list(r2r[s][:len(kept[s])]) == kept[s] and (r2r[s][len(kept[s]):] == -1).all(), (name, thr, s)
                assert list(kj[s]) == want_kj, (name, thr, s)
        if name == "ties":
            assert (dist == 70).all() and list(r2r[0]) == list(range(len(rows)))
