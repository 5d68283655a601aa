"""Long segments: a segment longer than what fits one CTA's shared memory is swept with the segment symbols streamed
from global memory (Geometry::stream) instead of being refused.  The CPU tests run the planner and the host pipeline
through the emulator and the C oracle; the streamed kernels themselves only run on the GPU (-m gpu)."""
import contextlib
import importlib.util
import json
import os
import subprocess

import pytest

import cases
import sd_oracle
from stringdecomposer_b200 import _lib, synth, Decomposer, SdError, device_count

_spec = importlib.util.spec_from_file_location("make_golden_plans", os.path.join(cases.GOLDEN, "make_golden_plans.py"))
golden_plans = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(golden_plans)

INF_MSG = "ERROR: scores can reach the reference's INF sentinel (-1000000): outside the supported domain"


@contextlib.contextmanager
def environ(env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def run(binary, reads, mons, part, extra=(), env=None):
    """-> (status, stdout, stderr) of a dp-compatible binary with the default scores and overlap 500."""
    e = dict(os.environ)
    e.update(env or {})
    cmd = [binary, reads, mons, "1", str(part), "500"] + [str(x) for x in extra]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=e)
    return p.returncode, p.stdout, p.stderr


def run_files_inproc(reads, mons, part, ed_thr=-1, tmp=None):
    with open(os.path.join(tmp, "o"), "w+b") as fo, open(os.path.join(tmp, "e"), "w+b") as fe:
        st = _lib.run_files(reads, mons, 1, part, 500, (-1, -1, -1, 1), ed_thr, out_fd=fo.fileno(), err_fd=fe.fileno())
        fo.seek(0)
        fe.seek(0)
        return st, fo.read(), fe.read()


@pytest.fixture(scope="module")
def emu_plan(tmp_path_factory):
    """make_plan of this checkout for a shape, without its segments (tests/emu/plan_probe.cpp)"""
    lib = golden_plans.load(golden_plans.build(str(tmp_path_factory.mktemp("plan_probe"))))
    return lambda mons, n, nseg=1: golden_plans.plan(lib, mons, n, nseg)


@pytest.fixture(scope="module")
def dxz1():
    names, mons = synth.load_dxz1()
    return names, mons, synth.hor_array(mons, 400_000, 0.02, seed=7)


@pytest.fixture(scope="module")
def inputs(tmp_path_factory, dxz1):
    """FASTA files of the reproduction: the 400 kb DXZ1 array, its first 250 kb, the 12 and the first 2 DXZ1 monomers."""
    names, mons, arr = dxz1
    d = tmp_path_factory.mktemp("long")
    p = {k: str(d / (k + ".fa")) for k in ("r400", "r250", "m12", "m2")}
    synth.write_fasta(p["r400"], ["array400"], [arr], width=80)
    synth.write_fasta(p["r250"], ["array250"], [arr[:250_000]], width=80)
    synth.write_fasta(p["m12"], names, mons)
    synth.write_fasta(p["m2"], names[:2], mons[:2])
    p["dir"] = str(d)
    return p


@pytest.fixture(scope="module")
def oracle_250(inputs):
    """oracle_dp on the 250 kb segment against 2 monomers (about 2 s and 1.4 GB of int64 table)"""
    return run(cases.DP_ORACLE, inputs["r250"], inputs["m2"], 250_000)


# ---- CPU: planner ---------------------------------------------------------------------------------------------------

def test_every_shape_that_planned_before_keeps_its_plan(emu_plan):
    # tests/golden/plans.json: the planner's choice for a grid of monomer sets x segment lengths x segment counts,
    # written before segments could be streamed
    gold = json.load(open(os.path.join(cases.GOLDEN, "plans.json")))
    sets = dict(golden_plans.monomer_sets())
    assert len(gold["plans"]) == len(sets) * len(golden_plans.SEG_LENS) * len(golden_plans.SEG_COUNTS)
    refused_before = 0
    for row in gold["plans"]:
        got = emu_plan(sets[row["set"]], row["seg_len"], row["nseg"])
        if "error" in row:
            refused_before += 1
            continue
        want = {k: row[k] for k in gold["fields"]}
        assert {k: got.get(k) for k in gold["fields"]} == want, row
        assert got["stream"] == 0, row
    assert refused_before < 10


@pytest.mark.parametrize("lat", ["0", "1"])
@pytest.mark.parametrize("s32", ["0", "1"])
def test_250kb_against_two_monomers_streams_and_matches_the_oracle(emu_plan, inputs, oracle_250, dxz1, lat, s32):
    env = {"SD_LAT": lat, "SD_FORCE_S32": s32}
    with environ(env):
        g = emu_plan(dxz1[1][:2], 250_000)
    assert g["stream"] == 1 and g["lat"] == int(lat) and g["packed"] == 1 - int(s32), g
    assert run(cases.DP_EMU, inputs["r250"], inputs["m2"], 250_000, env=env) == oracle_250
    assert oracle_250[0] == 0 and oracle_250[1].count(b"\n") > 1000


def test_160kb_against_the_dxz1_set_streams(emu_plan, dxz1):
    for lat in ("0", "-1"):
        with environ({"SD_LAT": lat}):
            g = emu_plan(dxz1[1], 160_000)
        assert g.get("stream") == 1, (lat, g)
    # a cluster of three CTAs splits the profile table: 160 kb of symbols still fit beside each slice
    with environ({"SD_LAT": "1"}):
        assert emu_plan(dxz1[1], 160_000)["stream"] == 0


def test_read_longer_than_a_chunk(inputs, oracle_250):
    # run_files plans for the longest segment of the whole file; a chunk then holds one segment larger than its nominal size
    assert run(cases.DP_EMU, inputs["r250"], inputs["m2"], 250_000, env={"SD_CHUNK_BASES": "20000"}) == oracle_250


def test_domain_edge(emu_plan, inputs, dxz1):
    # the reference's INF sentinel bounds the segment length: n + 2 * Lmax + 3 < 999000 with the default scores
    mons = dxz1[1][:2]
    edge = 999_000 - 2 * max(len(m) for m in mons) - 3 - 1
    assert emu_plan(mons, edge)["stream"] == 1
    assert "INF" in emu_plan(mons, edge + 1).get("error", "")
    arr = synth.hor_array(dxz1[1], edge + 1, 0.02, seed=13)
    inside, outside = os.path.join(inputs["dir"], "edge_in.fa"), os.path.join(inputs["dir"], "edge_out.fa")
    synth.write_fasta(inside, ["edge"], [arr[:edge]], width=80)
    synth.write_fasta(outside, ["edge"], [arr], width=80)
    st, out, err = run(cases.DP_EMU, inside, inputs["m2"], edge)
    assert st == 0 and out.count(b"\n") > 5000 and out.startswith(b"edge\t"), err[-300:]
    st, out, err = run(cases.DP_EMU, outside, inputs["m2"], edge + 1)
    assert st == 3 and out == b"" and err.decode().splitlines()[-1] == INF_MSG


def test_stream_override_sets_the_flag():
    names, mons = synth.load_dxz1()
    seg = synth.hor_array(mons, 3000, 0.02, seed=5)
    for env, want in (({}, 0), ({"SD_STREAM_SYMBOLS": "1"}, 1), ({"SD_STREAM_SYMBOLS": "1", "SD_LAT": "1"}, 1),
                      ({"SD_STREAM_SYMBOLS": "1", "SD_LAT": "0"}, 1), ({"SD_STREAM_SYMBOLS": "0"}, 0)):
        with environ(env):
            d = Decomposer(mons, flavour=cases.EMU_LIB)
            recs, off = d.decompose([seg])
            st = d.stats()
            d.close()
        assert st["stream"] == want, env
        assert [(int(r["row"]), int(r["start"]), int(r["end"]), float(r["score"])) for r in recs] == sd_oracle.align_segment(seg, mons)


@pytest.mark.parametrize("case", cases.load_cases(), ids=lambda c: c["name"])
def test_stream_override_keeps_the_edge_cases(case):
    cases.check_case(cases.DP_EMU, case, env={"SD_STREAM_SYMBOLS": "1"})


def test_a_wave_larger_than_the_device_is_refused():
    # 20 kb against 2,047 random 171 bp monomers: about 3.5 GB of backpointers for one segment, the emulator has 1 GiB
    import numpy as np
    rng = np.random.default_rng(2047)
    al = np.frombuffer(b"ACGT", dtype=np.uint8)
    mons = [al[rng.integers(0, 4, 171)].tobytes().decode() for _ in range(2047)]
    seg = al[rng.integers(0, 4, 20_000)].tobytes().decode()
    d = Decomposer(mons, flavour=cases.EMU_LIB)
    with pytest.raises(SdError) as e:
        d.decompose([seg])
    assert e.value.status == 3
    msg = str(e.value)
    assert "segment of 20000 bp needs" in msg and "bytes of device memory" in msg and "%d bytes are available" % (1 << 30) in msg
    need = int(msg.split("needs ")[1].split(" ")[0])
    assert need > 3 << 30
    st = d.stats()
    assert st["segments"] == 0 and st["launches"] == 0             # nothing ran, nothing was allocated
    d.close()


def test_wave_budget_override_stays_soft(dxz1):
    # a wave budget far below one segment still runs it, as a wave of one CTA
    mons = dxz1[1][:2]
    segs = [dxz1[2][:60_000], dxz1[2][100_000:130_000]]
    d = Decomposer(mons, flavour=cases.EMU_LIB)
    want = d.decompose(segs)
    d.close()
    with environ({"SD_WAVE_BYTES": "1000", "SD_STREAM_SYMBOLS": "1"}):
        d = Decomposer(mons, flavour=cases.EMU_LIB)
        got = d.decompose(segs)
        assert d.stats()["stream"] == 1
        d.close()
    assert (got[0] == want[0]).all() and (got[1] == want[1]).all()


def _cli_outputs(tmp, reads, mons, extra, flavour):
    from stringdecomposer_b200 import cli
    out = os.path.join(tmp, "_".join(extra).replace("-", "") or "default")
    assert cli.main([reads, mons, "-o", out] + extra, flavour=flavour) == 0
    names = ("final_decomposition_raw.tsv", "final_decomposition.tsv")
    return [open(os.path.join(out, n)).read() for n in names], open(os.path.join(out, "stringdecomposer.log")).read()


def _whole_reads_check(tmp, flavour, lens):
    names, mons = synth.load_dxz1()
    arr = synth.hor_array(mons, sum(lens), 0.03, seed=17)
    reads, o = [], 0
    for n in lens:
        reads.append(arr[o:o + n])
        o += n
    rp, mp = os.path.join(tmp, "reads.fa"), os.path.join(tmp, "mons.fa")
    synth.write_fasta(rp, ["r%d" % i for i in range(len(lens))], reads, width=60)
    synth.write_fasta(mp, names, mons)
    whole, log = _cli_outputs(tmp, rp, mp, ["--whole-reads"], flavour)
    fixed, _ = _cli_outputs(tmp, rp, mp, ["-b", str(max(lens))], flavour)
    assert whole == fixed
    assert "--whole-reads: segment size %d" % max(lens) in log


def test_whole_reads_cli(tmp_path):
    _whole_reads_check(str(tmp_path), cases.EMU_LIB, [7000, 12000, 3000])


# ---- GPU -------------------------------------------------------------------------------------------------------------

def _cuda_stats(mons, segs, env, ed_thr=-1):
    with environ(env):
        d = Decomposer(mons, devices=[0])
        if ed_thr >= 0:
            d.set_ed_thr(ed_thr)
        recs, off = d.decompose(segs)
        st = d.stats()
        d.close()
    return recs, off, st


@pytest.mark.gpu
@pytest.mark.parametrize("lat", ["0", "1"])
@pytest.mark.parametrize("s32", ["0", "1"])
def test_gpu_250kb_against_two_monomers_matches_the_oracle(inputs, oracle_250, dxz1, tmp_path, lat, s32):
    env = {"SD_LAT": lat, "SD_FORCE_S32": s32}
    assert run(cases.DP_CUDA, inputs["r250"], inputs["m2"], 250_000, env=env) == oracle_250
    with environ(env):
        assert run_files_inproc(inputs["r250"], inputs["m2"], 250_000, tmp=str(tmp_path)) == oracle_250
    _, _, st = _cuda_stats(dxz1[1][:2], [dxz1[2][:250_000]], env)
    assert st["stream"] == 1 and st["lat"] == int(lat) and st["packed"] == 1 - int(s32), st


@pytest.mark.gpu
@pytest.mark.parametrize("lat", ["0", "1"])
@pytest.mark.parametrize("ed_thr", [0, 20])
def test_gpu_250kb_with_the_ed_thr_filter(inputs, dxz1, tmp_path, lat, ed_thr):
    # ten arguments after the program name (argc == 11): the --ed_thr pre-filter walks the whole 250 kb text in tiles
    want = run(cases.DP_ORACLE, inputs["r250"], inputs["m2"], 250_000, extra=(-1, -1, -1, 1, ed_thr))
    assert want[0] == 0
    env = {"SD_LAT": lat}
    assert run(cases.DP_CUDA, inputs["r250"], inputs["m2"], 250_000, extra=(-1, -1, -1, 1, ed_thr), env=env) == want
    with environ(env):
        assert run_files_inproc(inputs["r250"], inputs["m2"], 250_000, ed_thr=ed_thr, tmp=str(tmp_path)) == want
    _, _, st = _cuda_stats(dxz1[1][:2], [dxz1[2][:250_000]], env, ed_thr=ed_thr)
    assert st["stream"] == 1


@pytest.mark.gpu
def test_gpu_dxz1_array_as_one_segment(inputs, dxz1):
    want = run(cases.DP_EMU, inputs["r400"], inputs["m12"], 400_000)
    assert want[0] == 0 and want[1].count(b"\n") > 2000
    for lat in ("-1", "0"):
        assert run(cases.DP_CUDA, inputs["r400"], inputs["m12"], 400_000, env={"SD_LAT": lat}) == want, lat
    _, _, st = _cuda_stats(dxz1[1], [dxz1[2]], {})
    assert st["stream"] == 1


@pytest.mark.gpu
def test_gpu_long_reads_file_against_two_monomers(inputs, dxz1):
    names, mons = dxz1[0], dxz1[1]
    lens = (150_000, 300_000, 990_000)
    arr = synth.hor_array(mons, sum(lens), 0.02, seed=11)
    reads = [arr[:lens[0]], arr[lens[0]:lens[0] + lens[1]], arr[lens[0] + lens[1]:]]
    rp = os.path.join(inputs["dir"], "long_reads.fa")
    synth.write_fasta(rp, ["read150k", "read300k", "read990k"], reads, width=80)
    want = run(cases.DP_EMU, rp, inputs["m2"], max(lens))
    assert want[0] == 0
    assert run(cases.DP_CUDA, rp, inputs["m2"], max(lens)) == want
    _, _, st = _cuda_stats(mons[:2], reads, {})
    assert st["stream"] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("case", cases.load_cases(), ids=lambda c: c["name"])
def test_gpu_stream_override_edge_cases(case):
    env = {"SD_STREAM_SYMBOLS": "1"}
    if case.get("argv_raw") is None and len(case["argv_tail"]) in (3, 7, 8) and all(x.lstrip("-").isdigit() for x in case["argv_tail"]):
        cases.check_case_inproc(case, env=env, check_stderr=True)
    else:
        cases.check_case(cases.DP_CUDA, case, env=env)


@pytest.mark.gpu
@pytest.mark.parametrize("scoring,fixture", [(None, "config1_raw_default.tsv"), ((-2, -2, -3, 1), "config1_raw_s-2-2-3+1.tsv")])
@pytest.mark.parametrize("lat", ["-1", "0"])
def test_gpu_stream_override_config1_golden(scoring, fixture, lat):
    e = dict(os.environ, SD_STREAM_SYMBOLS="1", SD_LAT=lat)
    cmd = [cases.DP_CUDA, os.path.join(cases.GOLDEN, "config1_read.fa"), os.path.join(cases.GOLDEN, "DXZ1_star_monomers.fa"), "1", "5000", "500"]
    p = subprocess.run(cmd + [str(x) for x in (scoring or ())], stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=e)
    assert p.returncode == 0, p.stderr
    assert p.stdout == open(os.path.join(cases.GOLDEN, fixture), "rb").read()
    read = open(os.path.join(cases.GOLDEN, "config1_read.fa")).read().split("\n", 1)[1].replace("\n", "")
    _, _, st = _cuda_stats(synth.load_dxz1()[1], [read[:5500], read[5000:10500]], {"SD_STREAM_SYMBOLS": "1", "SD_LAT": lat})
    assert st["stream"] == 1 and st["lat"] == (1 if lat == "-1" else 0)


GEOM_CASES = ("multi_read", "scoring_-3_-2_-4_2", "N_in_monomer", "dup_monomers_rev", "len_5501_default")


@pytest.mark.gpu
@pytest.mark.parametrize("geom", ["8,32,1", "16,16,1", "24,8,1", "24,8,2", "32,8,1", "48,4,2", "48,4,3", "12,16,1", "20,10,1", "20,10,2", "19,10,1", "19,10,3"])
@pytest.mark.parametrize("force32", ["0", "1"])
def test_gpu_stream_override_every_classic_geometry(geom, force32):
    env = {"SD_GEOM": geom, "SD_FORCE_S32": force32, "SD_STREAM_SYMBOLS": "1"}
    for case in [c for c in cases.load_cases() if c["name"] in GEOM_CASES]:
        cases.check_case_inproc(case, env=env)
    names, mons = synth.load_dxz1()
    if int(geom.split(",")[0]) * int(geom.split(",")[1]) >= max(len(m) for m in mons):
        _, _, st = _cuda_stats(mons, [synth.hor_array(mons, 2000, 0.02, seed=3)] * 3, dict(env, SD_LAT="0"))
        assert st["stream"] == 1 and st["lat"] == 0 and "%d,%d" % (st["C"], st["T"]) == ",".join(geom.split(",")[:2])


@pytest.mark.gpu
@pytest.mark.parametrize("geom,warps", [("6,32,1", "4"), ("6,32,1", "1"), ("6,32,1", "2"), ("12,16,1", "3"), ("12,16,1", "1"), ("24,8,1", "0"),
                                        ("24,8,1", "1"), ("12,32,1", "2"), ("24,16,1", "1"), ("24,32,1", "2"), ("48,32,1", "1")])
@pytest.mark.parametrize("force32", ["0", "1"])
def test_gpu_stream_override_every_deferred_jump_geometry(geom, warps, force32):
    env = {"SD_LAT": "1", "SD_GEOM": geom, "SD_LAT_WARPS": warps, "SD_FORCE_S32": force32, "SD_STREAM_SYMBOLS": "1"}
    for case in [c for c in cases.load_cases() if c["name"] in GEOM_CASES[:4]]:
        cases.check_case_inproc(case, env=env)
    names, mons = synth.load_dxz1()
    _, _, st = _cuda_stats(mons, [synth.hor_array(mons, 2000, 0.02, seed=3)], env)
    assert st["stream"] == 1 and st["lat"] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("chunk,wave", [("1", ""), ("5000", "300000"), ("100000", ""), ("", "300000")])
def test_gpu_stream_override_chunks_and_waves(chunk, wave):
    env = {"SD_STREAM_SYMBOLS": "1"}
    if chunk:
        env["SD_CHUNK_BASES"] = chunk
    if wave:
        env["SD_WAVE_BYTES"] = wave
    picked = [c for c in cases.load_cases() if c["name"] in ("multi_read", "len_10000_default", "part700_ov50", "blank_lines", "ed_thr_12")]
    for case in picked:
        cases.check_case_inproc(case, env=env, check_stderr=True)
    cases.check_case(cases.DP_CUDA, picked[0], env=env)


@pytest.mark.gpu
def test_gpu_one_long_segment_among_short_ones_on_two_devices(dxz1):
    if device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    names, mons, arr = dxz1
    segs = [arr[i * 5000:i * 5000 + 5500] for i in range(30)] + [arr[:300_000]] + [arr[200_000 + i * 5000:200_000 + i * 5000 + 5500] for i in range(30)]
    with environ({"SD_DEVICES": "1"}):
        r1, o1, _ = _cuda_stats(mons, segs, {})
    d = Decomposer(mons, devices=[0, 1])
    r2, o2 = d.decompose(segs)
    st = d.stats()
    d.close()
    assert st["n_devices"] == 2 and st["stream"] == 1
    assert (r1 == r2).all() and (o1 == o2).all()


@pytest.mark.gpu
def test_gpu_whole_reads_cli(tmp_path):
    _whole_reads_check(str(tmp_path), "cuda", [150_000, 20_000, 60_000])
