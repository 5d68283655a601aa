"""GPU parity tests (run on the B200 box with -m gpu).  Everything goes through the C ABI (libsd_b200.so) or the
drop-in dp binary; the oracle is only the checker."""
import hashlib
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import cases
import sd_oracle
from stringdecomposer_b200 import synth, Decomposer, decompose_reads, device_count, int_peak
from stringdecomposer_b200.hostpipe import segment_reads

pytestmark = pytest.mark.gpu


def as_tuples(recs):
    return [(int(r["row"]), int(r["start"]), int(r["end"]), float(r["score"])) for r in recs]


def test_native_library_is_the_one_running():
    # in a fresh interpreter: the CPU tests of a whole-suite run load the host emulator into this process
    code = textwrap.dedent("""
        import sys
        sys.path.insert(0, %r)
        from stringdecomposer_b200 import Decomposer
        d = Decomposer(["ACGTACGTAC"], devices=[0])
        recs, off = d.decompose(["ACGTACGTACGGTACGTAC"])
        st = d.stats()
        assert st["launches"] >= 2 and st["n_devices"] == 1 and st["cells"] == 19 * 20
        maps = open("/proc/self/maps").read()
        assert "libsd_b200.so" in maps and "libsd_emu.so" not in maps
    """) % cases.ROOT
    p = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert p.returncode == 0, p.stderr.decode()[-2000:]


@pytest.mark.parametrize("scoring,fixture", [(None, "config1_raw_default.tsv"), ((-2, -2, -3, 1), "config1_raw_s-2-2-3+1.tsv")])
def test_config1_golden_through_dp_binary(scoring, fixture):
    st, out, err = sd_oracle.run_cli(cases.DP_CUDA, os.path.join(cases.GOLDEN, "config1_read.fa"),
                                     os.path.join(cases.GOLDEN, "DXZ1_star_monomers.fa"), scoring=scoring)
    assert st == 0, err
    assert out == open(os.path.join(cases.GOLDEN, fixture), "rb").read()
    if scoring is None:
        got = ["\t".join(ln.split("\t")[:4]) for ln in out.decode().splitlines()]
        assert got == open(os.path.join(cases.GOLDEN, "config1_cols1-4.tsv")).read().splitlines()


def _plain_argv(case):
    """argv that sd_run_files can be given directly (three, seven or eight integer arguments after the two paths)"""
    if case.get("argv_raw") is not None or len(case["argv_tail"]) not in (3, 7, 8):
        return False
    try:
        [int(x) for x in case["argv_tail"]]
    except ValueError:
        return False
    return True


_ALL_CASES = cases.load_cases()
# A `dp` process pays a CUDA context per case (0.25 s on some boxes, 3 s and more on others: profiles/r02_startup.txt),
# so the full list of reference-generated cases runs inside this process through sd_run_files -- the function dp_main.cpp
# hands its argv to -- with stdout, stderr and status compared, and the binary itself runs every case that is about argv
# handling, every failing case and every tenth of the rest.
_BINARY_CASES = [c for i, c in enumerate(_ALL_CASES)
                 if not _plain_argv(c) or i % 10 == 0 or c["name"].startswith(("argc", "ed_thr_0", "scoring_0")) or c["status"] != 0]


@pytest.mark.parametrize("case", _BINARY_CASES, ids=lambda c: c["name"])
def test_edge_cases_through_dp_binary(case):
    cases.check_case(cases.DP_CUDA, case)


@pytest.mark.parametrize("case", [c for c in _ALL_CASES if _plain_argv(c)], ids=lambda c: c["name"])
def test_edge_cases_through_sd_run_files(case):
    cases.check_case_inproc(case, check_stderr=True)


@pytest.mark.parametrize("geom", ["8,32,1", "16,16,1", "24,8,1", "24,8,2", "32,8,1", "48,4,2", "48,4,3", "12,16,1", "20,10,1", "20,10,2", "12,16,1", "19,10,1", "19,10,3"])
@pytest.mark.parametrize("force32", ["0", "1"])
def test_every_geometry_and_both_widths(geom, force32):
    picked = [c for c in cases.load_cases() if c["name"] in ("multi_read", "scoring_-3_-2_-4_2", "N_in_monomer", "dup_monomers_rev",
                                                             "len_5501_default")]
    for case in picked:
        cases.check_case_inproc(case, env={"SD_GEOM": geom, "SD_FORCE_S32": force32})


@pytest.mark.parametrize("geom", ["8,1,4", "8,2,2", "16,1,1", "24,1,2", "32,2,1", "48,1,1", "8,4,3", "48,32,1"])
def test_small_and_large_slots(geom):
    C, T, _ = map(int, geom.split(","))
    for seed in range(4):
        rn, rr, mn, mm = synth.random_case(300 + seed, mono_len=(1, min(C * T, 700)), read_len=(1, 500), n_monomers=(1, 5))
        want = sd_oracle.decompose_reads(rn, rr, mn, mm, part_size=150, overlap=40)
        os.environ["SD_GEOM"] = geom
        try:
            got = decompose_reads(rn, rr, mn, mm, part_size=150, overlap=40)
        finally:
            del os.environ["SD_GEOM"]
        assert got == want


@pytest.mark.parametrize("seed", range(24))
def test_fuzz_against_oracle(seed):
    al = ["A", "AT", "AC", "ACGT", "ACGTN"][seed % 5]
    scorings = [(-1, -1, -1, 1), (-2, -2, -3, 1), (-3, -2, -4, 2), (0, -1, -1, 1), (-1, 0, -2, 2), (-4, -1, -1, 1), (-1, -4, -1, 2),
                (-9, -30, -9, 2), (1, -1, -1, 1)]
    sc = scorings[seed % len(scorings)]
    part, ov = [(50, 10), (120, 30), (300, 100), (5000, 500)][seed % 4]
    rn, rr, mn, mm = synth.random_case(5000 + seed, alphabet=al, mono_len=(1, 200), read_len=(1, 1500))
    want = sd_oracle.decompose_reads(rn, rr, mn, mm, part_size=part, overlap=ov, scoring=sc)
    got = decompose_reads(rn, rr, mn, mm, part_size=part, overlap=ov, scoring=sc)
    assert got == want


def test_segment_records_and_staged_api():
    names, mons = synth.load_dxz1()
    arr = synth.hor_array(mons, 20000, 0.04, seed=21)
    segs, _ = segment_reads([arr], 1500, 300)
    d = Decomposer(mons, devices=[0])
    recs, off = d.decompose(segs)
    for j in (0, 3, len(segs) - 1):
        assert as_tuples(recs[off[j]:off[j + 1]]) == sd_oracle.align_segment(segs[j], mons)
    d.stage(segs)
    ms = d.run_staged()
    ms2 = d.run_staged()
    r2, o2 = d.fetch_staged()
    assert ms > 0 and ms2 > 0 and (r2 == recs).all() and (o2 == off).all()
    d.close()


@pytest.mark.parametrize("chunk,wave", [("1", ""), ("5000", "300000"), ("100000", "")])
def test_streamed_chunks_and_waves_do_not_change_the_result(chunk, wave):
    picked = [c for c in cases.load_cases() if c["name"] in ("multi_read", "len_10000_default", "part700_ov50", "blank_lines", "ed_thr_12")]
    env = {"SD_CHUNK_BASES": chunk}
    if wave:
        env["SD_WAVE_BYTES"] = wave
    for case in picked:
        cases.check_case_inproc(case, env=env, check_stderr=True)
    cases.check_case(cases.DP_CUDA, picked[0], env=env)             # and once through the binary


def test_waves_do_not_change_the_result():
    rn, rr, mn, mm = synth.random_case(77, read_len=(2000, 3000), n_reads=(3, 3))
    want = sd_oracle.decompose_reads(rn, rr, mn, mm, part_size=300, overlap=100)
    os.environ["SD_WAVE_BYTES"] = "300000"
    try:
        got = decompose_reads(rn, rr, mn, mm, part_size=300, overlap=100)
    finally:
        del os.environ["SD_WAVE_BYTES"]
    assert got == want


def test_score_width_switch_on_device():
    names, mons = synth.load_dxz1()
    seg = synth.hor_array(mons, 3000, 0.05, seed=9)
    for sc, packed in (((-1, -1, -1, 1), 1), ((-2, -2, -3, 1), 1), ((-9, -30, -9, 2), 0), ((1, -1, -1, 1), 0)):
        d = Decomposer(mons, *sc, devices=[0])
        recs, off = d.decompose([seg])
        assert d.stats()["packed"] == packed
        assert as_tuples(recs) == sd_oracle.align_segment(seg, mons, sc)
        d.close()


def test_config2_full_size_properties_and_sampled_parity():
    # BASELINE config 2 at full size: 2 Mb array, 400 segments.  Size-independent properties on every segment,
    # oracle parity on a sample (the oracle needs ~0.2 s and 180 MB per segment).
    rn, reads, mn, mons = synth.config2()
    segs, where = segment_reads(reads, 5000, 500)
    assert len(segs) == 400
    d = Decomposer(mons, devices=[0])
    recs, off = d.decompose(segs)
    recs2, off2 = d.decompose(segs)
    assert (recs == recs2).all() and (off == off2).all()              # deterministic
    R = 2 * len(mons)
    for j, s in enumerate(segs):
        r = recs[off[j]:off[j + 1]]
        assert len(r) > 0 and r["start"][0] == 0 and r["end"][-1] == len(s) - 1
        assert (r["start"][1:] == r["end"][:-1] + 1).all()           # alignments tile the segment
        assert (r["row"] >= 0).all() and (r["row"] < R).all()
        assert (r["start"] <= r["end"]).all()
    for j in (0, 57, 199, 311, 399):
        want = sd_oracle.align_segment(segs[j], mons)
        assert as_tuples(recs[off[j]:off[j + 1]]) == want
        # the segment scores telescope to the best final score (main.cpp:253-257)
        assert sum(w[3] for w in want) == float(recs[off[j]:off[j + 1]]["score"].sum())
    st = d.stats()
    assert st["cells"] == 2 * sum(len(s) for s in segs) * 2 * sum(len(m) for m in mons)
    d.close()


def test_config2_full_output_identical_to_the_reference_binary(tmp_path):
    # BASELINE config 2 in full through the dp binary, against what the unmodified reference prints for it
    # (tests/golden/make_golden_full_runs.py: its size and MD5, a sample of its lines, its stderr)
    with open(os.path.join(cases.GOLDEN, "config2_raw_digest.json")) as f:
        ref = json.load(f)
    rp, mp = cases.write_config2(tmp_path)
    ours = subprocess.run([cases.DP_CUDA, rp, mp, str(os.cpu_count() or 1), "5000", "500"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert ours.returncode == 0
    lines = ours.stdout.decode().splitlines(True)
    for i, want in ref["sample"]:
        assert i < len(lines) and lines[i] == want, "raw TSV line %d differs from the reference" % i
    assert len(ours.stdout) == ref["bytes"] and len(lines) == ref["lines"] > 11000
    assert hashlib.md5(ours.stdout).hexdigest() == ref["md5"]
    assert [ln for ln in ours.stderr.decode().splitlines() if not ln.startswith("[sd_b200]")] == ref["stderr"]


def test_config4_custom_scoring_sample():
    rn, reads, mn, mons = synth.config4(n_reads=6, read_len=15000)
    sc = (-2, -2, -3, 1)
    want = sd_oracle.decompose_reads(rn, reads, mn, mons, scoring=sc)
    assert decompose_reads(rn, reads, mn, mons, scoring=sc) == want
    # part 20000 leaves the proven s16 range for this scoring (SURVEY App. A.6) -> s32 sweep, same answer as the oracle
    want = sd_oracle.decompose_reads(rn[:2], reads[:2], mn, mons, part_size=20000, overlap=500, scoring=sc)
    assert decompose_reads(rn[:2], reads[:2], mn, mons, part_size=20000, overlap=500, scoring=sc) == want


def test_config3_noisy_reads_sample():
    rn, reads, mn, mons = synth.config3(n_reads=3, read_len=30000)
    want = sd_oracle.decompose_reads(rn, reads, mn, mons)
    assert decompose_reads(rn, reads, mn, mons) == want


@pytest.mark.parametrize("ngpu", [2, 4, 8])
def test_multi_gpu_output_identical(ngpu):
    # BASELINE config 2 (one 2 Mb array, 400 segments) split over the GPUs of the box by Engine::split: records of
    # 1 / 2 / 4 / 8 devices must be identical, whatever sweep the planner picks for the smaller per-GPU shares
    if device_count() < ngpu:
        pytest.skip("needs >= %d GPUs" % ngpu)
    rn, reads, mn, mons = synth.config2()
    segs, _ = segment_reads(reads, 5000, 500)
    d1 = Decomposer(mons, devices=[0])
    r1, o1 = d1.decompose(segs)
    d1.close()
    dn = Decomposer(mons, devices=list(range(ngpu)))
    rn_, on_ = dn.decompose(segs)
    st = dn.stats()
    dn.stage(segs)
    dn.run_staged()
    rs, os_ = dn.fetch_staged()
    dn.close()
    assert st["n_devices"] == ngpu and sum(st["dev_segments"]) == len(segs) and min(st["dev_segments"]) > 0
    assert (rn_ == r1).all() and (on_ == o1).all()
    assert (rs == r1).all() and (os_ == o1).all()
    # and through the drop-in binary: SD_DEVICES=all, whole raw TSV
    rn3, reads3, mn3, mons3 = synth.config3(n_reads=4, read_len=30000)
    one = decompose_reads(rn3, reads3, mn3, mons3, devices=[0])
    allg = decompose_reads(rn3, reads3, mn3, mons3, devices=list(range(ngpu)))
    assert one == allg
    # and the streamed dp binary itself with SD_DEVICES (chunks small enough that several are in flight)
    picked = [c for c in cases.load_cases() if c["name"] in ("multi_read", "len_10000_default")]
    for case in picked:
        cases.check_case(cases.DP_CUDA, case, env={"SD_DEVICES": str(ngpu), "SD_CHUNK_BASES": "4000"})


LAT_SUBSET = ("multi_read", "scoring_-3_-2_-4_2", "N_in_monomer", "dup_monomers_rev", "len_5501_default", "short_monomers", "N_in_read")


@pytest.mark.parametrize("lat", ["0", "1"])
def test_edge_cases_with_the_sweep_forced(lat):
    # the planner picks the deferred-jump sweep for small batches; force both sweeps over a spread of the golden cases
    names = {c["name"] for c in cases.load_cases()}
    extra = ("ed_thr_0", "ed_thr_12", "ed_thr_dups", "ed_thr_short_monomers", "ed_thr_fuzz_00_AT", "ed_thr_fuzz_02_ACGT", "ed_thr_fuzz_03_ACGTN",
             "tiny_alphabet_ties", "poly_A", "len1_monomer_only", "scoring_-6_-6_-6_1", "scoring_-1_0_-1_1")
    picked = [c for c in cases.load_cases() if c["name"] in LAT_SUBSET + extra or c["name"].startswith("fuzz_0")]
    assert len(picked) >= 25 and set(LAT_SUBSET + extra) <= names
    for case in picked:
        cases.check_case_inproc(case, env={"SD_LAT": lat}, check_stderr=True)


@pytest.mark.parametrize("geom,warps", [("6,32,1", "4"), ("6,32,1", "1"), ("6,32,1", "2"), ("12,16,1", "3"), ("12,16,1", "1"), ("24,8,1", "0"),
                                        ("24,8,1", "1"), ("12,32,1", "2"), ("24,16,1", "1"), ("24,32,1", "2"), ("48,32,1", "1")])
@pytest.mark.parametrize("force32", ["0", "1"])
def test_deferred_jump_sweep_every_geometry(geom, warps, force32):
    # cluster shapes from one CTA per segment down to one warp per CTA (up to 8 CTAs exchanging keys through DSMEM)
    picked = [c for c in cases.load_cases() if c["name"] in ("multi_read", "scoring_-3_-2_-4_2", "N_in_monomer", "dup_monomers_rev")]
    for case in picked:
        cases.check_case_inproc(case, env={"SD_LAT": "1", "SD_GEOM": geom, "SD_LAT_WARPS": warps, "SD_FORCE_S32": force32})


def test_deferred_jump_sweep_config1_and_config2_sample():
    # config 1 in full (19 segments: the planner's own choice must be the deferred-jump sweep) and 40 segments of config 2
    names, mons = synth.load_dxz1()
    read = open(os.path.join(cases.GOLDEN, "config1_read.fa")).read().split("\n", 1)[1].replace("\n", "")
    segs, _ = segment_reads([read], 5000, 500)
    d = Decomposer(mons, devices=[0])
    recs, off = d.decompose(segs)
    assert d.stats()["lat"] == 1
    d.close()
    os.environ["SD_LAT"] = "0"
    try:
        d0 = Decomposer(mons, devices=[0])
        r0, o0 = d0.decompose(segs)
        assert d0.stats()["lat"] == 0
        d0.close()
    finally:
        del os.environ["SD_LAT"]
    assert (recs == r0).all() and (off == o0).all()
    rn, reads, mn, mons2 = synth.config2()
    segs2, _ = segment_reads(reads, 5000, 500)
    for env in ({"SD_LAT": "1"}, {"SD_LAT": "1", "SD_GEOM": "12,16,1"}, {"SD_LAT": "1", "SD_GEOM": "24,8,1"}, {"SD_LAT": "1", "SD_GEOM": "6,32,1", "SD_LAT_WARPS": "2"}):
        os.environ.update(env)
        try:
            d = Decomposer(mons2, devices=[0])
            recs, off = d.decompose(segs2[100:140])
            d.close()
        finally:
            for k in env:
                del os.environ[k]
        for j in (0, 17, 39):
            assert as_tuples(recs[off[j]:off[j + 1]]) == sd_oracle.align_segment(segs2[100 + j], mons2)


def test_int_peak_probe():
    alu, both, mhz = int_peak(0)
    assert 5e12 < alu < 4e13 and both >= alu * 0.9 and 500 < mhz < 2500


@pytest.mark.parametrize("sg", ["1", "4", "8"])
def test_group_mode_forced_on_small_sets(sg):
    picked = [c for c in cases.load_cases() if c["name"] in ("multi_read", "dup_monomers_rev", "short_monomers", "N_in_monomer", "len_5501_default")]
    for case in picked:
        cases.check_case_inproc(case, env={"SD_GROUP_SLOTS": sg})
    cases.check_case_inproc(picked[0], env={"SD_GROUP_SLOTS": sg, "SD_FORCE_S32": "1"})
    st, out, err = sd_oracle.run_cli(cases.DP_CUDA, os.path.join(cases.GOLDEN, "config1_read.fa"), os.path.join(cases.GOLDEN, "DXZ1_star_monomers.fa"))
    assert st == 0


def test_config5_large_monomer_set_sample():
    # BASELINE config 5 (large monomer set): 160 monomers cannot live in one CTA -> group sweep.  The reference needs
    # n * sum(L) * 8 B per segment, so parity is checked on a bounded sample (part 2000).
    rn, reads, mn, mons = synth.config5(n_monomers=160, total=60_000)
    reads = [r[:9000] for r in reads[:2]]
    want = sd_oracle.decompose_reads(rn[:2], reads, mn, mons, part_size=2000, overlap=300, threads=4)
    got = decompose_reads(rn[:2], reads, mn, mons, part_size=2000, overlap=300)
    assert got == want


def test_config5_full_monomer_set_against_the_reference_binary():
    # BASELINE config 5 at its defining scale: 1,000 monomers -> 2,000 DP rows, sum(L) = 342 kb, which the planner spreads
    # over 32 partner CTAs per segment (group sweep).  The reference needs n * sum(L) * 8 B per segment in flight
    # (5.5 GB for a 2,000-column segment), so parity is checked on two 2,000-column segments plus a short tail, against
    # the raw TSV the unmodified reference binary prints for them (tests/golden/make_golden_full_runs.py).
    rn, (read,), mn, mons = cases.config5_sample()
    with open(os.path.join(cases.GOLDEN, "config5_1000_monomers_raw.tsv"), newline="") as f:
        want = f.read()
    d = Decomposer(mons, devices=[0])
    segs, _ = segment_reads([read], 1700, 300)
    assert [len(x) for x in segs] == [2000, 2000, 300]
    d.decompose(segs)
    st = d.stats()
    d.close()
    assert st["NG"] >= 16 and st["lat"] == 0          # the many-CTA group geometry of the real config 5
    got = decompose_reads(rn[:1], [read], mn, mons, part_size=1700, overlap=300)
    assert got == want and got.count("\n") > 15



def test_pinned_host_buffer_through_the_c_abi():
    # sd_host_alloc: text in page-locked memory -> same records as from pageable memory
    from stringdecomposer_b200._lib import HostBuffer
    _, segs, _, mons = synth.random_case(12, n_reads=(3, 3))
    dec = Decomposer(mons)
    a = dec.decompose(segs)
    b = dec.decompose(HostBuffer.pack(segs))
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all()
    dec.close()
