"""Property-based parity (hypothesis): random monomer sets, segments and scorings -- the kernel algebra (host emulator on
CPU, CUDA on the B200) must reproduce the oracle's records exactly, whatever the launch geometry."""
import os

import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

import cases
import sd_oracle
from stringdecomposer_b200 import Decomposer


# SD_HYP_SCALE=<k> multiplies the number of examples of every property test (soak runs; 1 in the regular suites)
SCALE = max(1, int(os.environ.get("SD_HYP_SCALE", "1") or 1))


def seq(alphabet, lo, hi):
    return st.text(alphabet=alphabet, min_size=lo, max_size=hi)


@st.composite
def problems(draw):
    alphabet = draw(st.sampled_from(["A", "AC", "ACG", "ACGT", "ACGTN"]))
    monomers = draw(st.lists(seq(alphabet, 1, 70), min_size=1, max_size=6))
    if draw(st.booleans()) and len(monomers) > 1:
        monomers[-1] = monomers[0]                       # duplicate rows: arg-max ties (main.cpp:212, :230-236)
    segments = draw(st.lists(seq(alphabet, 1, 260), min_size=1, max_size=4))
    scoring = draw(st.sampled_from([(-1, -1, -1, 1), (-2, -2, -3, 1), (-3, -2, -4, 2), (0, -1, -1, 1), (-1, 0, -1, 1),
                                    (-1, -1, -1, 5), (-7, -25, -3, 2), (1, -1, -1, 1), (-1, -2, 0, 0)]))
    geom = draw(st.sampled_from(["", "8,32,1", "12,16,2", "19,10,1", "24,8,3", "16,4,2", "8,8,5", "48,2,1"]))
    group = draw(st.sampled_from(["", "", "1", "4"]))
    # deferred-jump sweep: "" = the planner decides, "0" = classic, "C,T,warps-per-CTA" = forced
    lat = draw(st.sampled_from(["", "0", "6,32,4", "6,32,1", "12,16,2", "24,8,1", "12,32,1"]))
    return monomers, segments, scoring, geom, group, lat


def problem_env(problem):
    """the test overrides of a problem (an empty value: unset)"""
    monomers, segments, scoring, geom, group, lat = problem
    lmax = max(len(m) for m in monomers)
    if geom:
        c, t, _ = map(int, geom.split(","))
        if c * t < lmax:
            geom = ""
    env = {"SD_GEOM": geom, "SD_GROUP_SLOTS": group, "SD_LAT": lat, "SD_LAT_WARPS": ""}
    if "," in lat:
        c, t, w = lat.split(",")
        env.update({"SD_LAT": "1", "SD_GEOM": "%s,%s,1" % (c, t), "SD_LAT_WARPS": w, "SD_GROUP_SLOTS": ""})
    return env


def run(flavour, problem):
    monomers, segments, scoring, geom, group, lat = problem
    env = problem_env(problem)
    for k, v in env.items():
        if v:
            os.environ[k] = v
        else:
            os.environ.pop(k, None)
    try:
        d = Decomposer(monomers, *scoring, flavour=flavour)
        recs, off = d.decompose(segments)
        d.close()
    finally:
        for k in env:
            os.environ.pop(k, None)
    for j, s in enumerate(segments):
        want = sd_oracle.align_segment(s, monomers, scoring)
        got = [(int(r["row"]), int(r["start"]), int(r["end"]), float(r["score"])) for r in recs[off[j]:off[j + 1]]]
        assert got == want, (monomers, s, scoring, geom, group, lat)


@settings(max_examples=120 * SCALE, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(problems())
def test_emulated_kernels_match_oracle(problem):
    run(cases.EMU_LIB, problem)


@pytest.mark.gpu
@settings(max_examples=60 * SCALE, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(problems())
def test_cuda_kernels_match_oracle(problem):
    run("cuda", problem)


# ---- the rescoring stage: sd_identity / sd_convert against the oracle on random inputs ---------------------------------
@st.composite
def rescoring_problems(draw):
    alphabet = draw(st.sampled_from(["A", "AC", "ACGT", "ACGTN"]))
    monomers = draw(st.lists(seq(alphabet, 1, 60), min_size=1, max_size=4))
    names = ["m%d" % i for i in range(len(monomers))]
    if draw(st.booleans()) and len(names) > 1:
        names[-1] = names[0]                              # repeated name: the `scores` dict of main.py:123 collapses it
    reads = draw(st.lists(seq(alphabet, 1, 200), min_size=1, max_size=3))
    lines = []
    for _ in range(draw(st.integers(0, 8))):
        r = draw(st.integers(0, len(reads) - 1))
        a = draw(st.integers(0, len(reads[r]) + 3))
        b = draw(st.integers(a - 1, a + 80))
        m = draw(st.sampled_from(names)) + draw(st.sampled_from(["", "'"]))
        lines.append("r%d\t%s\t%d\t%d\t1.0\t0\t0\n" % (r, m, a, b))
    return list(zip(names, monomers)), {"r%d" % i: s for i, s in enumerate(reads)}, "".join(lines), \
        draw(st.sampled_from([0, 50, 100])), draw(st.booleans())


def run_rescoring(flavour, problem, tmp):
    import sd_convert_oracle as CO
    from stringdecomposer_b200 import convert as cv
    monomers, reads, raw, thr, light = problem
    want, want_alt = CO.final_tsv(raw, reads, monomers, thr, light)
    rc = cv.add_rc_monomers(monomers)
    for fn in (cv.convert_tsv, cv.convert_tsv_native):
        out = os.path.join(tmp, "o.tsv")
        fn(raw, reads, rc, out, thr, light, flavour=flavour)
        assert open(out).read() == want and open(out[:-4] + "_alt.tsv").read() == want_alt, (problem, fn.__name__)


@settings(max_examples=60 * SCALE, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large,
                                                                 HealthCheck.function_scoped_fixture])
@given(rescoring_problems())
def test_emulated_rescoring_matches_oracle(tmp_path, problem):
    run_rescoring(cases.EMU_LIB, problem, str(tmp_path))


@pytest.mark.gpu
@settings(max_examples=40 * SCALE, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large,
                                                                 HealthCheck.function_scoped_fixture])
@given(rescoring_problems())
def test_cuda_rescoring_matches_oracle(tmp_path, problem):
    run_rescoring("cuda", problem, str(tmp_path))
