"""Helpers shared by the test modules: golden-case loading and running dp-compatible binaries."""
import json
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
DP_CUDA = os.path.join(ROOT, "stringdecomposer_b200", "build", "bin", "dp")
EMU_DIR = os.environ.get("SD_EMU_DIR") or os.path.join(HERE, "emu", "_build")     # override: a sanitizer build of the emulator
DP_EMU = os.path.join(EMU_DIR, "dp_emu")
EMU_LIB = os.path.join(EMU_DIR, "libsd_emu.so")
DP_ORACLE = os.path.join(ROOT, "oracle", "_build", "oracle_dp")
DP_REF = os.path.join(ROOT, "oracle", "_ref", "dp")


def load_cases():
    with open(os.path.join(GOLDEN, "edge_cases.json")) as f:
        return json.load(f)["cases"]


def write_config2(directory):
    """BASELINE config 2 in full (one 2 Mb array, 80-column FASTA) and its 12 monomers -> (reads path, monomers path)."""
    from stringdecomposer_b200 import synth
    rn, reads, mn, mons = synth.config2()
    rp, mp = os.path.join(str(directory), "reads.fa"), os.path.join(str(directory), "monomers.fa")
    synth.write_fasta(rp, rn, reads, width=80)
    synth.write_fasta(mp, mn, mons)
    return rp, mp


def config5_sample():
    """BASELINE config 5's 1,000 monomers against the first 3,700 bp of one of its arrays -> (names, reads, names, monomers)."""
    from stringdecomposer_b200 import synth
    rn, reads, mn, mons = synth.config5(n_monomers=1000, total=40_000)
    return rn[:1], [reads[0][:3700]], mn, mons


def run_case(binary, case, env=None):
    """-> (status, stdout, stderr) of `binary` on a golden case, temp paths stripped from stderr."""
    e = dict(os.environ)
    e.update(env or {})
    with tempfile.TemporaryDirectory() as td:
        if case.get("argv_raw") is not None:
            p = subprocess.run([binary] + case["argv_raw"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=e)
        else:
            rp, mp = os.path.join(td, "reads.fa"), os.path.join(td, "monomers.fa")
            open(rp, "w", newline="").write(case["reads_fa"])
            open(mp, "w", newline="").write(case["monomers_fa"])
            p = subprocess.run([binary, rp, mp] + case["argv_tail"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=td, env=e)
        return p.returncode, p.stdout.decode(), p.stderr.decode().replace(td + "/", "")


def check_case(binary, case, env=None, check_stderr=True):
    st, out, err = run_case(binary, case, env)
    assert st == case["status"], "%s: status %d != %d\n%s" % (case["name"], st, case["status"], err[-400:])
    assert out == case["stdout"], "%s: raw TSV differs from the reference" % case["name"]
    if check_stderr:
        keep = [ln for ln in err.splitlines() if not ln.startswith("[sd_b200]")]
        assert keep == case["stderr"].splitlines(), "%s: stderr differs:\n%s\n--- expected\n%s" % (case["name"], err, case["stderr"])


def check_case_inproc(case, env=None, flavour="cuda", check_stderr=False):
    """The same check through sd_run_files inside this process (no CUDA start-up per case): argv is interpreted the way
    csrc/dp_main.cpp does it (scores only with nine user arguments, ed_thr only with ten, main.cpp:381-391)."""
    from stringdecomposer_b200 import _lib
    tail = case["argv_tail"]
    assert case.get("argv_raw") is None and len(tail) >= 3
    threads, part, overlap = int(tail[0]), int(tail[1]), int(tail[2])
    scoring, ed_thr = (-1, -1, -1, 1), -1
    if len(tail) == 7:
        scoring = tuple(int(x) for x in tail[3:7])
    if len(tail) == 8:
        ed_thr = int(tail[7])
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        with tempfile.TemporaryDirectory() as td:
            rp, mp = os.path.join(td, "reads.fa"), os.path.join(td, "monomers.fa")
            open(rp, "w", newline="").write(case["reads_fa"])
            open(mp, "w", newline="").write(case["monomers_fa"])
            with open(os.path.join(td, "out"), "w+") as fo, open(os.path.join(td, "err"), "w+") as fe:
                st = _lib.run_files(rp, mp, threads, part, overlap, scoring, ed_thr, out_fd=fo.fileno(), err_fd=fe.fileno(), flavour=flavour)
                fo.seek(0); fe.seek(0)
                out, err = fo.read(), fe.read().replace(td + "/", "")
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    assert st == case["status"], "%s: status %d != %d\n%s" % (case["name"], st, case["status"], err[-400:])
    assert out == case["stdout"], "%s: raw TSV differs from the reference" % case["name"]
    if check_stderr:
        keep = [ln for ln in err.splitlines() if not ln.startswith("[sd_b200]")]
        assert keep == case["stderr"].splitlines(), "%s: stderr differs" % case["name"]
