"""Identity rescoring row (SURVEY §8 f1/f4; stringdecomposer/main.py:29-184).

CPU part: the oracle (oracle/sd_identity_oracle.c, oracle/sd_convert_oracle.py) is pinned against the reference's own
edlib (committed golden pairs + the compiled library where it exists) and against all 12 columns of the reference's
golden final TSV; the host logic (convert.py, main.py, C-ABI argument checks) runs over the host emulator of the kernel.
GPU part (-m gpu): the CUDA kernel through the C ABI against the same golden data and the oracle."""
import json
import os
import random

import numpy as np
import pytest

import cases
import sd_convert_oracle as CO
import sd_oracle as O
import stringdecomposer_b200 as sd
from stringdecomposer_b200 import convert as cv
from stringdecomposer_b200 import cli as sdmain

G = cases.GOLDEN


def golden_pairs():
    with open(os.path.join(G, "nw_pairs.json")) as f:
        return json.load(f)["pairs"]


def rnd_seq(r, n, alpha="ACGT"):
    return "".join(r.choice(alpha) for _ in range(n))


def noisy(r, s, rate=0.15, alpha="ACGT"):
    out = []
    for c in s:
        x = r.random()
        if x < rate / 3:
            continue
        if x < rate:
            out.append(r.choice(alpha))
            if x < 2 * rate / 3:
                continue
        out.append(c)
    return "".join(out)


def check_against_oracle(res, qs, ts, pairs=None):
    idx = [(i, j) for i in range(len(qs)) for j in range(len(ts))] if pairs is None else list(zip(*pairs))
    assert len(idx) == len(res["matches"])
    for k, (i, j) in enumerate(idx):
        d, m, c = O.nw_path_counts(qs[i], ts[j])
        assert (res["distance"][k], res["matches"][k], res["columns"][k]) == (d, m, c), (qs[i], ts[j])


# ------------------------------------------------------------------------------------------ oracle pinning (CPU)
def test_oracle_equals_reference_edlib_golden_pairs():
    for p in golden_pairs():
        assert O.nw_path_counts(p["q"], p["t"]) == (p["distance"], p["matches"], p["columns"]), p["note"]


@pytest.mark.skipif(not os.path.exists(O.REF_EDLIB), reason="reference edlib not compiled here")
def test_oracle_equals_compiled_reference_edlib_fuzz():
    r = random.Random(5)
    for it in range(1500):
        alpha = r.choice(["A", "AC", "ACGT", "ACGTN"])
        q = rnd_seq(r, r.randint(1, 220 if it % 50 else 900), alpha)
        t = noisy(r, q, r.choice((0.05, 0.3)), alpha) or "A" if it % 3 else rnd_seq(r, r.randint(1, 220), alpha)
        assert O.nw_path_counts(q, t) == O.ref_nw_path_counts(q, t)


def test_oracle_empty_and_identity_rule():
    assert O.nw_path_counts("", "ACGT")[0] == -1 and O.identity("", "ACGT") == 0      # main.py:30-33
    assert O.identity("ACGT", "") == 0
    assert O.identity("ACGT", "ACGT") == 100
    assert O.identity("ACGT*", "ACGT") == 100                                           # main.py:38-41
    assert O.nw_uses_traceback(171, 171) and not O.nw_uses_traceback(2200, 1536)


def _golden_inputs():
    reads = dict(CO.fasta_records(os.path.join(G, "config1_read.fa")))
    mons = CO.fasta_records(os.path.join(G, "DXZ1_star_monomers.fa"))
    raw = open(os.path.join(G, "config1_raw_default.tsv")).read()
    return reads, mons, raw


def test_convert_oracle_reproduces_reference_golden_file_all_columns():
    reads, mons, raw = _golden_inputs()
    fin, alt = CO.final_tsv(raw, reads, mons, 0, light=False)
    assert fin == open(os.path.join(G, "config1_final_decomposition.tsv")).read()
    assert alt.count("\n") == 557 * 24


# ------------------------------------------------------------------------------------------ host logic over the emulator (CPU)
def test_library_exports_identity_symbol():
    import ctypes
    for path in (sd.library_path("cuda"), cases.EMU_LIB):
        assert hasattr(ctypes.CDLL(path), "sd_identity")


def test_identity_has_no_cpu_path():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(sd.SdError) as e:                    # the CUDA library refuses, it does not fall back
        sd.nw_identity(["ACGT"], ["ACGA"])
    assert e.value.status == 2 and "no CPU path" in str(e.value)


def test_emulated_kernel_equals_golden_pairs():
    ps = golden_pairs()
    qs, ts = [p["q"] for p in ps], [p["t"] for p in ps]
    k = np.arange(len(ps), dtype=np.int32)
    res = sd.nw_identity(qs, ts, pairs=(k, k), flavour=cases.EMU_LIB)
    assert list(res["distance"]) == [p["distance"] for p in ps]
    assert list(res["matches"]) == [p["matches"] for p in ps]
    assert list(res["columns"]) == [p["columns"] for p in ps]


@pytest.mark.parametrize("maxlen", [40, 100, 180, 250, 700])
def test_emulated_kernel_all_against_all_and_pair_list(maxlen):
    r = random.Random(maxlen)
    qs = [rnd_seq(r, r.randint(1, maxlen)) for _ in range(7)] + [""]
    ts = [noisy(r, q) or "A" for q in qs[:4]] + [rnd_seq(r, r.randint(1, maxlen)), ""]
    check_against_oracle(sd.nw_identity(qs, ts, flavour=cases.EMU_LIB), qs, ts)
    pairs = ([0, 3, 6, 7, 2], [1, 1, 4, 0, 5])
    check_against_oracle(sd.nw_identity(qs, ts, pairs=pairs, flavour=cases.EMU_LIB), qs, ts, pairs)


def test_identity_argument_errors():
    with pytest.raises(sd.SdError) as e:
        sd.nw_identity(["A" * 16383], ["A"], flavour=cases.EMU_LIB)
    assert e.value.status == 3
    with pytest.raises(sd.SdError):
        sd.nw_identity(["A"], ["A"], pairs=([0], [1]), flavour=cases.EMU_LIB)
    res = sd.nw_identity([], ["A"], flavour=cases.EMU_LIB)
    assert len(res["matches"]) == 0
    # long sequences: all mismatches, a pure length difference, a periodic pair
    ext = sd.nw_identity(["A" * 8000, "A" * 8000, "ACGT" * 2000], ["C" * 8000, "A" * 7000, "ACGA" * 2000], pairs=([0, 1, 2], [0, 1, 2]),
                         flavour=cases.EMU_LIB)
    assert list(ext["distance"]) == [8000, 1000, 2000] and list(ext["matches"]) == [0, 7000, 6000]
    assert list(ext["columns"]) == [8000, 8000, 8000]
    edge = sd.nw_identity(["A" * 16382, "C" * 5], ["C" * 5, "A" * 16382], pairs=([0, 1], [0, 1]), flavour=cases.EMU_LIB)   # the longest
    assert list(edge["distance"]) == [16382, 16382] and list(edge["columns"]) == [16382, 16382]
    big = sd.nw_identity(["A" * 2300], ["A" * 1536], flavour=cases.EMU_LIB)
    assert big["hirschberg_pairs"] == 1 and big["distance"][0] == 764


@pytest.mark.parametrize("light", [False, True])
def test_convert_tsv_over_emulator(tmp_path, light):
    reads, mons, raw = _golden_inputs()
    out = str(tmp_path / "o.tsv")
    stats = {}
    cv.convert_tsv(raw, cv.load_fasta(os.path.join(G, "config1_read.fa"), "map"),
                   cv.add_rc_monomers(cv.load_fasta(os.path.join(G, "DXZ1_star_monomers.fa"))), out, 0, light,
                   flavour=cases.EMU_LIB, stats=stats)
    fin, alt = CO.final_tsv(raw, reads, mons, 0, light)
    assert open(out).read() == fin
    assert open(out[:-4] + "_alt.tsv").read() == alt
    if not light:
        assert fin == open(os.path.join(G, "config1_final_decomposition.tsv")).read()
        assert stats["pairs"] == 557 * 24 * 2


def test_convert_min_identity_duplicates_and_chunking(tmp_path, monkeypatch):
    r = random.Random(9)
    mons = [("m1", rnd_seq(r, 60)), ("m2", rnd_seq(r, 70)), ("m1", rnd_seq(r, 65))]       # repeated name
    read = "".join(noisy(r, mons[r.randrange(3)][1], 0.1) for _ in range(12))
    raw, pos = [], 0
    for k in range(12):
        raw.append("rd extra\t%s\t%d\t%d\t1.0\t0\t0\n" % (r.choice(["m1", "m2", "m1'"]), pos, pos + 59))
        pos += 60
    raw = "".join(raw)
    monkeypatch.setattr(cv, "MAX_PAIRS_PER_CALL", 24)                                      # several device calls
    for light in (True, False):
        for thr in (0, 60):
            out = str(tmp_path / ("o%d%d.tsv" % (light, thr)))
            cv.convert_tsv(raw, {"rd": read}, cv.add_rc_monomers(mons), out, thr, light, flavour=cases.EMU_LIB)
            fin, alt = CO.final_tsv(raw, {"rd": read}, mons, thr, light)
            assert open(out).read() == fin and open(out[:-4] + "_alt.tsv").read() == alt
            # the per-read entry points of the reference (print_read / convert_read dicts) give the same text
            import io
            fo, fa = io.StringIO(), io.StringIO()
            dec = [{"m": ln.split("\t")[1], "start": int(ln.split("\t")[2]), "end": int(ln.split("\t")[3])} for ln in raw.splitlines()]
            cv.print_read(fo, fa, dec, read, cv.add_rc_monomers(mons), thr, light, read_name="rd", flavour=cases.EMU_LIB)
            assert fo.getvalue() == fin and fa.getvalue() == alt


def test_convert_edge_cases_follow_the_reference(tmp_path):
    mons = [("m1", "ACGTACGTTACG"), ("m2", "TTGACCAGTAGC")]
    rc = cv.add_rc_monomers(mons)
    reads = {"r1": "ACGTACGTTACGTTGACCAGTAGCACGT", "r2": "GCTACTGGTCAA"}
    out = str(tmp_path / "o.tsv")
    cv.convert_tsv("", reads, rc, out, 0, True, flavour=cases.EMU_LIB)                      # no raw lines at all
    assert open(out).read() == "" and open(out[:-4] + "_alt.tsv").read() == ""
    # columns 1 and 2 are cut at the first blank (main.py:175-176); the last three columns of the raw file are unused
    raw = "r1 tail words\tm1 x\t0\t11\t9.0\t0\t11\nr1\tm2\t12\t23\t9.0\t0\t11\nr2\tm2'\t0\t11\t1.0\t0\t11\nr1\tm1\t24\t27\t1.0\t0\t3\n"
    for light in (True, False):
        cv.convert_tsv(raw, reads, rc, out, 0, light, flavour=cases.EMU_LIB)
        fin, alt = CO.final_tsv(raw, reads, mons, 0, light)
        assert open(out).read() == fin and open(out[:-4] + "_alt.tsv").read() == alt
        assert fin.splitlines()[0].startswith("r1\tm1\t0\t11\t100.00\t") and fin.splitlines()[2].startswith("r2\tm2'\t0\t11\t100.00\t")
    with pytest.raises(KeyError):                                                            # reads[prev_read], main.py:178
        cv.convert_tsv("nope\tm1\t0\t3\t1\t0\t3\n", reads, rc, out, 0, True, flavour=cases.EMU_LIB)
    with pytest.raises(KeyError):                                                            # scores[monomer], main.py:117
        cv.convert_tsv("r1\tother\t0\t3\t1\t0\t3\n", reads, rc, out, 0, True, flavour=cases.EMU_LIB)
    # an interval that runs past the end of the read is cut by the slice (main.py:115), an empty one scores 0
    raw = "r2\tm1\t8\t40\t1\t0\t3\nr2\tm1\t30\t40\t1\t0\t3\n"
    cv.convert_tsv(raw, reads, rc, out, 0, True, flavour=cases.EMU_LIB)
    assert open(out).read() == CO.final_tsv(raw, reads, mons, 0, True)[0]
    assert open(out).read().splitlines()[1].split("\t")[4] == "0.00"


@pytest.mark.parametrize("light", [False, True])
def test_native_convert_equals_python_mirror_and_golden(tmp_path, light):
    reads, mons, raw = _golden_inputs()
    out = str(tmp_path / "n.tsv")
    st = cv.convert_tsv_native(raw, cv.load_fasta(os.path.join(G, "config1_read.fa"), "map"),
                               cv.add_rc_monomers(cv.load_fasta(os.path.join(G, "DXZ1_star_monomers.fa"))), out, 0, light,
                               flavour=cases.EMU_LIB)
    fin, alt = CO.final_tsv(raw, reads, mons, 0, light)
    assert open(out).read() == fin and open(out[:-4] + "_alt.tsv").read() == alt
    assert st["lines_in"] == 557 and st["lines_out"] == 557 and st["pairs"] == (557 if light else 557 * 48)
    if not light:
        assert fin == open(os.path.join(G, "config1_final_decomposition.tsv")).read()


def test_native_convert_edge_cases(tmp_path, monkeypatch):
    r = random.Random(12)
    mons = [("m1", rnd_seq(r, 60)), ("m2", rnd_seq(r, 70) + "*"), ("m1", rnd_seq(r, 65)), ("m3", "AAAAAACCCCCCGGGGGTTTT")]
    rc = cv.add_rc_monomers(mons)
    read = "".join(noisy(r, mons[r.randrange(3)][1].rstrip("*"), 0.1) for _ in range(12)) + "*"
    reads = {"rd": read, "other": "ACGTTTGACA"}
    raw = []
    pos = 0
    for k in range(12):
        raw.append("rd extra words\t%s more\t%d\t%d\t1.0\t0\t0\n" % (r.choice(["m1", "m2", "m1'", "m3'"]), pos, pos + 59))
        pos += 60
    raw += ["other\tm3\t2\t400\t1\t0\t0\n", "other\tm2\t50\t60\t1\t0\t0\n", "rd\tm1\t%d\t%d\t1\t0\t0\n" % (len(read) - 20, len(read) - 1),
            "rd\tm2\t0\t10\ttrailing line without newline"]
    raw = "".join(raw)
    for light in (True, False):
        for thr in (0, 55, 101):
            a, b = str(tmp_path / "p.tsv"), str(tmp_path / "n.tsv")
            cv.convert_tsv(raw, reads, rc, a, thr, light, flavour=cases.EMU_LIB)
            st = cv.convert_tsv_native(raw, reads, rc, b, thr, light, flavour=cases.EMU_LIB)
            assert open(a).read() == open(b).read() and open(a[:-4] + "_alt.tsv").read() == open(b[:-4] + "_alt.tsv").read()
            assert st["lines_in"] == 15 and open(b).read() == CO.final_tsv(raw, reads, mons, thr, light)[0]
    monkeypatch.setenv("SD_CONVERT_LINES", "4")                                  # four device calls instead of one
    for light in (True, False):
        a, b = str(tmp_path / "p.tsv"), str(tmp_path / "n.tsv")
        cv.convert_tsv(raw, reads, rc, a, 0, light, flavour=cases.EMU_LIB)
        cv.convert_tsv_native(raw, reads, rc, b, 0, light, flavour=cases.EMU_LIB)
        assert open(a).read() == open(b).read() and open(a[:-4] + "_alt.tsv").read() == open(b[:-4] + "_alt.tsv").read()
    monkeypatch.delenv("SD_CONVERT_LINES")
    out = str(tmp_path / "e.tsv")
    assert cv.convert_tsv_native("", reads, rc, out, 0, True, flavour=cases.EMU_LIB)["lines_in"] == 0 and open(out).read() == ""
    with pytest.raises(KeyError):
        cv.convert_tsv_native("nope\tm1\t0\t3\t1\t0\t3\n", reads, rc, out, 0, True, flavour=cases.EMU_LIB)
    with pytest.raises(KeyError):
        cv.convert_tsv_native("rd\tnope\t0\t3\t1\t0\t3\n", reads, rc, out, 0, False, flavour=cases.EMU_LIB)
    with pytest.raises(sd.SdError):
        cv.convert_tsv_native("rd\tm1\t0\n", reads, rc, out, 0, True, flavour=cases.EMU_LIB)
    with pytest.raises(sd.SdError):
        cv.convert_tsv_native("rd\tm1\tx\t3\t1\n", reads, rc, out, 0, True, flavour=cases.EMU_LIB)


def test_helpers_follow_the_reference():
    assert cv.convert_to_homo("AAACCGTTTA") == "ACGTA" and cv.convert_to_homo("") == ""
    assert cv.add_rc_monomers([("x", "AACGN")]) == [("x", "AACGN"), ("x'", "NCGTT")]
    blob, off = cv._collapse(b"AAACCAAT", np.array([0, 3, 5, 8]))
    assert (blob, list(off)) == (b"ACAT", [0, 1, 2, 4])
    blob, off = cv._pack(["ACGT*", "", "A*", "*", "AC", "**"])                      # one trailing '*' dropped, main.py:38-41
    assert (blob, list(off)) == (b"ACGTAAC*", [0, 4, 4, 5, 5, 7, 8])
    assert list(cv.classify([95.0, 20.0], [-1, -1])) == ["+", "?"]
    assert cv.aai(["ACGT*", "ACGT"], flavour=cases.EMU_LIB) == 100.0
    assert cv.aai(["", "ACGT"], flavour=cases.EMU_LIB) == 0.0


def test_command_line_over_emulator(tmp_path):
    names, seqs = sd.read_fasta(os.path.join(G, "config1_read.fa"))
    rp = tmp_path / "reads.fa"
    rp.write_text(">%s words after the id\n%s\n>second\n%s\n" % (names[0], seqs[0][:9000], seqs[0][20000:23000]))
    mp = os.path.join(G, "DXZ1_star_monomers.fa")
    assert sdmain.main([str(rp), mp, "-o", str(tmp_path / "out"), "--second-best", "-i", "70"], flavour=cases.EMU_LIB) == 0
    raw = (tmp_path / "out" / "final_decomposition_raw.tsv").read_text()
    fin, alt = CO.final_tsv(raw, dict(CO.fasta_records(str(rp))), CO.fasta_records(mp), 70, light=False)
    assert (tmp_path / "out" / "final_decomposition.tsv").read_text() == fin and fin
    assert (tmp_path / "out" / "final_decomposition_alt.tsv").read_text() == alt
    assert (tmp_path / "out" / "stringdecomposer.log").exists()
    with pytest.raises(sd.SdError):                                   # lower-case read: dp exits 255, main.py raises
        bad = tmp_path / "bad.fa"
        bad.write_text(">x\nacgt\n")
        sdmain.main([str(bad), mp, "-o", str(tmp_path / "out2")], flavour=cases.EMU_LIB)


# ------------------------------------------------------------------------------------------ CUDA kernel through the C ABI
@pytest.mark.gpu
def test_gpu_identity_golden_pairs_from_reference_edlib():
    ps = golden_pairs()
    qs, ts = [p["q"] for p in ps], [p["t"] for p in ps]
    k = np.arange(len(ps), dtype=np.int32)
    res = sd.nw_identity(qs, ts, pairs=(k, k))
    assert list(res["distance"]) == [p["distance"] for p in ps]
    assert list(res["matches"]) == [p["matches"] for p in ps]
    assert list(res["columns"]) == [p["columns"] for p in ps]
    assert res["kernel_ms"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("maxlen", [30, 64, 100, 128, 180, 192, 250, 256, 600, 1300])
def test_gpu_identity_fuzz_against_oracle(maxlen):
    r = random.Random(1000 + maxlen)
    qs = [rnd_seq(r, r.randint(1, maxlen), r.choice(["AC", "ACGT", "ACGTN"])) for _ in range(20)] + ["A" * maxlen, ""]
    ts = [noisy(r, q, r.choice((0.05, 0.3))) or "C" for q in qs[:12]] + [rnd_seq(r, r.randint(1, maxlen)) for _ in range(4)] + [""]
    check_against_oracle(sd.nw_identity(qs, ts), qs, ts)
    pq = [r.randrange(len(qs)) for _ in range(50)]
    pt = [r.randrange(len(ts)) for _ in range(50)]
    check_against_oracle(sd.nw_identity(qs, ts, pairs=(pq, pt)), qs, ts, (pq, pt))


@pytest.mark.gpu
def test_gpu_identity_longest_supported_sequences():
    ext = sd.nw_identity(["A" * 16382, "A" * 16382, "ACGT" * 4000, "G"], ["C" * 16382, "A" * 15000, "ACGA" * 4000, "T" * 16382],
                         pairs=([0, 1, 2, 3, 0], [0, 1, 2, 3, 3]))
    assert list(ext["distance"]) == [16382, 1382, 4000, 16382, 16382] and list(ext["matches"]) == [0, 15000, 12000, 0, 0]
    assert list(ext["columns"]) == [16382, 16382, 16000, 16382, 16382]
    with pytest.raises(sd.SdError):
        sd.nw_identity(["A" * 16383], ["A"])


@pytest.mark.gpu
@pytest.mark.parametrize("light", [False, True])
def test_gpu_final_tsv_equals_reference_golden_file(tmp_path, light):
    reads, mons, raw = _golden_inputs()
    out = str(tmp_path / "o.tsv")
    stats = {}
    cv.convert_tsv(raw, cv.load_fasta(os.path.join(G, "config1_read.fa"), "map"),
                   cv.add_rc_monomers(cv.load_fasta(os.path.join(G, "DXZ1_star_monomers.fa"))), out, 0, light, stats=stats)
    fin, alt = CO.final_tsv(raw, reads, mons, 0, light)
    assert open(out).read() == fin and open(out[:-4] + "_alt.tsv").read() == alt
    if not light:
        assert fin == open(os.path.join(G, "config1_final_decomposition.tsv")).read()      # the reference's own file
    assert stats["kernel_ms"] > 0 and stats["hirschberg_pairs"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("light", [False, True])
def test_gpu_native_convert_equals_reference_golden_file(tmp_path, light):
    reads, mons, raw = _golden_inputs()
    out = str(tmp_path / "n.tsv")
    st = cv.convert_tsv_native(raw, cv.load_fasta(os.path.join(G, "config1_read.fa"), "map"),
                               cv.add_rc_monomers(cv.load_fasta(os.path.join(G, "DXZ1_star_monomers.fa"))), out, 0, light)
    fin, alt = CO.final_tsv(raw, reads, mons, 0, light)
    assert open(out).read() == fin and open(out[:-4] + "_alt.tsv").read() == alt
    if not light:
        assert fin == open(os.path.join(G, "config1_final_decomposition.tsv")).read()      # the reference's own file
    assert st["kernel_ms"] > 0 and st["lines_out"] == 557


@pytest.mark.gpu
def test_gpu_command_line_end_to_end_equals_reference_golden_file(tmp_path):
    assert sdmain.main([os.path.join(G, "config1_read.fa"), os.path.join(G, "DXZ1_star_monomers.fa"), "-o", str(tmp_path),
                        "--second-best"]) == 0
    assert (tmp_path / "final_decomposition.tsv").read_text() == open(os.path.join(G, "config1_final_decomposition.tsv")).read()
    assert (tmp_path / "final_decomposition_raw.tsv").read_text() == open(os.path.join(G, "config1_raw_default.tsv")).read()


@pytest.mark.gpu
def test_gpu_identity_full_size_properties():
    """Config-2-sized rescoring (12k intervals x 24 monomers, plain): properties that need no oracle, and every pair
    against the oracle."""
    from stringdecomposer_b200 import synth
    r = random.Random(2)
    _, mons = sd.read_fasta(os.path.join(G, "DXZ1_star_monomers.fa"))
    rows = mons + [synth.revcomp(m) for m in mons]
    truth = [r.randrange(len(rows)) for _ in range(12000)]
    qs = [noisy(r, rows[t], 0.02) for t in truth]
    res = sd.nw_identity(qs, rows)
    m = res["matches"].reshape(len(qs), len(rows)); c = res["columns"].reshape(m.shape); d = res["distance"].reshape(m.shape)
    ql = np.array([len(q) for q in qs])[:, None]; tl = np.array([len(t) for t in rows])[None, :]
    assert (c == m + d).all() and (c >= np.maximum(ql, tl)).all() and (c <= ql + tl).all()
    assert (d >= np.abs(ql - tl)).all() and (m <= np.minimum(ql, tl)).all()
    assert (np.argmax(m / c, axis=1) == np.array(truth)).mean() > 0.99
    again = sd.nw_identity(qs[:500], rows)
    assert (again["matches"] == res["matches"][:500 * len(rows)]).all()
    qb, qo = cv._pack(qs)
    tb, to = cv._pack(rows)
    want = O.nw_path_counts_batch(qb, qo, tb, to, np.repeat(np.arange(len(qs)), len(rows)), np.tile(np.arange(len(rows)), len(qs)))
    for name, got, w in zip(("distance", "matches", "columns"), (res["distance"], res["matches"], res["columns"]), want):
        bad = np.flatnonzero(got != w)
        assert len(bad) == 0, "%s: %d pairs differ from the oracle, first (interval %d, row %d): %d != %d" % (
            name, len(bad), bad[0] // len(rows), bad[0] % len(rows), got[bad[0]], w[bad[0]])


def test_raw_file_is_streamed_in_chunks_of_whole_reads(tmp_path):
    # main.py:195-197 reads the raw file into one string; the rescoring stage here streams it (convert.raw_chunks) and
    # must produce the same two files whatever the chunk size
    from stringdecomposer_b200 import convert as cv
    G = cases.GOLDEN
    raw = open(os.path.join(G, "config1_raw_default.tsv")).read()
    lines = raw.splitlines(True)
    two = "".join(lines[:300]) + "".join(ln.replace(lines[0].split("\t")[0], "second_read", 1) for ln in lines[:200])
    rp = tmp_path / "raw.tsv"
    rp.write_text(two)
    chunks = list(cv.raw_chunks(str(rp), 4000))
    assert "".join(chunks) == two and len(chunks) == 2            # cut only where the read name changes
    reads = cv.load_fasta(os.path.join(G, "config1_read.fa"), "map")
    reads["second_read"] = next(iter(reads.values()))
    mons = cv.add_rc_monomers(cv.load_fasta(os.path.join(G, "DXZ1_star_monomers.fa")))
    a, b = str(tmp_path / "a.tsv"), str(tmp_path / "b.tsv")
    cv.convert_tsv_native(two, reads, mons, a, 0, True, flavour=cases.EMU_LIB)
    cv.convert_raw_file_native(str(rp), reads, mons, b, 0, True, flavour=cases.EMU_LIB, max_bytes=4000)
    assert open(a).read() == open(b).read() and open(a[:-4] + "_alt.tsv").read() == open(b[:-4] + "_alt.tsv").read()

