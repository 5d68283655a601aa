"""The identity rescoring kernel (identity_kernel<R, L>, csrc/identity_kernels.cu) against the oracle on every cell.

A pair reports one (distance, matches, columns) triple, that of its last cell, so an error in a row, a lane hand-over or
a tile the kernel does not report would only show when it reaches that cell.  Here the queries are all prefixes of q
and the targets all prefixes of t: with edlib's boundary the NW matrix of a prefix pair is the top-left block of the
full one, so the results of the all-against-all call, reshaped to [len(q), len(t)], must equal the triple of the walk
started at every cell (sd_oracle.nw_prefix_counts), and every tile edge of every geometry is crossed.  Each case runs
at every compiled geometry (SD_NW_GEOM) and at the natural pick, and the SD_PROFILE line shows which one ran.  Pair
lists with repeats, the longest sequences, batch-scale calls over the grow-only arena and sd_convert with several
device calls complete it.  Every GPU case has a twin on the host emulator (tests/emu) at a smaller size."""
import json
import os
import random
import re

import numpy as np
import pytest

import cases
import sd_convert_oracle as CO
import sd_oracle as O
import stringdecomposer_b200 as sd
from stringdecomposer_b200 import convert as cv
from stringdecomposer_b200 import synth

GEOMS = [(8, 8), (8, 16), (8, 24), (16, 12), (32, 6), None]          # (L, R); None: the pick of nw_choose_rows
GEOM_IDS = ["L8R8", "L8R16", "L8R24", "L16R12", "L32R6", "natural"]
PROFILE = re.compile(r"sd_identity(?: \(emulator\))?: pairs (\d+) L (\d+) R (\d+)(?: blocks (\d+) x (\d+) pairs)?")


def golden_pairs():
    with open(os.path.join(cases.GOLDEN, "nw_pairs.json")) as f:
        return json.load(f)["pairs"]


def rnd(r, n, alpha="ACGT"):
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


def choose_rows(qlens):
    """nw_choose_rows (identity_core.cuh): the strip that minimises tiles x (7 R + 25) over the batch's queries"""
    cost = {R: sum(-(-ql // (8 * R)) * (7 * R + 25) for ql in qlens) for R in (8, 16, 24)}
    return min((8, 16, 24), key=lambda R: (cost[R], R))


def run(monkeypatch, capfd, flavour, geom, qs, ts, pairs=None):
    """sd.nw_identity at `geom` -> (result, (L, R, blocks, pairs per block)); asserts that `geom` is what ran"""
    if geom is None:
        monkeypatch.delenv("SD_NW_GEOM", raising=False)
    else:
        monkeypatch.setenv("SD_NW_GEOM", "%d,%d" % geom)
    monkeypatch.setenv("SD_PROFILE", "1")
    capfd.readouterr()
    res = sd.nw_identity(qs, ts, pairs=pairs, flavour=flavour)
    lines = PROFILE.findall(capfd.readouterr().err)
    assert len(lines) == 1, "expected one sd_identity profile line"
    n, L, R, blocks, per_block = (int(x) if x else 0 for x in lines[0])
    qlens = [len(q) for q in qs] if isinstance(qs, list) else list(np.diff(qs[1]))
    want = geom or (8, choose_rows(qlens))
    assert (L, R) == want and n == len(res["matches"]), "geometry %s ran as L %d R %d" % (want, L, R)
    return res, (L, R, blocks, per_block)


def triple(res):
    return res["distance"], res["matches"], res["columns"]


def assert_same(got, want, what, index_name="pair"):
    """got, want: (distance, matches, columns) arrays of one shape; names the first wrong index with both triples"""
    bad = np.zeros(np.shape(want[0]), bool)
    for g, w in zip(got, want):
        bad |= np.asarray(g).reshape(np.shape(w)) != w
    if bad.any():
        k = tuple(int(x) for x in np.argwhere(bad)[0])
        gt = tuple(int(np.asarray(g).reshape(np.shape(w))[k]) for g, w in zip(got, want))
        wt = tuple(int(w[k]) for w in want)
        raise AssertionError("%s: %d of %d wrong; first at %s %s: kernel (d, m, c) = %s, oracle %s"
                             % (what, int(bad.sum()), bad.size, index_name, k if len(k) > 1 else k[0], gt, wt))


def prefixes(s):
    return [s[:i + 1] for i in range(len(s))]


# ------------------------------------------------------------------------------------------ the oracle's prefix table
@pytest.mark.parametrize("alpha", ["A", "AC", "ACGT", "ACGTN", "bytes"])
def test_prefix_table_equals_the_walk_on_every_cell(alpha):
    r = random.Random(alpha)
    for it in range(60):
        if alpha == "bytes":
            q = bytes(r.choice(b"AC*a\x00\xff") for _ in range(r.randint(1, 24)))
            t = bytes(r.choice(b"AC*a\x00\xff") for _ in range(r.randint(1, 24)))
        else:
            q = rnd(r, r.randint(1, 24), alpha)
            t = noisy(r, q, 0.3, alpha) or alpha[0] if it % 2 else rnd(r, r.randint(1, 24), alpha)
        want = np.array([[O.nw_path_counts(q[:i + 1], t[:j + 1]) for j in range(len(t))] for i in range(len(q))])
        assert_same(O.nw_prefix_counts(q, t), tuple(np.moveaxis(want, 2, 0)), "prefix table of %r, %r" % (q, t), "(i, j)")


def test_prefix_table_corner_equals_reference_edlib_golden_pairs():
    for p in golden_pairs():
        d, m, c = O.nw_prefix_counts(p["q"], p["t"])
        assert (d[-1, -1], m[-1, -1], c[-1, -1]) == (p["distance"], p["matches"], p["columns"]), p["note"]


def test_batch_oracle_equals_the_walk():
    r = random.Random(3)
    qs = [rnd(r, r.randint(1, 300), r.choice(["AC", "ACGT"])) for _ in range(30)] + [""]
    ts = [noisy(r, q) or "G" for q in qs[:20]] + [rnd(r, r.randint(1, 300)) for _ in range(5)] + [""]
    pq = np.array([r.randrange(len(qs)) for _ in range(400)])
    pt = np.array([r.randrange(len(ts)) for _ in range(400)])
    got = O.nw_path_counts_batch(*pack(qs), *pack(ts), pq, pt)
    want = np.array([O.nw_path_counts(qs[i], ts[j]) for i, j in zip(pq, pt)]).T
    assert_same(got, tuple(want), "batch oracle")


# ------------------------------------------------------------------------------------------ prefix tables
def prefix_case(name, small):
    """(q, t) of a prefix-table case; `small` for the emulator.  Every geometry's tiles are 64, 128 or 192 rows tall, and
    the prefixes of q run past three tiles of 192 rows (577 rows) on the GPU and past one (197 rows) on the emulator."""
    r = random.Random(name)
    nq = 197 if small else 3 * 192 + 1
    if name == "noisy":
        q = rnd(r, nq)
        return q, noisy(r, q)[:nq + 40] or "A"
    if name == "A":
        return "A" * nq, "A" * (60 if small else 600)
    if name == "AC":
        return rnd(r, nq, "AC"), rnd(r, 70 if small else 560, "AC")
    if name == "unrelated":
        return rnd(r, nq), rnd(r, 60 if small else 500)
    if name == "short_long":
        return rnd(r, 40), noisy(r, rnd(r, 400 if small else 1500))
    if name == "odd_bytes":                      # '*' in the middle, lower case, 0xff (not the NW_NOCHAR padding)
        al = b"ACGTNacgt*\xff"
        q = bytes(r.choice(al) for _ in range(nq))
        return q, bytes(r.choice(al) for _ in range(60 if small else 300))
    raise KeyError(name)


PREFIX_CASES = ["noisy", "A", "AC", "unrelated", "short_long", "odd_bytes"]
_tables = {}


def prefix_table(name, small):
    if (name, small) not in _tables:
        q, t = prefix_case(name, small)
        _tables[name, small] = (q, t, O.nw_prefix_counts(q, t))
    return _tables[name, small]


def check_prefix_table(monkeypatch, capfd, flavour, geom, name, small):
    q, t, want = prefix_table(name, small)
    res, (L, R, _, _) = run(monkeypatch, capfd, flavour, geom, prefixes(q), prefixes(t))
    assert_same(triple(res), want, "prefix table %r (%d x %d) at L %d R %d" % (name, len(q), len(t), L, R), "(i, j)")


def check_pair_list(monkeypatch, capfd, flavour, geom, small):
    q, t, want = prefix_table("noisy", small)
    rng = np.random.default_rng(7)
    n = 3000 if small else 60000
    pq, pt = rng.integers(0, len(q), n), rng.integers(0, len(t), n)
    pq[n // 2:] = pq[:n - n // 2]                                # repeats: the same pair on other lane groups
    res, (L, R, _, _) = run(monkeypatch, capfd, flavour, geom, prefixes(q), prefixes(t), pairs=(pq, pt))
    assert_same(triple(res), tuple(w[pq, pt] for w in want), "pair list of %d at L %d R %d" % (n, L, R))


@pytest.mark.parametrize("name", PREFIX_CASES)
@pytest.mark.parametrize("geom", GEOMS, ids=GEOM_IDS)
def test_emulated_prefix_tables(monkeypatch, capfd, geom, name):
    check_prefix_table(monkeypatch, capfd, cases.EMU_LIB, geom, name, True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", PREFIX_CASES)
@pytest.mark.parametrize("geom", GEOMS, ids=GEOM_IDS)
def test_gpu_prefix_tables(monkeypatch, capfd, geom, name):
    check_prefix_table(monkeypatch, capfd, "cuda", geom, name, False)


@pytest.mark.parametrize("geom", GEOMS, ids=GEOM_IDS)
def test_emulated_pair_list_with_repeats(monkeypatch, capfd, geom):
    check_pair_list(monkeypatch, capfd, cases.EMU_LIB, geom, True)


@pytest.mark.gpu
@pytest.mark.parametrize("geom", GEOMS, ids=GEOM_IDS)
def test_gpu_pair_list_with_repeats(monkeypatch, capfd, geom):
    check_pair_list(monkeypatch, capfd, "cuda", geom, False)


def test_unsupported_geometry_is_refused(monkeypatch):
    monkeypatch.setenv("SD_NW_GEOM", "8,12")
    with pytest.raises(sd.SdError) as e:
        sd.nw_identity(["ACGT"], ["ACGA"], flavour=cases.EMU_LIB)
    assert "SD_NW_GEOM" in str(e.value)


# ------------------------------------------------------------------------------------------ the longest sequences
def long_pairs(small):
    """(queries, targets, pair list) at the 16,382 limit and next to tile multiples (64 * 255 = 192 * 85 = 16,320,
    128 * 127 = 16,256).  The last tile of a 16,382-row query has padding rows at 16,383 and above, whose initial D
    wraps past 14 bits."""
    r = random.Random(16382)
    if small:                                   # long against short: cheap on the emulator and for the oracle
        qs = ["A" * 16382, rnd(r, 16320), rnd(r, 250), rnd(r, 193)]
        ts = [rnd(r, 250, "CGT"), rnd(r, 16382), noisy(r, rnd(r, 16257))]
        return qs, ts, ([0, 1, 2, 3, 0], [0, 0, 1, 2, 1])
    a = rnd(r, 16382)
    qs = [a, rnd(r, 16320), "A" * 16321, rnd(r, 16256), rnd(r, 300)]
    ts = [noisy(r, a, 0.1)[:16382], rnd(r, 16382, "CGT"), noisy(r, a[:16256], 0.3), rnd(r, 16257)]
    return qs, ts, ([0, 1, 2, 3, 0, 4], [0, 0, 1, 2, 2, 3])


_long = {}


def long_oracle(small):
    if small not in _long:
        qs, ts, (pq, pt) = long_pairs(small)
        _long[small] = np.array([O.nw_path_counts(qs[i], ts[j]) for i, j in zip(pq, pt)]).T   # ~1 GB per 16k x 16k pair
    return _long[small]


def check_long(monkeypatch, capfd, flavour, geom, small):
    qs, ts, pairs = long_pairs(small)
    want = long_oracle(small)
    res, (L, R, _, _) = run(monkeypatch, capfd, flavour, geom, qs, ts, pairs=pairs)
    assert_same(triple(res), tuple(want), "longest sequences at L %d R %d" % (L, R))
    return want


@pytest.mark.parametrize("geom", GEOMS, ids=GEOM_IDS)
def test_emulated_longest_sequences(monkeypatch, capfd, geom):
    want = check_long(monkeypatch, capfd, cases.EMU_LIB, geom, True)
    assert want[0][0] == 16382                                     # D at the top of its 14 bits


@pytest.mark.gpu
@pytest.mark.parametrize("geom", GEOMS, ids=GEOM_IDS)
def test_gpu_longest_sequences(monkeypatch, capfd, geom):
    want = check_long(monkeypatch, capfd, "cuda", geom, False)
    assert want[0][2] == 16382 and want[1][0] > 10000               # D at the top of its 14 bits, M in the thousands


# ------------------------------------------------------------------------------------------ scale and the arena
def scale_inputs(small):
    """DXZ1 rows (24) and longer targets (two and three monomers), config-2-like noisy intervals, 300-1,300 bp intervals"""
    r = random.Random(24)
    _, mons = sd.read_fasta(os.path.join(cases.GOLDEN, "DXZ1_star_monomers.fa"))
    rows = mons + [synth.revcomp(m) for m in mons]
    longer = [rows[k] + rows[k + 1] for k in range(0, 6, 2)] + [rows[k] + rows[k + 1] + rows[k + 2] for k in range(12, 21, 3)]
    arr = synth.hor_array(mons, 400_000, 0.03, seed=24)
    n_short, n_long, hi = (300, 20, 700) if small else (12000, 2000, 1300)
    short = [noisy(r, rows[r.randrange(24)], 0.02) for _ in range(n_short)]
    long_ = []
    for _ in range(n_long):
        s = r.randrange(len(arr) - hi)
        long_.append(arr[s:s + r.randint(300, hi)])
    return rows, longer, short, long_


def pack(seqs):
    blob = "".join(seqs).encode()
    off = np.zeros(len(seqs) + 1, np.int64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    return blob, off


def all_pairs(nq, nt):
    return np.repeat(np.arange(nq, dtype=np.int32), nt), np.tile(np.arange(nt, dtype=np.int32), nq)


def check_scale(monkeypatch, capfd, flavour, small):
    rows, longer, short, long_ = scale_inputs(small)
    targets, queries = rows + longer, short + long_
    qb, qo = pack(queries)
    tb, to = pack(targets)
    want = np.stack(O.nw_path_counts_batch(qb, qo, tb, to, *all_pairs(len(queries), len(targets))))
    want = want.reshape(3, len(queries), len(targets))
    calls = []

    def call(what, qi, ti, pairs=None):
        qsub, tsub = [queries[i] for i in qi], [targets[j] for j in ti]
        res, geo = run(monkeypatch, capfd, flavour, None, qsub, tsub, pairs=pairs)
        exp = want[:, qi][:, :, ti]
        exp = exp.reshape(3, -1) if pairs is None else exp[:, pairs[0], pairs[1]]
        assert_same(triple(res), tuple(exp), "%s (%d pairs) at L %d R %d" % (what, exp.shape[1], geo[0], geo[1]))
        calls.append((what, exp.shape[1]) + geo)

    ns, nl = len(short), len(long_)
    call("config-2-shaped batch", range(ns), range(24))
    collapsed_q, collapsed_t = [cv.convert_to_homo(s) for s in short], [cv.convert_to_homo(t) for t in rows]
    res, geo = run(monkeypatch, capfd, flavour, None, collapsed_q, collapsed_t)
    cb, co = pack(collapsed_q)
    tb2, to2 = pack(collapsed_t)
    exp = O.nw_path_counts_batch(cb, co, tb2, to2, *all_pairs(ns, 24))
    assert_same(triple(res), exp, "homopolymer-collapsed batch (%d pairs) at L %d R %d" % (len(exp[0]), geo[0], geo[1]))
    calls.append(("homopolymer-collapsed batch", len(exp[0])) + geo)
    call("300-%d bp intervals" % max(map(len, long_)), range(ns, ns + nl), range(len(targets)))
    call("small call", [ns + 1, 3], range(24))
    rng = np.random.default_rng(5)
    big = len(queries) * len(targets) * 5 // 4                    # larger than every call before: the arena grows
    call("pair list over everything", range(len(queries)), range(len(targets)),
         pairs=(rng.integers(0, len(queries), big), rng.integers(0, len(targets), big)))
    return calls


def test_emulated_scale_and_arena(monkeypatch, capfd):
    assert len(check_scale(monkeypatch, capfd, cases.EMU_LIB, True)) == 5


@pytest.mark.gpu
def test_gpu_scale_and_arena(monkeypatch, capfd):
    calls = check_scale(monkeypatch, capfd, "cuda", False)
    for what, npairs, L, R, blocks, per_block in calls:
        if npairs > 100000:
            assert blocks * per_block < npairs, "%s: the grid-stride loop made one trip only" % what


# ------------------------------------------------------------------------------------------ sd_convert at scale
def check_convert(tmp_path, monkeypatch, flavour, length, lines_per_call):
    names, mons = synth.load_dxz1()
    arr = synth.hor_array(mons, length, 0.02, seed=31)
    raw = sd.decompose_reads(["cfg2_like"], [arr], names, mons, flavour=flavour)
    n_lines = raw.count("\n")
    monkeypatch.setenv("SD_CONVERT_LINES", str(lines_per_call))
    out = str(tmp_path / "f.tsv")
    st = cv.convert_tsv_native(raw, {"cfg2_like": arr}, cv.add_rc_monomers(list(zip(names, mons))), out, 0, False,
                               flavour=flavour)
    fin, alt = CO.final_tsv(raw, {"cfg2_like": arr}, list(zip(names, mons)), 0, light=False)
    got = open(out).read().splitlines()
    for k, (g, w) in enumerate(zip(got, fin.splitlines())):
        assert g == w, "final_decomposition line %d differs:\n%s\n%s" % (k, g, w)
    assert len(got) == len(fin.splitlines()) == n_lines and open(out[:-4] + "_alt.tsv").read() == alt
    assert st["lines_out"] == n_lines and n_lines > 3 * lines_per_call
    return n_lines


def test_emulated_convert_several_calls(tmp_path, monkeypatch):
    assert check_convert(tmp_path, monkeypatch, cases.EMU_LIB, 30_000, 40) > 150


@pytest.mark.gpu
def test_gpu_convert_several_calls(tmp_path, monkeypatch):
    assert check_convert(tmp_path, monkeypatch, "cuda", 342_000, 450) > 1900


# ------------------------------------------------------------------------------------------ Hirschberg count
def test_hirschberg_pairs_count_at_the_one_mebibyte_limit():
    # edlib walks back a traceback only below 1 MiB of state: 20 bytes per 64-row block and column + 8 per column
    ql, tl = [], []
    for qlen in (64, 641, 1600, 12800, 16382):
        blocks = (qlen + 63) // 64
        t0 = (1 << 20) // (20 * blocks + 8)                        # the longest target below the limit, about
        for tlen in (t0 - 1, t0, t0 + 1, t0 + 2):
            if 0 < tlen <= 16382:
                ql.append(qlen); tl.append(tlen)
    res = sd.nw_identity(["A" * q for q in ql], ["C" * t for t in tl], pairs=(range(len(ql)), range(len(tl))),
                         flavour=cases.EMU_LIB)
    want = sum(not O.nw_uses_traceback(q, t) for q, t in zip(ql, tl))
    assert 0 < want < len(ql) and res["hirschberg_pairs"] == want
