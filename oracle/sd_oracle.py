"""ctypes wrapper of the CPU oracle (oracle/sd_oracle.c).  TEST INFRASTRUCTURE ONLY -- imported by tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline leg, never by the product package."""
import ctypes as C
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_build", "libsd_oracle.so")
BIN = os.path.join(HERE, "_build", "oracle_dp")
REF_BIN = os.path.join(HERE, "_ref", "dp")


class Rec(C.Structure):
    _fields_ = [("row", C.c_int), ("start", C.c_int), ("end", C.c_int), ("score", C.c_float)]


def build():
    subprocess.run(["make", "-s", "-C", HERE, "port"], check=True)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            build()
        _lib = C.CDLL(LIB)
        _lib.sdo_align_segment.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int,
                                           C.c_int, C.c_int, C.POINTER(Rec), C.c_int]
        _lib.sdo_align_segment.restype = C.c_int
        _lib.sdo_dp_tables.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.sdo_dp_tables.restype = C.c_int
        _lib.sdo_segment_read.argtypes = [C.c_long, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int]
        _lib.sdo_segment_read.restype = C.c_int
        _lib.sdo_postprocess.argtypes = [C.POINTER(Rec), C.c_int, C.POINTER(Rec)]
        _lib.sdo_postprocess.restype = C.c_int
        _lib.sdo_filter_rows.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(C.c_int)]
        _lib.sdo_filter_rows.restype = C.c_int
        _lib.sdo_nw_prefix_counts.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.sdo_nw_prefix_counts.restype = C.c_int
        _lib.sdo_nw_path_counts_batch.argtypes = [C.c_char_p, C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                  C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.sdo_nw_path_counts_batch.restype = C.c_int
    return _lib


_COMP = {"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}


def rows_of(monomers):
    """forward monomers, then all reverse complements (main.cpp:364-371)"""
    return list(monomers) + ["".join(_COMP[c] for c in reversed(m)) for m in monomers]


def filter_rows(seg, rows, ed_thr):
    """FilterMonomersForRead (main.cpp:135-149): indices of the rows kept for `seg`, in their new order"""
    off = (C.c_int * (len(rows) + 1))()
    for i, r in enumerate(rows):
        off[i + 1] = off[i] + len(r)
    keep = (C.c_int * max(len(rows), 1))()
    n = lib().sdo_filter_rows(seg.encode(), len(seg), "".join(rows).encode(), off, len(rows), ed_thr, keep)
    return [keep[i] for i in range(n)]


def align_segment(seg, monomers, scoring=(-1, -1, -1, 1), ed_thr=-1):
    """AlignPartClassicDP on one segment -> list of (row, start, end, score); ed_thr > -1 runs the rows that
    FilterMonomersForRead keeps, with any scoring (the dp command line only combines --ed_thr with the default one)"""
    rows = rows_of(monomers)
    keep = list(range(len(rows)))
    if ed_thr > -1:
        keep = filter_rows(seg, rows, ed_thr)
        rows = [rows[k] for k in keep]
    off = (C.c_int * (len(rows) + 1))()
    for i, r in enumerate(rows):
        off[i + 1] = off[i] + len(r)
    out = (Rec * (len(seg) + 1))()
    n = lib().sdo_align_segment(seg.encode(), len(seg), "".join(rows).encode(), off, len(rows), scoring[0], scoring[1],
                                scoring[2], scoring[3], out, len(seg) + 1)
    if n < 0:
        raise RuntimeError("oracle failed (%d)" % n)
    return [(keep[out[i].row], out[i].start, out[i].end, out[i].score) for i in range(n)]


def dp_tables(seg, monomers, scoring=(-1, -1, -1, 1), ed_thr=-1):
    """The DP table of one segment as the reference's traceback reads it (main.cpp:217-267) -> dict of numpy arrays:
      code  int8 [n][row_off[R]]: the traceback's move at cell (i, r, k) = code[i, row_off[r] + k]: 0 deletion,
            1 insertion, 2 diagonal, 3 close the alignment (the first equality of main.cpp:242-253 that holds)
      J     int64 [n+1]: J[i] = max_r H[i-1][r][last] for i = 1..n (J[n] is the final maximum)
      argJ  int32 [n+1]: the lowest row attaining J[i] (argJ[n] is the top row)
      row_off int32 [R+1], keep: the rows of the table as indices into rows_of(monomers).  With ed_thr > -1 the table
            covers the rows that FilterMonomersForRead keeps, in rank order, as align_segment does."""
    import numpy as np
    rows = rows_of(monomers)
    keep = list(range(len(rows)))
    if ed_thr > -1:
        keep = filter_rows(seg, rows, ed_thr)
        rows = [rows[k] for k in keep]
    n = len(seg)
    ro = np.zeros(len(rows) + 1, np.int32)
    ro[1:] = np.cumsum([len(r) for r in rows])
    code = np.zeros((n, int(ro[-1])), np.int8)
    J = np.zeros(n + 1, np.int64)
    argJ = np.zeros(n + 1, np.int32)
    st = lib().sdo_dp_tables(seg.encode(), n, "".join(rows).encode(), ro.ctypes.data_as(C.POINTER(C.c_int)), len(rows),
                             scoring[0], scoring[1], scoring[2], scoring[3], code.ctypes.data, J.ctypes.data, argJ.ctypes.data)
    if st < 0:
        raise RuntimeError("oracle failed (%d)" % st)
    return {"code": code, "J": J, "argJ": argJ, "row_off": ro, "keep": keep}


def segment_read(read_len, part, overlap):
    n = lib().sdo_segment_read(read_len, part, overlap, None, None, 0)
    offs, lens = (C.c_int * max(n, 1))(), (C.c_int * max(n, 1))()
    lib().sdo_segment_read(read_len, part, overlap, offs, lens, n)
    return [(offs[i], lens[i]) for i in range(n)]


def postprocess(recs):
    a = (Rec * max(len(recs), 1))(*[Rec(*r) for r in recs])
    b = (Rec * max(len(recs), 1))()
    n = lib().sdo_postprocess(a, len(recs), b)
    return [(b[i].row, b[i].start, b[i].end, b[i].score) for i in range(n)]


def run_cli(binary, reads_fa, monomers_fa, threads=1, part=5000, overlap=500, scoring=None, extra=()):
    """Run a dp-compatible binary; returns (status, stdout bytes, stderr bytes)."""
    cmd = [binary, reads_fa, monomers_fa, str(threads), str(part), str(overlap)]
    if scoring is not None:
        cmd += [str(x) for x in scoring]
    cmd += list(extra)
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    return p.returncode, p.stdout, p.stderr


def decompose_reads(read_names, reads, monomer_names, monomers, part_size=5000, overlap=500, scoring=(-1, -1, -1, 1),
                    binary=None, threads=None):
    """Whole `dp` run of the oracle port (or of `binary`, e.g. the compiled reference) on in-memory sequences."""
    if not os.path.exists(BIN):
        build()
    with tempfile.TemporaryDirectory() as td:
        rp, mp = os.path.join(td, "r.fa"), os.path.join(td, "m.fa")
        with open(rp, "w") as f:
            for n, s in zip(read_names, reads):
                f.write(">%s\n%s\n" % (n, s))
        with open(mp, "w") as f:
            for n, s in zip(monomer_names, monomers):
                f.write(">%s\n%s\n" % (n, s))
        st, out, err = run_cli(binary or BIN, rp, mp, threads or min(8, os.cpu_count() or 1), part_size, overlap,
                               None if tuple(scoring) == (-1, -1, -1, 1) else scoring)
        if st != 0:
            raise RuntimeError("oracle dp exited with %d: %s" % (st, err.decode()[-300:]))
        return out.decode()


# ---- identity rescoring (SURVEY §8 f1): sd_identity_oracle.c and the reference's own edlib ----------------
REF_EDLIB = os.path.join(HERE, "_ref", "libedlib_ref.so")
_ref_edlib = None


def _counts(fn, q, t):
    qb, tb = (s.encode() if isinstance(s, str) else bytes(s) for s in (q, t))
    m, c = C.c_int(), C.c_int()
    d = fn(qb, len(qb), tb, len(tb), C.byref(m), C.byref(c))
    return d, m.value, c.value


def nw_path_counts(q, t):
    """(edit distance, '=' columns, alignment columns) of edlib's NW path; distance -1 when either is empty."""
    f = lib().sdo_nw_path_counts
    f.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    return _counts(f, q, t)


def nw_prefix_counts(q, t):
    """The triple of nw_path_counts for every prefix pair (q[:i+1], t[:j+1]) -> (distance, matches, columns), three int32
    numpy arrays of shape [len(q), len(t)]; q and t non-empty str or bytes."""
    import numpy as np
    qb = q.encode() if isinstance(q, str) else bytes(q)
    tb = t.encode() if isinstance(t, str) else bytes(t)
    out = [np.zeros((len(qb), len(tb)), np.int32) for _ in range(3)]
    st = lib().sdo_nw_prefix_counts(qb, len(qb), tb, len(tb), *[C.c_void_p(a.ctypes.data) for a in out])
    if st:
        raise RuntimeError("sdo_nw_prefix_counts failed (%d)" % st)
    return tuple(out)


def nw_path_counts_batch(qtext, qoff, ttext, toff, pair_q, pair_t):
    """nw_path_counts of every pair (qtext[qoff[pair_q[k]]:qoff[pair_q[k]+1]], the same for t), packed inputs as
    sd_identity takes them, computed in parallel -> (distance, matches, columns) int32 arrays."""
    import numpy as np
    qo, to = np.ascontiguousarray(qoff, np.int64), np.ascontiguousarray(toff, np.int64)
    pq, pt = np.ascontiguousarray(pair_q, np.int32), np.ascontiguousarray(pair_t, np.int32)
    assert pq.shape == pt.shape and (pq.size == 0 or (0 <= pq.min() and pq.max() < len(qo) - 1 and 0 <= pt.min() and pt.max() < len(to) - 1))
    out = [np.zeros(len(pq), np.int32) for _ in range(3)]
    st = lib().sdo_nw_path_counts_batch(bytes(qtext), C.c_void_p(qo.ctypes.data), bytes(ttext), C.c_void_p(to.ctypes.data),
                                        C.c_void_p(pq.ctypes.data), C.c_void_p(pt.ctypes.data), C.c_int64(len(pq)),
                                        *[C.c_void_p(a.ctypes.data) for a in out])
    if st:
        raise RuntimeError("sdo_nw_path_counts_batch failed (%d)" % st)
    return tuple(out)


def nw_uses_traceback(qlen, tlen):
    return bool(lib().sdo_nw_uses_traceback(int(qlen), int(tlen)))


def ref_nw_path_counts(q, t):
    """The same triple from the reference's vendored edlib.cpp (oracle/_ref/libedlib_ref.so); non-empty inputs only."""
    global _ref_edlib
    if _ref_edlib is None:
        _ref_edlib = C.CDLL(REF_EDLIB)
        _ref_edlib.ref_nw_path_counts.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    return _counts(_ref_edlib.ref_nw_path_counts, q, t)


def identity(q, t):
    """aai of main.py:36-60: percent of '=' columns in edlib's NW alignment; 0 when either string is empty."""
    q = q[:-1] if q.endswith("*") else q                      # main.py:38-41
    t = t[:-1] if t.endswith("*") else t
    d, m, c = nw_path_counts(q, t)
    if d == -1:
        return 0
    return m / c * 100
