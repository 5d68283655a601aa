"""ctypes binding of include/sd_b200.h (the C ABI of libsd_b200.so)."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

RECORD_DTYPE = np.dtype([("row", "<i4"), ("start", "<i4"), ("end", "<i4"), ("score", "<i4")])


class SdError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("sd_b200 status %d: %s" % (status, msg))
        self.status = status


class _Stats(C.Structure):
    _fields_ = [("sweep_ms", C.c_double), ("traceback_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("cells", C.c_int64), ("segments", C.c_int64),
                ("columns", C.c_int64), ("launches", C.c_int64), ("n_devices", C.c_int32), ("packed", C.c_int32),
                ("C", C.c_int32), ("T", C.c_int32), ("NS", C.c_int32), ("NT", C.c_int32),
                ("NG", C.c_int32), ("lat", C.c_int32), ("scanw", C.c_int32), ("stream", C.c_int32),
                ("sweep_store_bytes", C.c_int64), ("dev_segments", C.c_int32 * 8)]


# every symbol include/sd_b200.h declares (tests/test_abi.py checks the header against this list)
class _ConvertStats(C.Structure):
    _fields_ = [("lines_in", C.c_int64), ("lines_out", C.c_int64), ("pairs", C.c_int64), ("hirschberg_pairs", C.c_int64),
                ("kernel_ms", C.c_double)]


SYMBOLS = ["sd_create", "sd_decompose", "sd_stage", "sd_run_staged", "sd_fetch_staged", "sd_segment_read",
           "sd_postprocess", "sd_run_files", "sd_set_ed_thr", "sd_hw_distance", "sd_get_stats", "sd_reset_stats", "sd_last_error", "sd_free", "sd_host_alloc", "sd_host_free",
           "sd_destroy", "sd_device_count", "sd_version", "sd_int_peak", "sd_identity", "sd_convert",
           "sd_convert_error"]

_libs = {}


def library_path(flavour="cuda"):
    """Path of the in-tree product library (CUDA, sm_100a).  Any other value of ``flavour`` is taken as the path of a
    library with the same C ABI -- the CPU test-suite passes its host emulator (tests/emu) this way; the package itself
    ships no CPU implementation."""
    if flavour == "cuda":
        return os.path.join(_HERE, "libsd_b200.so")
    return str(flavour)


def load_library(flavour="cuda"):
    if flavour in _libs:
        return _libs[flavour]
    path = library_path(flavour)
    if not os.path.exists(path):
        raise SdError(2, "%s is not built (run `python -c 'import __graft_entry__ as g; g.build()'` or "
                         "`make -C stringdecomposer_b200/csrc`); there is no fallback path" % path)
    lib = C.CDLL(path)
    p = C.c_void_p
    lib.sd_create.argtypes = [C.c_char_p, C.POINTER(C.c_int64), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                              C.POINTER(C.c_int32), C.c_int32, C.POINTER(p)]
    lib.sd_create.restype = C.c_int
    lib.sd_decompose.argtypes = [p, C.c_char_p, C.POINTER(C.c_int64), C.c_int64, C.POINTER(p), C.POINTER(p)]
    lib.sd_decompose.restype = C.c_int
    lib.sd_stage.argtypes = [p, C.c_char_p, C.POINTER(C.c_int64), C.c_int64]
    lib.sd_stage.restype = C.c_int
    lib.sd_run_staged.argtypes = [p, C.POINTER(C.c_double)]
    lib.sd_run_staged.restype = C.c_int
    lib.sd_fetch_staged.argtypes = [p, C.POINTER(p), C.POINTER(p)]
    lib.sd_fetch_staged.restype = C.c_int
    lib.sd_segment_read.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.c_int64]
    lib.sd_segment_read.restype = C.c_int64
    lib.sd_postprocess.argtypes = [p, C.c_int64, p]
    lib.sd_postprocess.restype = C.c_int64
    lib.sd_run_files.argtypes = [C.c_char_p, C.c_char_p] + [C.c_int32] * 8 + [C.c_int, C.c_int]
    lib.sd_run_files.restype = C.c_int
    lib.sd_set_ed_thr.argtypes = [p, C.c_int32]
    lib.sd_set_ed_thr.restype = C.c_int
    lib.sd_hw_distance.argtypes = [C.c_char_p, C.c_int32, C.c_char_p, C.c_int32]
    lib.sd_hw_distance.restype = C.c_int32
    lib.sd_get_stats.argtypes = [p, C.POINTER(_Stats)]
    lib.sd_get_stats.restype = C.c_int
    lib.sd_reset_stats.argtypes = [p]
    lib.sd_reset_stats.restype = None
    lib.sd_last_error.argtypes = [p]
    lib.sd_last_error.restype = C.c_char_p
    lib.sd_free.argtypes = [p]
    lib.sd_free.restype = None
    lib.sd_host_alloc.argtypes = [C.c_int64]
    lib.sd_host_alloc.restype = C.c_void_p
    lib.sd_host_free.argtypes = [C.c_void_p]
    lib.sd_host_free.restype = None
    lib.sd_destroy.argtypes = [p]
    lib.sd_destroy.restype = None
    lib.sd_device_count.restype = C.c_int
    lib.sd_version.restype = C.c_char_p
    lib.sd_int_peak.argtypes = [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.sd_int_peak.restype = C.c_int
    i32p, i64p = C.POINTER(C.c_int32), C.POINTER(C.c_int64)
    lib.sd_identity.argtypes = [C.c_char_p, i64p, C.c_int64, C.c_char_p, i64p, C.c_int64, i32p, i32p, C.c_int64,
                                i32p, i32p, i32p, C.c_int32, i64p, C.POINTER(C.c_double)]
    lib.sd_identity.restype = C.c_int
    lib.sd_convert.argtypes = [C.c_char_p, C.c_int64, C.c_char_p, i64p, C.c_char_p, i64p, C.c_int64, C.c_char_p, i64p, C.c_char_p,
                               i64p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int, C.c_int, C.POINTER(_ConvertStats)]
    lib.sd_convert.restype = C.c_int
    lib.sd_convert_error.restype = C.c_char_p
    _libs[flavour] = lib
    return lib


def device_count(flavour="cuda"):
    return int(load_library(flavour).sd_device_count())


def _pack(seqs):
    """list of str/bytes -> (bytes blob, int64 offsets)"""
    bs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    off = np.zeros(len(bs) + 1, dtype=np.int64)
    if bs:
        np.cumsum([len(b) for b in bs], out=off[1:])
    return b"".join(bs), off


class HostBuffer:
    """Segment text in page-locked host memory (sd_host_alloc): accepted wherever a `blob` is, copied to the device by
    plain DMA.  ``HostBuffer.pack(segments)`` -> (buffer, offsets)."""

    def __init__(self, data, flavour="cuda"):
        self._lib = load_library(flavour)
        self.size = len(data)
        self.ptr = self._lib.sd_host_alloc(self.size)
        if not self.ptr:
            raise MemoryError("sd_host_alloc(%d) failed" % self.size)
        C.memmove(self.ptr, data, self.size)

    @classmethod
    def pack(cls, segments, flavour="cuda"):
        blob, off = segments if isinstance(segments, tuple) else _pack(segments)
        return cls(blob, flavour), off

    def __len__(self):
        return self.size

    def __del__(self):
        if getattr(self, "ptr", None):
            self._lib.sd_host_free(self.ptr)
            self.ptr = None


def _text(blob):
    return C.c_char_p(blob.ptr) if isinstance(blob, HostBuffer) else blob


class Decomposer:
    """Mirror of the reference's MonomersAligner (main.cpp:56-66): monomers + scoring bound once, then
    batches of read segments are decomposed.  ``devices``: None -> GPU 0, "all" -> every visible GPU, or a list."""

    def __init__(self, monomers, ins=-1, dele=-1, mismatch=-1, match=1, devices=None, flavour="cuda"):
        self._lib = load_library(flavour)
        self._h = C.c_void_p()
        blob, off = _pack(monomers)
        if devices is None:
            ids, n = None, 0
        elif devices == "all":
            ids, n = None, -1
        else:
            arr = (C.c_int32 * len(devices))(*devices)
            ids, n = arr, len(devices)
        st = self._lib.sd_create(blob, off.ctypes.data_as(C.POINTER(C.c_int64)), len(monomers), ins, dele, mismatch, match,
                                 ids, n, C.byref(self._h))
        if st:
            raise SdError(st, (self._lib.sd_last_error(None) or b"").decode())
        self.n_monomers = len(monomers)

    def close(self):
        if self._h:
            self._lib.sd_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _err(self, st):
        raise SdError(st, (self._lib.sd_last_error(self._h) or b"").decode())

    def _take(self, recs, offs, nseg):
        # plain memmove into fresh arrays: np.ctypeslib.as_array / ctypes array types cost ~0.25 ms per call
        o = np.empty(nseg + 1, dtype=np.int64)
        C.memmove(o.ctypes.data, offs.value, 8 * (nseg + 1))
        n = int(o[-1])
        r = np.empty(n, dtype=RECORD_DTYPE)
        if n:
            C.memmove(r.ctypes.data, recs.value, n * RECORD_DTYPE.itemsize)
        self._lib.sd_free(recs)
        self._lib.sd_free(offs)
        return r, o

    def decompose(self, segments):
        """segments: list of ACGTN strings, or (blob, offsets).  Returns (records, rec_offsets)."""
        blob, off = segments if isinstance(segments, tuple) else _pack(segments)
        nseg = len(off) - 1
        recs, offs = C.c_void_p(), C.c_void_p()
        st = self._lib.sd_decompose(self._h, _text(blob), off.ctypes.data_as(C.POINTER(C.c_int64)), nseg, C.byref(recs), C.byref(offs))
        if st:
            self._err(st)
        return self._take(recs, offs, nseg)

    def stage(self, segments):
        blob, off = segments if isinstance(segments, tuple) else _pack(segments)
        self._staged = len(off) - 1
        st = self._lib.sd_stage(self._h, _text(blob), off.ctypes.data_as(C.POINTER(C.c_int64)), self._staged)
        if st:
            self._err(st)

    def run_staged(self):
        ms = C.c_double()
        st = self._lib.sd_run_staged(self._h, C.byref(ms))
        if st:
            self._err(st)
        return ms.value

    def fetch_staged(self):
        recs, offs = C.c_void_p(), C.c_void_p()
        st = self._lib.sd_fetch_staged(self._h, C.byref(recs), C.byref(offs))
        if st:
            self._err(st)
        return self._take(recs, offs, self._staged)

    def decompose_timed(self, segments, warmup, steps):
        """sd_decompose() `steps` times back to back from native code (libsd_bench.so: a loop around the C-ABI call, no
        Python between the calls); returns (seconds, records of the last call).  bench.py's end-to-end leg."""
        bl = C.CDLL(os.path.join(_HERE, "libsd_bench.so"))
        bl.sd_bench_decompose.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_int64), C.c_int64, C.c_int32, C.c_int32,
                                          C.POINTER(C.c_double), C.POINTER(C.c_int64)]
        bl.sd_bench_decompose.restype = C.c_int
        blob, off = segments if isinstance(segments, tuple) else _pack(segments)
        sec, nrec = C.c_double(), C.c_int64()
        st = bl.sd_bench_decompose(self._h, _text(blob), off.ctypes.data_as(C.POINTER(C.c_int64)), len(off) - 1, warmup, steps,
                                   C.byref(sec), C.byref(nrec))
        if st:
            self._err(st)
        return sec.value, nrec.value

    def set_ed_thr(self, ed_thr):
        """--ed_thr monomer pre-filter (FilterMonomersForRead, main.cpp:135-149); -1 switches it off."""
        st = self._lib.sd_set_ed_thr(self._h, ed_thr)
        if st:
            self._err(st)

    def stats(self):
        s = _Stats()
        self._lib.sd_get_stats(self._h, C.byref(s))
        d = {k: getattr(s, k) for k, _ in _Stats._fields_}
        d["dev_segments"] = [int(x) for x in d["dev_segments"]][:max(1, d["n_devices"])]
        return d

    def reset_stats(self):
        self._lib.sd_reset_stats(self._h)


def segment_read(read_len, part_size, overlap, flavour="cuda"):
    """AlignReadsSet segmentation (main.cpp:70-81): list of (offset, length)."""
    lib = load_library(flavour)
    n = lib.sd_segment_read(read_len, part_size, overlap, None, None, 0)
    if n < 0:
        raise SdError(1, "bad segmentation arguments")
    offs = np.zeros(max(n, 1), dtype=np.int64)
    lens = np.zeros(max(n, 1), dtype=np.int32)
    lib.sd_segment_read(read_len, part_size, overlap, offs.ctypes.data_as(C.POINTER(C.c_int64)),
                        lens.ctypes.data_as(C.POINTER(C.c_int32)), n)
    return [(int(offs[i]), int(lens[i])) for i in range(n)]


def postprocess(records, flavour="cuda"):
    """PostProcessing (main.cpp:287-302) on a structured array of read-relative records."""
    lib = load_library(flavour)
    rin = np.ascontiguousarray(records, dtype=RECORD_DTYPE)
    out = np.zeros(len(rin), dtype=RECORD_DTYPE)
    n = lib.sd_postprocess(rin.ctypes.data, len(rin), out.ctypes.data)
    return out[:n]


def run_files(reads_path, monomers_path, threads=1, part_size=5000, overlap=500, scoring=(-1, -1, -1, 1), ed_thr=-1,
              out_fd=1, err_fd=2, flavour="cuda"):
    lib = load_library(flavour)
    return lib.sd_run_files(str(reads_path).encode(), str(monomers_path).encode(), threads, part_size, overlap,
                            scoring[0], scoring[1], scoring[2], scoring[3], ed_thr, out_fd, err_fd)


def hw_distance(query, target, flavour="cuda"):
    """MonomerEditDistance (main.cpp:128-133): infix edit distance of query inside target."""
    return int(load_library(flavour).sd_hw_distance(query.encode(), len(query), target.encode(), len(target)))


def int_peak(device=0):
    """Measured integer-pipe issue rates (lane-ops/s): (ALU pipe only, ALU+FMA pipes, implied SM clock MHz)."""
    lib = load_library("cuda")
    a, b, m = C.c_double(), C.c_double(), C.c_double()
    st = lib.sd_int_peak(device, C.byref(a), C.byref(b), C.byref(m))
    if st:
        raise SdError(st, (lib.sd_last_error(None) or b"").decode())
    return a.value, b.value, m.value


def nw_identity(queries, targets, pairs=None, device=0, flavour="cuda"):
    """Batched edist/aai of the reference (main.py:29-60): for every (query, target) pair the edit distance, the number
    of '=' columns and the alignment length of edlib's global ("NW") alignment path.

    queries / targets: lists of str/bytes, or ``(blob, int64 offsets)`` tuples.  pairs: ``(query index array, target
    index array)`` or None for all queries x all targets (query-major).  Returns a dict of int32 arrays ``matches``,
    ``columns``, ``distance`` plus ``kernel_ms`` and ``hirschberg_pairs``; identity = 100 * matches / columns
    (0 where columns == 0)."""
    lib = load_library(flavour)
    qb, qo = queries if isinstance(queries, tuple) else _pack(queries)
    tb, to = targets if isinstance(targets, tuple) else _pack(targets)
    qo = np.ascontiguousarray(qo, dtype=np.int64)
    to = np.ascontiguousarray(to, dtype=np.int64)
    nq, nt = len(qo) - 1, len(to) - 1
    i32p, i64p = C.POINTER(C.c_int32), C.POINTER(C.c_int64)
    if pairs is None:
        n, pq, pt = nq * nt, None, None
    else:
        pq = np.ascontiguousarray(pairs[0], dtype=np.int32)
        pt = np.ascontiguousarray(pairs[1], dtype=np.int32)
        if pq.shape != pt.shape:
            raise SdError(1, "pairs: index arrays of different length")
        n = len(pq)
    m = np.zeros(n, dtype=np.int32)
    c = np.zeros(n, dtype=np.int32)
    d = np.zeros(n, dtype=np.int32)
    hb, ms = C.c_int64(0), C.c_double(0)
    st = lib.sd_identity(bytes(qb), qo.ctypes.data_as(i64p), nq, bytes(tb), to.ctypes.data_as(i64p), nt,
                         pq.ctypes.data_as(i32p) if pq is not None else None,
                         pt.ctypes.data_as(i32p) if pt is not None else None, n,
                         m.ctypes.data_as(i32p), c.ctypes.data_as(i32p), d.ctypes.data_as(i32p), device,
                         C.byref(hb), C.byref(ms))
    if st:
        raise SdError(st, (lib.sd_last_error(None) or b"").decode())
    return {"matches": m, "columns": c, "distance": d, "kernel_ms": ms.value, "hirschberg_pairs": hb.value}


def convert_raw(raw, reads, monomers, out_fd, alt_fd, min_identity=0, light=True, device=0, flavour="cuda"):
    """sd_convert: raw `dp` text -> final TSV on out_fd (and the `_alt` lines on alt_fd with light=False).
    reads: {id: sequence}; monomers: [(name, sequence)] in add_rc_monomers() order.  Returns the stage's counters."""
    lib = load_library(flavour)
    rb = raw.encode() if isinstance(raw, str) else bytes(raw)
    rn, rno = _pack(list(reads.keys()))
    rs, rso = _pack(list(reads.values()))
    mn, mno = _pack([m[0] for m in monomers])
    ms, mso = _pack([m[1] for m in monomers])
    i64p = C.POINTER(C.c_int64)
    st = _ConvertStats()
    rc = lib.sd_convert(rb, len(rb), rn, rno.ctypes.data_as(i64p), rs, rso.ctypes.data_as(i64p), len(reads),
                        mn, mno.ctypes.data_as(i64p), ms, mso.ctypes.data_as(i64p), len(monomers),
                        int(min_identity), 1 if light else 0, device, out_fd, alt_fd, C.byref(st))
    if rc:
        msg = (lib.sd_convert_error() or b"").decode()
        if msg.startswith("KeyError"):
            raise KeyError(msg)
        raise SdError(rc, msg)
    return {k: getattr(st, k) for k, _ in _ConvertStats._fields_}
