"""ctypes binding of libmotifs_b200.so (C ABI declared in include/motifs_b200.h).

This is the same surface a Julia host binds with `ccall` (INTEGRATION.md); nothing here computes
anything — it marshals numpy arrays to plain pointers and raises on error codes.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))


def library_path() -> str:
    # MB200_LIBRARY: another build of the same ABI (A/B measurements of kernel changes on one box)
    return os.environ.get("MB200_LIBRARY") or os.path.join(_HERE, "lib", "libmotifs_b200.so")


class MB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libmotifs_b200 error {code}: {msg}")
        self.code = code


OK, E_INVALID, E_CUDA, E_NOMEM, E_BAD_SEQUENCE, E_HITS_OVERFLOW, E_UNSUPPORTED, E_COMM = 0, -1, -2, -3, -4, -5, -6, -7
SCAN_FWD, SCAN_RC, SCAN_WANT_HITS, SCAN_WANT_COUNTS, SCAN_NO_TENSOR, SCAN_REDUCE = 1, 2, 4, 8, 16, 32
COMM_ID_BYTES = 128
MAX_MOTIF_LEN = 64

HIT_DTYPE = np.dtype([("seq", "<u4"), ("pos", "<u4"), ("motif", "<u2"), ("score_f16", "<u2"),
                      ("comp", "u1"), ("_pad", "u1", (3,))])
assert HIT_DTYPE.itemsize == 16

BEST_DTYPE = np.dtype([("pos", "<u4"), ("score_f16", "<u2"), ("comp", "u1"), ("found", "u1")])
assert BEST_DTYPE.itemsize == 8

ANCHOR_DTYPE = np.dtype([("row", "<i8"), ("start", "<i8"), ("len", "<i4"), ("primary", "<u2"), ("comp", "u1"), ("_pad", "u1")])
assert ANCHOR_DTYPE.itemsize == 24

SITE_DTYPE = np.dtype([("motif", "<u4"), ("seq", "<u4"), ("pos", "<u4"), ("comp", "<u4")])
CODE_DTYPE = np.dtype([("position", "<u2"), ("fil", "<u2"), ("seq", "<u4"), ("mag_f16", "<u2"), ("_pad", "<u2")])
assert CODE_DTYPE.itemsize == 12
KEYCOUNT_DTYPE = np.dtype([("key", "<u8"), ("count", "<u4"), ("reserved", "<u4"), ("first", "<u8")])
TRIPVAL_DTYPE = np.dtype([("key_index", "<u4"), ("range_index", "<u4"), ("position", "<u4"), ("reserved", "<u4"), ("order", "<u8")])
assert KEYCOUNT_DTYPE.itemsize == 24 and TRIPVAL_DTYPE.itemsize == 24


class HParams(C.Structure):
    """mb200_hparams = Hyperparam (model.jl:1-14)."""
    _fields_ = [("filter_len", C.c_int32), ("M", C.c_int32), ("h", C.c_int32), ("K", C.c_int32), ("q", C.c_int32),
                ("batch_size", C.c_int32), ("num_pass_xyz", C.c_int32), ("num_pass_df", C.c_int32),
                ("magnifying_factor", C.c_float), ("gamma", C.c_float)]


_lib = None


def load():
    """dlopen the library; fails loudly when it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise MB200Error(E_UNSUPPORTED, f"{path} not built: run `python -c 'import __graft_entry__ as g; g.build()'` or `make`")
    lib = C.CDLL(path)
    p, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    sig = {
        "mb200_version": (i32, []),
        "mb200_create": (i32, [C.POINTER(p), i32]),
        "mb200_destroy": (i32, [p]),
        "mb200_last_error": (C.c_char_p, [p]),
        "mb200_set_stream": (i32, [p, p]),
        "mb200_last_timing": (i32, [p, p, p]),
        "mb200_comm_unique_id": (i32, [p]),
        "mb200_comm_init": (i32, [p, p, i32, i32]),
        "mb200_comm_destroy": (i32, [p]),
        "mb200_comm_info": (i32, [p, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
        "mb200_comm_broadcast": (i32, [p, p, i64, i32]),
        "mb200_comm_allreduce_i64": (i32, [p, p, i64]),
        "mb200_comm_allgather": (i32, [p, p, p, i64]),
        "mb200_seqs_from_ascii": (i32, [p, p, i64, i64, C.POINTER(p)]),
        "mb200_seqs_from_ascii_async": (i32, [p, p, i64, i64, C.POINTER(p)]),
        "mb200_seqs_wait": (i32, [p, p]),
        "mb200_seqs_from_device_ascii": (i32, [p, p, i64, i64, C.POINTER(p)]),
        "mb200_seqs_from_onehot_f32": (i32, [p, p, i64, i64, C.POINTER(p)]),
        "mb200_seqs_from_ascii_ragged": (i32, [p, p, p, i64, C.POINTER(p)]),
        "mb200_seqs_lengths": (i32, [p, p]),
        "mb200_seqs_free": (i32, [p, p]),
        "mb200_seqs_shape": (i32, [p, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
        "mb200_seqs_download": (i32, [p, p, p, i64]),
        "mb200_fasta_read": (i32, [C.c_char_p, i64, C.POINTER(p), C.POINTER(i64), C.POINTER(i64)]),
        "mb200_fasta_rows": (i32, [p, p]),
        "mb200_fasta_free": (i32, [p]),
        "mb200_records_read": (i32, [C.c_char_p, C.POINTER(p)]),
        "mb200_records_counts": (i32, [p, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
        "mb200_records_names": (i32, [p, p, p]),
        "mb200_records_fragments": (i32, [p, p, p, p, p]),
        "mb200_records_free": (i32, [p]),
        "mb200_fasta_split": (i32, [i64, C.c_double, i32, C.c_uint64, p, p, C.POINTER(i64), C.POINTER(i64)]),
        "mb200_seqs_gather": (i32, [p, p, p, i64, C.POINTER(p)]),
        "mb200_seqs_windows": (i32, [p, p, p, p, i64, i64, C.POINTER(p)]),
        "mb200_seqs_shuffle": (i32, [p, p, i32, C.c_uint64, i64, C.POINTER(p)]),
        "mb200_seqs_base_counts": (i32, [p, p, p, p]),
        "mb200_seqs_to_ascii": (i32, [p, p, p]),
        "mb200_scan": (i32, [p, p, p, p, i32, i32, p, C.c_uint32, p, i64, C.POINTER(i64), p]),
        "mb200_scan_take_hits": (i32, [p, p, i64, C.POINTER(i64)]),
        "mb200_scan_last_path": (i32, [p]),
        "mb200_scan_prefilter_bound": (i32, [p, i32, C.c_uint16, p, p, p, p]),
        "mb200_scan_hist": (i32, [p, p, p, p, i32, i32, C.c_uint32, p]),
        "mb200_scan_best": (i32, [p, p, p, p, i32, i32, C.c_uint32, p]),
        "mb200_scan_spacing": (i32, [p, p, p, i64, i32, i32, p, p, i32, i32, p, p, p]),
        "mb200_csc_create": (i32, [p, C.POINTER(HParams), i64, i32, i32, C.POINTER(p)]),
        "mb200_csc_destroy": (i32, [p, p]),
        "mb200_csc_n_params": (i32, [p, C.POINTER(i64), C.POINTER(i64)]),
        "mb200_csc_set_params": (i32, [p, p, p, i64]),
        "mb200_csc_get_params": (i32, [p, p, p, i64]),
        "mb200_csc_reset_optimizer": (i32, [p, p]),
        "mb200_csc_get_grads": (i32, [p, p, p, i64]),
        "mb200_csc_device_ptrs": (i32, [p, C.POINTER(p), C.POINTER(p)]),
        "mb200_csc_broadcast_params": (i32, [p, p, i32]),
        "mb200_csc_codes_sharded": (i32, [p, p, p, i64, i64, i32, i32, p, i64, C.POINTER(i64)]),
        "mb200_csc_loss_grad": (i32, [p, p, p, p, p, p]),
        "mb200_csc_step_begin": (i32, [p, p, p, p]),
        "mb200_csc_step_begin_host": (i32, [p, p, p, i64]),
        "mb200_csc_adabelief_step": (i32, [p, p, C.c_float, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
        "mb200_csc_get_buffer": (i32, [p, p, C.c_char_p, p, i64]),
        "mb200_csc_median_mask": (i32, [p, p, p, p, p, p]),
        "mb200_csc_codes": (i32, [p, p, p, i64, i64, p, i64, C.POINTER(i64)]),
        "mb200_count_matrices": (i32, [p, p, p, i64, p, i32, i32, p]),
        "mb200_pvalue2score": (i32, [p, p, i32, C.c_double, C.c_double, p, p, p]),
        "mb200_triplets_create": (i32, [p, p, p, p, i64, p, p, p]),
        "mb200_triplets_destroy": (i32, [p, p]),
        "mb200_triplets_ranges": (i32, [p, p, p, p]),
        "mb200_triplets_frequent": (i32, [p, p, C.c_uint32, p, i64, p]),
        "mb200_triplets_values": (i32, [p, p, p, i64, p, i64, p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    """One CUDA device + stream (mb200_ctx).  Not thread-safe."""

    def __init__(self, device: int = 0):
        self._lib = load()
        h = C.c_void_p()
        rc = self._lib.mb200_create(C.byref(h), int(device))
        if rc != OK:
            raise MB200Error(rc, "mb200_create failed (no CUDA device / not a B200-class GPU?)")
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.mb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != OK:
            raise MB200Error(rc, self._lib.mb200_last_error(self._h).decode())

    def set_stream(self, cuda_stream_ptr):
        self._check(self._lib.mb200_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)))

    def last_timing(self):
        ms = np.zeros(8, np.float32)
        n = np.zeros(8, np.int64)
        self._check(self._lib.mb200_last_timing(self._h, _ptr(ms), _ptr(n)))
        names = ["pack", "scan", "count", "emit", "csc", "h2d", "d2h", "total"]
        return {k: float(v) for k, v in zip(names, ms)}, {k: int(v) for k, v in zip(names, n)}

    # ---- multi-GPU (csrc/comm.cu): one NCCL communicator per ctx, created from a 128-byte id that rank 0 hands out --------
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (C.c_uint8 * COMM_ID_BYTES)()
        rc = load().mb200_comm_unique_id(buf)
        if rc != OK:
            raise MB200Error(rc, "mb200_comm_unique_id failed (libnccl.so.2 not loadable?)")
        return bytes(buf)

    def comm_init(self, unique_id: bytes, rank: int, world: int):
        if len(unique_id) != COMM_ID_BYTES:
            raise ValueError("unique_id must be 128 bytes (mb200_comm_unique_id)")
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(unique_id)
        self._check(self._lib.mb200_comm_init(self._h, buf, int(rank), int(world)))

    def comm_destroy(self):
        self._check(self._lib.mb200_comm_destroy(self._h))

    def comm_info(self):
        r, w, v = C.c_int32(), C.c_int32(), C.c_int32()
        self._check(self._lib.mb200_comm_info(self._h, C.byref(r), C.byref(w), C.byref(v)))
        return r.value, w.value, v.value

    @property
    def rank(self):
        return self.comm_info()[0]

    @property
    def world(self):
        return self.comm_info()[1]

    def comm_broadcast(self, arr: np.ndarray, root: int = 0) -> np.ndarray:
        """in-place broadcast of a contiguous numpy array from `root` (blocking, collective)."""
        assert arr.flags.c_contiguous
        self._check(self._lib.mb200_comm_broadcast(self._h, _ptr(arr), arr.nbytes, int(root)))
        return arr

    def comm_allreduce_i64(self, arr: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(arr, np.int64)
        self._check(self._lib.mb200_comm_allreduce_i64(self._h, _ptr(a), a.size))
        return a

    def comm_allgather(self, arr: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(arr)
        out = np.zeros((self.world,) + a.shape, a.dtype)
        self._check(self._lib.mb200_comm_allgather(self._h, _ptr(a), _ptr(out), a.nbytes))
        return out

    # ---- sequences ---------------------------------------------------------------------------
    def seqs_from_ascii(self, ascii_rows: np.ndarray) -> "Sequences":
        a = np.ascontiguousarray(ascii_rows, dtype=np.uint8)
        if a.ndim != 2:
            raise ValueError("ascii_rows must be (N, Lb) uint8")
        h = C.c_void_p()
        self._check(self._lib.mb200_seqs_from_ascii(self._h, _ptr(a), a.shape[0], a.shape[1], C.byref(h)))
        return Sequences(self, h, a.shape[0], a.shape[1])

    def seqs_from_ragged(self, ascii: np.ndarray, offsets) -> "Sequences":
        """Rows of different lengths: row i = ascii[offsets[i]:offsets[i+1]] (mb200_seqs_from_ascii_ragged).  `ascii` is the
        concatenated uint8 bases (or a bytes object), offsets N+1 non-decreasing int64.  Lb of the store = the longest row."""
        a = np.frombuffer(ascii, np.uint8) if isinstance(ascii, (bytes, bytearray)) else np.ascontiguousarray(ascii, np.uint8).reshape(-1)
        off = np.ascontiguousarray(offsets, np.int64)
        if off.ndim != 1 or len(off) < 1:
            raise ValueError("offsets must be N+1 int64 values")
        if len(off) > 1 and (off[0] < 0 or off[-1] > a.size):
            raise ValueError("offsets must lie inside ascii")
        h = C.c_void_p()
        self._check(self._lib.mb200_seqs_from_ascii_ragged(self._h, _ptr(a), _ptr(off), len(off) - 1, C.byref(h)))
        N, Lb = C.c_int64(), C.c_int64()
        self._lib.mb200_seqs_shape(h, C.byref(N), C.byref(Lb), None)
        return Sequences(self, h, N.value, Lb.value)

    def seqs_from_host_ptr(self, ptr: int, N: int, Lb: int, wait: bool = True) -> "Sequences":
        """ASCII rows at a raw host address (e.g. a pinned torch tensor's data_ptr()).  wait=False: the upload is queued on the
        ctx's copy stream and overlaps the first scan of these sequences (mb200_seqs_from_ascii_async); the caller keeps the host
        buffer alive until that scan or Sequences.wait() has returned."""
        h = C.c_void_p()
        fn = self._lib.mb200_seqs_from_ascii if wait else self._lib.mb200_seqs_from_ascii_async
        self._check(fn(self._h, C.c_void_p(ptr), N, Lb, C.byref(h)))
        return Sequences(self, h, N, Lb)

    def seqs_from_device_ptr(self, ptr: int, N: int, Lb: int) -> "Sequences":
        h = C.c_void_p()
        self._check(self._lib.mb200_seqs_from_device_ascii(self._h, C.c_void_p(ptr), N, Lb, C.byref(h)))
        return Sequences(self, h, N, Lb)

    def seqs_from_onehot(self, onehot: np.ndarray) -> "Sequences":
        """onehot: the reference's data_matrix, Float32 (4*Lb, 1, N) or (4*Lb, N), Fortran (Julia) order,
        i.e. a C-order numpy array of shape (N, 4*Lb) / (N, Lb, 4)."""
        a = np.ascontiguousarray(onehot, dtype=np.float32)
        a = a.reshape(a.shape[0], -1)
        if a.shape[1] % 4:
            raise ValueError("one-hot rows must have 4*Lb entries")
        h = C.c_void_p()
        self._check(self._lib.mb200_seqs_from_onehot_f32(self._h, _ptr(a), a.shape[0], a.shape[1] // 4, C.byref(h)))
        return Sequences(self, h, a.shape[0], a.shape[1] // 4)

    # ---- scan --------------------------------------------------------------------------------
    @staticmethod
    def _pwm_arrays(pwms_f16, lens):
        pw = np.ascontiguousarray(pwms_f16)
        if pw.dtype == np.float16:
            pw = pw.view(np.uint16)
        if pw.dtype != np.uint16 or pw.ndim != 3 or pw.shape[1] != 4:
            raise ValueError("pwms_f16 must be float16/uint16 of numpy shape (maxlen, 4, K)")
        ln = np.ascontiguousarray(lens, dtype=np.int64)
        if ln.shape != (pw.shape[2],):
            raise ValueError("lens must have K entries")
        return pw, ln

    def scan(self, seqs: "Sequences", pwms_f16: np.ndarray, lens, thresh_f16=None, *, fwd=True, rc=True,
             want_hits=True, want_counts=True, hits_cap=None, tensor=True, reduce=False):
        """pwms_f16: (K, 4, maxlen) array in Julia memory order, i.e. numpy shape (maxlen, 4, K) C-order
        holding float16 (or uint16 bits).  Returns (hits structured array | None, counts (K,4) int64 | None).
        tensor=False keeps a thresholded scan on the SIMT kernel (MB200_SCAN_NO_TENSOR); results are identical either way.
        reduce=True: counts are summed over the ranks of the ctx's communicator inside the call (MB200_SCAN_REDUCE)."""
        pw, ln = self._pwm_arrays(pwms_f16, lens)
        maxlen, _, K = pw.shape
        th = None
        if thresh_f16 is not None:
            th = np.ascontiguousarray(thresh_f16)
            if th.dtype == np.float16:
                th = th.view(np.uint16)
            if th.dtype != np.uint16 or th.shape != (K,):
                raise ValueError("thresh_f16 must be K float16/uint16 values")
        flags = (SCAN_FWD if fwd else 0) | (SCAN_RC if rc else 0) | (SCAN_WANT_HITS if want_hits else 0) | \
                (SCAN_WANT_COUNTS if want_counts else 0) | (0 if tensor else SCAN_NO_TENSOR) | (SCAN_REDUCE if reduce else 0)
        counts = np.zeros((K, 4), np.int64) if want_counts else None
        n_hits = C.c_int64(0)
        cap = int(hits_cap) if hits_cap is not None else (1 << 16)
        hits = np.zeros(cap if want_hits else 0, HIT_DTYPE)
        rc_ = self._lib.mb200_scan(self._h, seqs._h, _ptr(pw), _ptr(ln), K, maxlen, _ptr(th), flags,
                                   _ptr(hits) if want_hits else None, cap if want_hits else 0,
                                   C.byref(n_hits), _ptr(counts))
        if rc_ == E_HITS_OVERFLOW and hits_cap is None:
            # the library kept the complete list: fetch it instead of scanning again (counts are already final)
            hits = np.zeros(int(n_hits.value), HIT_DTYPE)
            rc_ = self._lib.mb200_scan_take_hits(self._h, _ptr(hits), len(hits), C.byref(n_hits))
        self._check(rc_)
        return (hits[: n_hits.value] if want_hits else None), counts

    def scan_best(self, seqs: "Sequences", pwms_f16: np.ndarray, lens, *, fwd=True, rc=True) -> np.ndarray:
        """Best site of every (row, motif) (mb200_scan_best): (N, K) BEST_DTYPE array {pos, score_f16, comp, found}.  pwms_f16 and
        lens as for scan.  Highest score, then lowest position, then the forward strand; found = 0 (pos = 2**32 - 1) when the row
        has no window of the motif on the requested strands or every window is NaN."""
        pw, ln = self._pwm_arrays(pwms_f16, lens)
        maxlen, _, K = pw.shape
        out = np.empty((seqs.N, K), BEST_DTYPE)                   # every record is written
        flags = (SCAN_FWD if fwd else 0) | (SCAN_RC if rc else 0)
        self._check(self._lib.mb200_scan_best(self._h, seqs._h, _ptr(pw), _ptr(ln), K, maxlen, flags, _ptr(out)))
        return out

    def seqs_windows(self, seqs: "Sequences", rows, starts, length: int) -> "Sequences":
        """mb200_seqs_windows: a new fixed-length store whose row i holds bases [starts[i], starts[i] + length) of row rows[i] of
        seqs (fixed or ragged)."""
        r = np.ascontiguousarray(rows, np.int64)
        s = np.ascontiguousarray(starts, np.int64)
        if r.shape != s.shape or r.ndim != 1:
            raise ValueError("rows and starts must be 1-D arrays of one length")
        h = C.c_void_p()
        self._check(self._lib.mb200_seqs_windows(self._h, seqs._h, _ptr(r), _ptr(s), len(r), int(length), C.byref(h)))
        return Sequences(self, h, len(r), int(length))

    def scan_spacing(self, seqs: "Sequences", anchors, n_primary: int, pwms_f16: np.ndarray, lens, thresh=None, *, margin: int,
                     want_sites: bool = False):
        """mb200_scan_spacing: (hist (n_primary, K, 4, margin) uint32, sites (n_anchors, K) BEST_DTYPE or None).  anchors:
        ANCHOR_DTYPE array (row, start, len, primary, comp) of primary sites in rows of seqs; pwms_f16 and lens: the K secondaries
        as for scan; thresh: K Float16 thresholds or None (a counted site needs score > 0 and > thresh).  hist[p, k, q, g] counts
        the anchors of primary p whose best site of k in the two margins is counted and lies at gap g in quadrant q (0: same strand
        upstream, 1: same strand downstream, 2: opposite upstream, 3: opposite downstream, in the primary's orientation)."""
        pw, ln = self._pwm_arrays(pwms_f16, lens)
        maxlen, _, K = pw.shape
        an = np.ascontiguousarray(anchors, ANCHOR_DTYPE)
        th = None
        if thresh is not None:
            th = np.ascontiguousarray(thresh)
            if th.dtype != np.uint16:
                th = np.ascontiguousarray(th, np.float16).view(np.uint16)
            if th.shape != (K,):
                raise ValueError("thresh must hold K float16 values")
        hist = np.zeros((int(n_primary), K, 4, int(margin)), np.uint32) if 0 < n_primary and 0 < margin else np.zeros(1, np.uint32)
        sites = np.empty((len(an), K), BEST_DTYPE) if want_sites else None
        self._check(self._lib.mb200_scan_spacing(self._h, seqs._h, _ptr(an), len(an), int(n_primary), int(margin), _ptr(pw), _ptr(ln),
                                                  K, maxlen, _ptr(th), _ptr(hist), _ptr(sites)))
        return hist, sites


def fasta_read(path: str, max_entries: int = 100000) -> np.ndarray:
    """mb200_fasta_read: (N, L) uint8 matrix of the reads the reference's read_fasta keeps (helpers.jl:83-108)."""
    h, n, l = C.c_void_p(), C.c_int64(), C.c_int64()
    rc = load().mb200_fasta_read(os.fsencode(path), int(max_entries), C.byref(h), C.byref(n), C.byref(l))
    if rc != OK:
        raise MB200Error(rc, f"mb200_fasta_read({path}) failed")
    out = np.zeros((n.value, l.value), np.uint8)
    try:
        if out.size:
            load().mb200_fasta_rows(h, _ptr(out))
    finally:
        load().mb200_fasta_free(h)
    return out


def fasta_split(n: int, ratio: float, shuffle: bool, seed: int):
    """mb200_fasta_split: 0-based (train_idx, test_idx) following get_train_test_inds (helpers.jl:141-159)."""
    tr, te = np.zeros(max(n, 1), np.int64), np.zeros(max(n, 1), np.int64)
    ntr, nte = C.c_int64(), C.c_int64()
    rc = load().mb200_fasta_split(int(n), float(ratio), int(bool(shuffle)), C.c_uint64(int(seed) & (2 ** 64 - 1)), _ptr(tr), _ptr(te), C.byref(ntr), C.byref(nte))
    if rc != OK:
        raise MB200Error(rc, "mb200_fasta_split failed")
    return tr[: ntr.value].copy(), te[: nte.value].copy()


def scan_last_path(ctx: "Context") -> int:
    """0: the last mb200_scan ran scan_kernel (SIMT), 1: tensor-core pre-filter + exact re-scoring, 2: started on the tensor-core
    path and fell back (candidate list overflow)."""
    return int(ctx._lib.mb200_scan_last_path(ctx._h))


def scan_prefilter_bound(cols_f16, thresh_f16):
    """mb200_scan_prefilter_bound: (E, t', column 0 of the B operand as float16[4], possible) for one slot; cols_f16: (len, 4)."""
    c = np.ascontiguousarray(cols_f16, np.float16).view(np.uint16)
    E, tp, ok = C.c_double(), C.c_double(), C.c_int32()
    col0 = np.zeros(4, np.uint16)
    rc = load().mb200_scan_prefilter_bound(_ptr(c), c.shape[0], int(np.float16(thresh_f16).view(np.uint16)), C.byref(E), C.byref(tp), _ptr(col0), C.byref(ok))
    if rc != 0:
        raise ValueError(f"mb200_scan_prefilter_bound failed ({rc})")
    return E.value, tp.value, col0.view(np.float16), bool(ok.value)


def count_matrices(ctx: "Context", seqs: "Sequences", sites, lens):
    """sites: structured array (motif, seq, pos, comp), 0-based -> list of (4, len_k) uint32 count matrices."""
    st = np.ascontiguousarray(sites, SITE_DTYPE)
    ln = np.ascontiguousarray(lens, np.int64)
    K, maxlen = len(ln), int(ln.max())
    out = np.zeros((K, maxlen, 4), np.uint32)
    ctx._check(ctx._lib.mb200_count_matrices(ctx._h, seqs._h, _ptr(st), len(st), _ptr(ln), K, maxlen, _ptr(out)))
    return [out[k, : ln[k]].T.copy() for k in range(K)]


def scan_hist(ctx: "Context", seqs: "Sequences", pwms_f16, lens, fwd=True, rc=True, reduce=False):
    """(K, 32768) uint32 histogram of the Float16 bit patterns of all hit scores (score > 0)."""
    pw = np.ascontiguousarray(pwms_f16)
    if pw.dtype == np.float16:
        pw = pw.view(np.uint16)
    maxlen, _, K = pw.shape
    ln = np.ascontiguousarray(lens, dtype=np.int64)
    out = np.zeros((K, 32768), np.uint32)
    flags = (SCAN_FWD if fwd else 0) | (SCAN_RC if rc else 0) | (SCAN_REDUCE if reduce else 0)
    ctx._check(ctx._lib.mb200_scan_hist(ctx._h, seqs._h, _ptr(pw), _ptr(ln), K, maxlen, flags, _ptr(out)))
    return out


class Sequences:
    """2 bit/base packed sequences resident in HBM (mb200_seqs)."""

    def __init__(self, ctx: Context, handle, N, Lb):
        self.ctx, self._h, self.N, self.Lb = ctx, handle, int(N), int(Lb)

    @property
    def words_per_seq(self):
        return (self.Lb + 15) // 16

    def download(self) -> np.ndarray:
        out = np.zeros((self.N, self.words_per_seq), np.uint32)
        self.ctx._check(self.ctx._lib.mb200_seqs_download(self.ctx._h, self._h, _ptr(out), out.size))
        return out

    @property
    def lengths(self) -> np.ndarray:
        """(N,) int64 row lengths (all Lb for a fixed-length store)."""
        out = np.zeros(self.N, np.int64)
        rc = self.ctx._lib.mb200_seqs_lengths(self._h, _ptr(out))
        if rc != OK:
            raise MB200Error(rc, "mb200_seqs_lengths failed")
        return out

    def gather(self, idx) -> "Sequences":
        """rows idx of this store as a new store (device gather)."""
        i = np.ascontiguousarray(idx, np.int64)
        h = C.c_void_p()
        self.ctx._check(self.ctx._lib.mb200_seqs_gather(self.ctx._h, self._h, _ptr(i), len(i), C.byref(h)))
        return Sequences(self.ctx, h, len(i), self.Lb)

    def shuffle(self, k: int, seed: int, first_stream: int = 0) -> "Sequences":
        """seq_shuffle.(reads; k): k-mer-count-preserving shuffle of every sequence on the device, from a host seed.  Row i draws
        from random stream first_stream + i; rows of a ragged store keep their lengths and zero padding."""
        h = C.c_void_p()
        self.ctx._check(self.ctx._lib.mb200_seqs_shuffle(self.ctx._h, self._h, int(k), C.c_uint64(int(seed) & (2 ** 64 - 1)), int(first_stream), C.byref(h)))
        return Sequences(self.ctx, h, self.N, self.Lb)

    def base_counts(self):
        """(counts[4] of A,C,G,T, transitions[4,4] base a -> base b) as int64."""
        c, t = np.zeros(4, np.int64), np.zeros((4, 4), np.int64)
        self.ctx._check(self.ctx._lib.mb200_seqs_base_counts(self.ctx._h, self._h, _ptr(c), _ptr(t)))
        return c, t

    def to_ascii(self) -> np.ndarray:
        """(N, Lb) uint8 "ACGT" rows; bytes past a row's length (ragged stores) are 0."""
        out = np.zeros((self.N, self.Lb), np.uint8)
        self.ctx._check(self.ctx._lib.mb200_seqs_to_ascii(self.ctx._h, self._h, _ptr(out)))
        return out

    def wait(self):
        """block until an asynchronous upload has finished (raises MB200Error on symbols other than A,C,G,T)."""
        self.ctx._check(self.ctx._lib.mb200_seqs_wait(self.ctx._h, self._h))

    def free(self):
        if self._h and self.ctx._h:
            self.ctx._lib.mb200_seqs_free(self.ctx._h, self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class CscModel:
    """mb200_csc: the unrolled CSC network for one (hyper-parameters, Lb, n_groups) shape on one device."""

    def __init__(self, ctx: Context, hp, Lb: int, n_groups: int = 1, forward_only: bool = False, tensor_cores: bool = False, fused: bool = True, fused_df: bool = True):
        self.ctx = ctx
        self.hp = hp
        self.Lb, self.n_groups, self.forward_only = int(Lb), int(n_groups), bool(forward_only)
        chp = HParams(hp.filter_len, hp.M, hp.h, hp.K, hp.q, hp.batch_size, hp.num_pass_xyz, hp.num_pass_df,
                      float(hp.magnifying_factor), float(hp.gamma))
        h = C.c_void_p()
        if tensor_cores and not forward_only:
            raise ValueError("the tensor-core path is forward-only (code retrieval)")
        ctx._check(ctx._lib.mb200_csc_create(ctx._h, C.byref(chp), self.Lb, self.n_groups, (2 if tensor_cores else int(self.forward_only)) | (0 if fused else 0x100) | (0 if fused_df else 0x200), C.byref(h)))
        self._h = h
        nt, na = C.c_int64(), C.c_int64()
        ctx._check(ctx._lib.mb200_csc_n_params(self._h, C.byref(nt), C.byref(na)))
        self.n_trainable, self.n_total = nt.value, na.value
        self.batch = hp.batch_size * self.n_groups

    def free(self):
        if getattr(self, "_h", None) and self.ctx._h:
            self.ctx._lib.mb200_csc_destroy(self.ctx._h, self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def set_params(self, flat):
        a = np.ascontiguousarray(flat, np.float32)
        self.ctx._check(self.ctx._lib.mb200_csc_set_params(self.ctx._h, self._h, _ptr(a), a.size))

    def get_params(self):
        a = np.zeros(self.n_total, np.float32)
        self.ctx._check(self.ctx._lib.mb200_csc_get_params(self.ctx._h, self._h, _ptr(a), a.size))
        return a

    def get_grads(self):
        a = np.zeros(self.n_trainable, np.float32)
        self.ctx._check(self.ctx._lib.mb200_csc_get_grads(self.ctx._h, self._h, _ptr(a), a.size))
        return a

    def reset_optimizer(self):
        self.ctx._check(self.ctx._lib.mb200_csc_reset_optimizer(self.ctx._h, self._h))

    def device_ptrs(self):
        a, b = C.c_void_p(), C.c_void_p()
        self.ctx._check(self.ctx._lib.mb200_csc_device_ptrs(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def broadcast_params(self, root: int = 0):
        """rank `root`'s parameters + AdaBelief state become every rank's (collective; no-op without a communicator)."""
        self.ctx._check(self.ctx._lib.mb200_csc_broadcast_params(self.ctx._h, self._h, int(root)))

    def loss_grad(self, seqs: "Sequences", seq_idx, want_grads=True):
        idx = np.ascontiguousarray(seq_idx, np.int64)
        if idx.size != self.batch:
            raise ValueError(f"need {self.batch} sequence indices")
        loss = np.zeros((self.n_groups, 3), np.float32)
        g = np.zeros(self.n_trainable, np.float32) if want_grads else None
        self.ctx._check(self.ctx._lib.mb200_csc_loss_grad(self.ctx._h, self._h, seqs._h, _ptr(idx), _ptr(loss), _ptr(g)))
        return loss, g

    def step_begin(self, seqs: "Sequences", seq_idx):
        idx = np.ascontiguousarray(seq_idx, np.int64)
        if idx.size != self.batch:
            raise ValueError(f"need {self.batch} sequence indices")
        self.ctx._check(self.ctx._lib.mb200_csc_step_begin(self.ctx._h, self._h, seqs._h, _ptr(idx)))

    def step_begin_host(self, ascii_rows):
        """batch handed over as host ASCII rows (batch x Lb uint8, or a raw host address for pinned buffers)."""
        if isinstance(ascii_rows, int):
            self.ctx._check(self.ctx._lib.mb200_csc_step_begin_host(self.ctx._h, self._h, C.c_void_p(ascii_rows), self.batch))
            return
        a = np.ascontiguousarray(ascii_rows, np.uint8)
        if a.shape != (self.batch, self.Lb):
            raise ValueError(f"need a ({self.batch}, {self.Lb}) uint8 array")
        self.ctx._check(self.ctx._lib.mb200_csc_step_begin_host(self.ctx._h, self._h, _ptr(a), self.batch))

    def adabelief_step(self, eta=1e-3, beta1=0.9, beta2=0.999, eps=1e-8):
        loss, l1 = C.c_float(), C.c_float()
        self.ctx._check(self.ctx._lib.mb200_csc_adabelief_step(self.ctx._h, self._h, eta, beta1, beta2, eps, C.byref(loss), C.byref(l1)))
        return loss.value, l1.value

    def get_buffer(self, name: str, n: int):
        a = np.zeros(int(n), np.float32)
        self.ctx._check(self.ctx._lib.mb200_csc_get_buffer(self.ctx._h, self._h, name.encode(), _ptr(a), a.size))
        return a

    def median_mask(self, z, y):
        """cat_ZY + create_ZY_mask (model.jl:194-210) alone: z,y (G, B*c, M) float32 -> zy (G, B*c, 2M), med (G,)."""
        z = np.ascontiguousarray(z, np.float32); y = np.ascontiguousarray(y, np.float32)
        G, rows, M = z.shape
        if y.shape != z.shape or G != self.n_groups or M != self.hp.M:
            raise ValueError("z,y must be (n_groups, batch*c, M)")
        zy = np.zeros((G, rows, 2 * M), np.float32); med = np.zeros(G, np.float32)
        self.ctx._check(self.ctx._lib.mb200_csc_median_mask(self.ctx._h, self._h, _ptr(z), _ptr(y), _ptr(zy), _ptr(med)))
        return zy, med

    def codes(self, seqs: "Sequences", first_seq=0, n_seqs=None, shard=None):
        """shard=None: this GPU decodes everything.  shard="comm": the ranks of the ctx's communicator each decode a contiguous
        range of whole batches and all-gather the records (every rank returns the full result).  shard=(rank, world): only that
        shard, no communication."""
        B = self.hp.batch_size
        if n_seqs is None:
            n_seqs = (seqs.N - first_seq) - (seqs.N - first_seq) % B          # DataLoader(partial=false)
        cap = max(1024, 64 * int(n_seqs))
        n = C.c_int64()
        while True:
            out = np.zeros(cap, CODE_DTYPE)
            if shard is None:
                rc = self.ctx._lib.mb200_csc_codes(self.ctx._h, self._h, seqs._h, int(first_seq), int(n_seqs), _ptr(out), cap, C.byref(n))
            else:
                r, w = (-1, -1) if shard == "comm" else shard
                rc = self.ctx._lib.mb200_csc_codes_sharded(self.ctx._h, self._h, seqs._h, int(first_seq), int(n_seqs), int(r), int(w),
                                                           _ptr(out), cap, C.byref(n))
            if rc == E_HITS_OVERFLOW and n.value > cap:      # more codes than the guess (large q, ties): decode again into the reported size
                cap = int(n.value)
                continue
            self.ctx._check(rc)
            return out[: n.value]


def pvalue2score(ctx: "Context", pwm, pval, eps, bg):
    """mb200_pvalue2score: Touzet p-value -> score of a (4, m) PWM segment in Float64; None when no score qualifies."""
    p = np.ascontiguousarray(pwm, np.float64)
    b = np.ascontiguousarray(bg, np.float64)
    score, found = C.c_double(), C.c_int32()
    if ctx is None:                                     # host arithmetic only: usable without a context
        rc = load().mb200_pvalue2score(None, _ptr(p), p.shape[1], float(pval), float(eps), _ptr(b), C.byref(score), C.byref(found))
        if rc != 0:
            raise ValueError(f"mb200_pvalue2score failed ({rc})")
    else:
        ctx._check(ctx._lib.mb200_pvalue2score(ctx._h, _ptr(p), p.shape[1], float(pval), float(eps), _ptr(b), C.byref(score), C.byref(found)))
    return score.value if found.value else None


class Triplets:
    """mb200_triplets: the triplet dictionary of one set of filtered code components, resident on the device
    (enumerate_triplets / insert_H!, inference/_2_enumerate.jl:25-65)."""

    def __init__(self, ctx: "Context", codes):
        self.ctx = ctx
        pos = np.ascontiguousarray(codes["position"], np.uint16)
        fil = np.ascontiguousarray(codes["fil"], np.uint16)
        seq = np.ascontiguousarray(codes["seq"], np.uint32)
        h, nr, nt = C.c_void_p(), C.c_int64(), C.c_int64()
        ctx._check(ctx._lib.mb200_triplets_create(ctx._h, _ptr(pos), _ptr(fil), _ptr(seq), len(pos), C.byref(h), C.byref(nr), C.byref(nt)))
        self._h, self.n_ranges, self.n_triplets = h, nr.value, nt.value

    def ranges(self):
        a, b = np.zeros(self.n_ranges, np.int32), np.zeros(self.n_ranges, np.int32)
        self.ctx._check(self.ctx._lib.mb200_triplets_ranges(self.ctx._h, self._h, _ptr(a), _ptr(b)))
        return a, b

    def frequent(self, min_count: int):
        """keys with more than min_count values, sorted by first insertion: structured array (key, count, first)."""
        n = C.c_int64()
        self.ctx._check(self.ctx._lib.mb200_triplets_frequent(self.ctx._h, self._h, int(min_count), None, 0, C.byref(n)))
        out = np.zeros(n.value, KEYCOUNT_DTYPE)
        if n.value:
            self.ctx._check(self.ctx._lib.mb200_triplets_frequent(self.ctx._h, self._h, int(min_count), _ptr(out), n.value, C.byref(n)))
        return out[np.argsort(out["first"], kind="stable")]

    def values(self, keys, total=None):
        """dictionary values of `keys` in insertion order: list of (n, 2) int64 arrays (range index, position), both 1-based."""
        keys = np.ascontiguousarray(keys, np.uint64)
        if len(keys) == 0:
            return []
        cap = int(total) if total is not None else 1 << 20
        while True:
            out = np.zeros(max(cap, 1), TRIPVAL_DTYPE)
            n = C.c_int64()
            self.ctx._check(self.ctx._lib.mb200_triplets_values(self.ctx._h, self._h, _ptr(keys), len(keys), _ptr(out), cap, C.byref(n)))
            if n.value <= cap:
                break
            cap = n.value
        out = out[: n.value]
        out = out[np.lexsort((out["order"], out["key_index"]))]
        cuts = np.searchsorted(out["key_index"], np.arange(len(keys) + 1))
        vals = np.stack([out["range_index"].astype(np.int64), out["position"].astype(np.int64)], axis=1)
        return [vals[cuts[i]: cuts[i + 1]] for i in range(len(keys))]

    def free(self):
        if self._h:
            self.ctx._lib.mb200_triplets_destroy(self.ctx._h, self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
