"""aligntools.c_b200 -- Python host-side mirror of the reference's operator interface for
the DP hot path, bound to the C-ABI library (include/aligntools_b200.h) with ctypes.

There is no CPU fallback: importing works anywhere (so the build can be checked), but
every compute entry raises unless libaligntools_b200.so is built AND a B200 is visible.

Reference interface mirrored here (src/alignment.h):
    align_gla :417, align_local_affine :805, align_fit_affine_jump :596,
    align_overlap :926, edit_dist :291, opt_t/init_opt :57-65/:102-114.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AT_LIB_PATH") or os.path.join(HERE, "libaligntools_b200.so")   # AT_LIB_PATH: A/B runs of two builds

MODES = {"global": 0, "local": 1, "fit": 2, "overlap": 3, "edit": 4}
OUT_CIGAR, OUT_ALN = 1, 2
OUT_EDIT_PATH = 4      # AT_OUT_EDIT_PATH: "edit" honours OUT_CIGAR / OUT_ALN (otherwise it is score-only)
SEQ_BYTES, SEQ_2BIT = 0, 1
RC_NAMES = {0: "AT_OK", -1: "AT_E_ARG", -2: "AT_E_CUDA", -3: "AT_E_NOMEM", -4: "AT_E_FITLEN",
            -5: "AT_E_NOSPACE", -6: "AT_E_RANGE", -7: "AT_E_UNDEF"}

# every symbol include/aligntools_b200.h declares
EXPORTS = ["at_default_params", "at_strerror", "at_version", "at_create", "at_destroy", "at_last_error",
           "at_device_count", "at_launch_count", "at_align_gla", "at_align_local_affine",
           "at_align_fit_affine_jump", "at_align_overlap", "at_edit_dist", "at_batch_create",
           "at_batch_run", "at_batch_sizes", "at_batch_fetch", "at_batch_free", "at_batch_align",
           "at_pack_2bit", "at_cigar_to_string", "at_plan_slices", "at_host_alloc", "at_host_free", "at_host_register", "at_host_unregister",
           "at_batch_create_banded", "at_batch_align_banded", "at_batch_create_scored", "at_batch_align_scored"]


class AtError(RuntimeError):
    def __init__(self, rc, msg=""):
        self.rc = rc
        super().__init__(f"{RC_NAMES.get(rc, rc)}: {msg}")


class _Params(C.Structure):
    _fields_ = [("m", C.c_int32), ("u", C.c_int32), ("o", C.c_int32), ("e", C.c_int32),
                ("j", C.c_int32), ("jump", C.c_int32)]


class _Input(C.Structure):
    _fields_ = [("n_pairs", C.c_uint64), ("encoding", C.c_uint32),
                ("q", C.c_void_p), ("q_off", C.c_void_p), ("q_len", C.c_void_p),
                ("t", C.c_void_p), ("t_off", C.c_void_p), ("t_len", C.c_void_p),
                ("sites", C.c_void_p), ("site_off", C.c_void_p)]


class _Band(C.Structure):
    _fields_ = [("lo", C.c_void_p), ("hi", C.c_void_p)]


def _band_arrays(band, n):
    """band = (lo, hi): per-pair int32 diagonals d = j - i (include/aligntools_b200.h, at_band); None = unbanded."""
    if band is None:
        return None
    lo, hi = (np.ascontiguousarray(np.broadcast_to(np.asarray(x, dtype=np.int32), (n,))) for x in band)
    return lo, hi


class _Scoring(C.Structure):
    _fields_ = [("matrix", C.c_void_p)]


def _scoring_matrix(scoring):
    """scoring: None, or a 256 x 256 int8 substitution table, s(a, b) = scoring[a, b] for read byte a and target byte b."""
    if scoring is None:
        return None
    m = np.asarray(scoring)
    if m.shape != (256, 256):
        raise ValueError("scoring: a 256 x 256 table of int8 scores is expected")
    if m.dtype != np.int8:
        if m.min(initial=0) < -128 or m.max(initial=0) > 127:
            raise ValueError("scoring: entries must fit int8")
        m = m.astype(np.int8)
    return np.ascontiguousarray(m)


def scoring_matrix(alphabet, scores, default=0):
    """A 256 x 256 int8 substitution table from a K-letter alphabet (bytes or str) and a K x K table of scores:
    s(alphabet[a], alphabet[b]) = scores[a][b]; every pair with a byte outside the alphabet scores `default`.
    Example, DNA with transitions scored above transversions and N neutral:
        scoring_matrix("ACGTN", [[2, -3, -1, -3, 0], [-3, 2, -3, -1, 0], [-1, -3, 2, -3, 0], [-3, -1, -3, 2, 0], [0] * 5])"""
    ab = alphabet.encode() if isinstance(alphabet, str) else bytes(alphabet)
    sc = np.asarray(scores, dtype=np.int64)
    if len(set(ab)) != len(ab) or sc.shape != (len(ab), len(ab)):
        raise ValueError("scoring_matrix: distinct letters and a K x K score table are expected")
    if sc.min(initial=0) < -128 or sc.max(initial=0) > 127 or not -128 <= default <= 127:
        raise ValueError("scoring_matrix: scores must fit int8")
    m = np.full((256, 256), default, dtype=np.int8)
    idx = np.frombuffer(ab, dtype=np.uint8)
    m[np.ix_(idx, idx)] = sc.astype(np.int8)
    return m


def identity_scoring(m, u):
    """The table that scores like match / mismatch: m on equal bytes, u otherwise (at_batch_align's scoring)."""
    t = np.full((256, 256), u, dtype=np.int8)
    np.fill_diagonal(t, m)
    return t


class _Output(C.Structure):
    _fields_ = [("score", C.c_void_p), ("end_i", C.c_void_p), ("end_j", C.c_void_p),
                ("beg_i", C.c_void_p), ("beg_j", C.c_void_p),
                ("cigar", C.c_void_p), ("cigar_cap", C.c_uint64), ("cigar_off", C.c_void_p),
                ("aln1", C.c_void_p), ("aln2", C.c_void_p), ("aln_cap", C.c_uint64), ("aln_off", C.c_void_p)]


class _Timing(C.Structure):
    _fields_ = [("fill_ms", C.c_double), ("traceback_ms", C.c_double), ("device_ms", C.c_double),
                ("cells", C.c_uint64), ("launches", C.c_uint64), ("ptr_bytes", C.c_uint64),
                ("fill_kernel_ms", C.c_double), ("fill_kernel_cells", C.c_uint64),
                ("fill_kernel_kind", C.c_uint32), ("fill_kernel_rows", C.c_uint32),
                ("fill_kernel_flags", C.c_uint32), ("reserved_", C.c_uint32)]


_lib = None


def _build_entry(force=False, verbose=False):
    """Compile libaligntools_b200.so and the C host in-tree (see build.py)."""
    import importlib
    mod = importlib.import_module(__name__ + ".build")
    globals()["build"] = _build_entry        # importing the submodule rebinds the package attribute `build`: undo
    return mod.build(force=force, verbose=verbose)


build = _build_entry


def load_library():
    """dlopen the C-ABI library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -m aligntools.c_b200.build` "
                           "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.at_strerror.restype = C.c_char_p
    lib.at_version.restype = C.c_char_p
    lib.at_last_error.restype = C.c_char_p
    lib.at_last_error.argtypes = [C.c_void_p]
    lib.at_create.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
    lib.at_destroy.argtypes = [C.c_void_p]
    lib.at_launch_count.restype = C.c_uint64
    lib.at_launch_count.argtypes = [C.c_void_p]
    lib.at_device_count.argtypes = [C.c_void_p]
    lib.at_batch_create.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Params), C.POINTER(_Input), C.c_uint32,
                                    C.POINTER(C.c_void_p)]
    lib.at_batch_run.argtypes = [C.c_void_p, C.POINTER(_Timing)]
    lib.at_batch_sizes.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.at_batch_fetch.argtypes = [C.c_void_p, C.POINTER(_Output)]
    lib.at_batch_free.argtypes = [C.c_void_p]
    lib.at_batch_align.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Params), C.POINTER(_Input), C.c_uint32,
                                   C.POINTER(_Output), C.POINTER(_Timing)]
    lib.at_batch_create_banded.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Params), C.POINTER(_Input), C.POINTER(_Band),
                                           C.c_uint32, C.POINTER(C.c_void_p)]
    lib.at_batch_align_banded.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Params), C.POINTER(_Input), C.POINTER(_Band),
                                          C.c_uint32, C.POINTER(_Output), C.POINTER(_Timing)]
    lib.at_batch_create_scored.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Params), C.POINTER(_Input), C.POINTER(_Scoring),
                                           C.c_uint32, C.POINTER(C.c_void_p)]
    lib.at_batch_align_scored.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Params), C.POINTER(_Input), C.POINTER(_Scoring),
                                          C.c_uint32, C.POINTER(_Output), C.POINTER(_Timing)]
    lib.at_pack_2bit.restype = C.c_int64
    lib.at_pack_2bit.argtypes = [C.c_char_p, C.c_uint64, C.c_void_p]
    lib.at_cigar_to_string.restype = C.c_int64
    lib.at_cigar_to_string.argtypes = [C.c_void_p, C.c_uint64, C.c_char_p, C.c_uint64]
    lib.at_plan_slices.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
    lib.at_host_alloc.restype = C.c_void_p
    lib.at_host_alloc.argtypes = [C.c_size_t]
    lib.at_host_free.argtypes = [C.c_void_p]
    lib.at_host_register.argtypes = [C.c_void_p, C.c_size_t]
    lib.at_host_unregister.argtypes = [C.c_void_p]
    _lib = lib
    return lib


def plan_slices(q_len, t_len, parts):
    """Contiguous slices of the batch with nearly equal numbers of DP cells (at_plan_slices):
    returns parts + 1 cut indices.  The same plan shards a batch over the devices of one handle."""
    lib = load_library()
    q_len = np.ascontiguousarray(q_len, dtype=np.uint32)
    t_len = np.ascontiguousarray(t_len, dtype=np.uint32)
    cut = np.zeros(parts + 1, dtype=np.uint64)
    rc = lib.at_plan_slices(q_len.ctypes.data, t_len.ctypes.data, len(q_len), parts, cut.ctypes.data)
    if rc:
        raise AtError(rc, "at_plan_slices")
    return cut


@dataclass
class Opt:
    """opt_t (src/alignment.h:57-65) with init_opt() defaults (:102-114)."""
    m: int = 1
    u: int = -2
    o: int = -5
    e: int = -1
    j: int = -10
    jump: bool = False          # `-s`
    sites: list = field(default_factory=list)
    whitelist: bool = False     # jump state with the site list as a WHITELIST (at_params.jump == 2): entering J only
                                # on the listed indices, as the comment at src/alignment.h:542-544 describes

    def c(self):
        return _Params(self.m, self.u, self.o, self.e, self.j, 2 if (self.jump and self.whitelist) else int(self.jump))


@dataclass
class Timing:
    fill_ms: float
    traceback_ms: float
    device_ms: float
    cells: int
    launches: int
    ptr_bytes: int
    fill_kernel_ms: float
    fill_kernel_cells: int
    fill_kernel_kind: int = 0       # enum at_kernel_kind
    fill_kernel_rows: int = 0
    fill_kernel_flags: int = 0


def _mode(mode):
    return MODES[mode] if isinstance(mode, str) else int(mode)


def _has_path(md, out_flags):
    """Whether a run produces alignments: every mode but "edit", which needs OUT_EDIT_PATH as well."""
    return md != 4 or bool(out_flags & OUT_EDIT_PATH)


def pack_seqs(seqs):
    """list[bytes] -> (uint8 concat, uint64 offsets[n], uint32 lens[n])"""
    lens = np.fromiter((len(s) for s in seqs), dtype=np.uint32, count=len(seqs))
    off = np.zeros(len(seqs), dtype=np.uint64)
    if len(seqs) > 1:
        np.cumsum(lens[:-1], out=off[1:])
    buf = np.frombuffer(b"".join(seqs), dtype=np.uint8)
    if buf.size == 0:
        buf = np.zeros(1, np.uint8)
    return np.ascontiguousarray(buf), off, lens


def pack_2bit(buf, off, lens, align=1):
    """byte batch (ACGT only) -> 2-bit batch (AT_SEQ_2BIT).  Records start on a multiple of `align` bytes: 1 = densest
    (the format only asks for byte alignment); 16 lets the fill kernels read them with 128-bit loads."""
    lut = np.full(256, 255, np.uint8)
    for k, ch in enumerate(b"ACGT"):
        lut[ch] = k
    n = len(lens)
    nb = (lens.astype(np.uint64) + 3) // 4
    nb_raw = nb
    nb = (nb + np.uint64(align - 1)) // np.uint64(align) * np.uint64(align)
    poff = np.zeros(n, dtype=np.uint64)
    if n > 1:
        np.cumsum(nb[:-1], out=poff[1:])
    total = int(nb.sum())
    out = np.zeros(total + 1, dtype=np.uint8)
    same = n > 0 and np.all(lens == lens[0]) and np.all(np.diff(off.astype(np.int64)) == int(lens[0]))
    if same:
        L = int(lens[0])
        codes = lut[buf[int(off[0]):int(off[0]) + n * L]].reshape(n, L)
        if codes.max(initial=0) > 3:
            raise ValueError("2-bit packing needs upper-case ACGT only")
        pad = (-L) % 4
        if pad:
            codes = np.concatenate([codes, np.zeros((n, pad), np.uint8)], axis=1)
        c4 = codes.reshape(n, -1, 4)
        packed = (c4[:, :, 0] | (c4[:, :, 1] << 2) | (c4[:, :, 2] << 4) | (c4[:, :, 3] << 6)).astype(np.uint8)
        out[:total].reshape(n, int(nb[0]))[:, :int(nb_raw[0])] = packed
    else:
        for p in range(n):
            codes = lut[buf[int(off[p]):int(off[p]) + int(lens[p])]]
            if codes.size and codes.max() > 3:
                raise ValueError("2-bit packing needs upper-case ACGT only")
            pad = (-codes.size) % 4
            c4 = np.concatenate([codes, np.zeros(pad, np.uint8)]).reshape(-1, 4)
            out[int(poff[p]):int(poff[p]) + c4.shape[0]] = c4[:, 0] | (c4[:, 1] << 2) | (c4[:, 2] << 4) | (c4[:, 3] << 6)
    return out, poff, lens


class BatchResult:
    def __init__(self, n):
        self.n = n
        self.score = np.zeros(n, np.int32)
        self.end_i = np.zeros(n, np.uint32)
        self.end_j = np.zeros(n, np.uint32)
        self.beg_i = np.zeros(n, np.uint32)
        self.beg_j = np.zeros(n, np.uint32)
        self.cigar = None
        self.cigar_off = None
        self.aln1 = None
        self.aln2 = None
        self.aln_off = None
        self.timing = None

    def aln(self, p):
        a, b = int(self.aln_off[p]), int(self.aln_off[p + 1])
        return self.aln1[a:b].tobytes(), self.aln2[a:b].tobytes()

    def cigar_ops(self, p):
        a, b = int(self.cigar_off[p]), int(self.cigar_off[p + 1])
        return self.cigar[a:b]

    def cigar_string(self, p):
        ops = self.cigar_ops(p)
        return "".join(f"{int(o) >> 4}{'MIDN'[int(o) & 3]}" for o in ops)


class Batch:
    """A batch resident on the device(s): create (H2D) -> run (kernels) -> fetch (D2H)."""

    def __init__(self, aligner, mode, opt, q, q_off, q_len, t, t_off, t_len, sites=None, site_off=None,
                 out_flags=OUT_CIGAR | OUT_ALN, encoding=SEQ_BYTES, band=None, scoring=None):
        """band: None, or (lo, hi) -- per-pair int32 diagonals (d = j - i) of a banded "overlap" or "global" alignment
        (at_batch_create_banded; a global pair's band must hold its end diagonal l2 - l1); a scalar applies to every
        pair.  scoring: None, or a 256 x 256 int8 substitution table (at_batch_create_scored; see scoring_matrix) for
        "global", "local", "fit" or "overlap"; it takes no band."""
        self.al = aligner
        self.lib = aligner.lib
        self.n = int(len(q_len))
        self.out_flags = out_flags
        self.mode = _mode(mode)
        self._keep = [np.ascontiguousarray(x) if x is not None else None
                      for x in (q, q_off, q_len, t, t_off, t_len, sites, site_off)]
        q, q_off, q_len, t, t_off, t_len, sites, site_off = self._keep
        assert q_off.dtype == np.uint64 and t_off.dtype == np.uint64
        assert q_len.dtype == np.uint32 and t_len.dtype == np.uint32
        assert q.dtype == np.uint8 and t.dtype == np.uint8
        inp = _Input(self.n, encoding, q.ctypes.data, q_off.ctypes.data, q_len.ctypes.data,
                     t.ctypes.data, t_off.ctypes.data, t_len.ctypes.data,
                     sites.ctypes.data if sites is not None else None,
                     site_off.ctypes.data if site_off is not None else None)
        if sites is not None:
            assert sites.dtype == np.int32 and site_off.dtype == np.uint64
        self.h = C.c_void_p()
        prm = opt.c()
        self._band = _band_arrays(band, self.n)
        self._scoring = _scoring_matrix(scoring)
        if self._scoring is not None:
            if self._band is not None:
                raise ValueError("scoring: a substitution matrix takes no band")
            sc = _Scoring(self._scoring.ctypes.data)
            rc = self.lib.at_batch_create_scored(aligner.h, self.mode, C.byref(prm), C.byref(inp), C.byref(sc), out_flags,
                                                 C.byref(self.h))
        elif self._band is None:
            rc = self.lib.at_batch_create(aligner.h, self.mode, C.byref(prm), C.byref(inp), out_flags, C.byref(self.h))
        else:
            bd = _Band(self._band[0].ctypes.data, self._band[1].ctypes.data)
            rc = self.lib.at_batch_create_banded(aligner.h, self.mode, C.byref(prm), C.byref(inp), C.byref(bd), out_flags,
                                                 C.byref(self.h))
        if rc:
            raise AtError(rc, aligner.last_error())

    def run(self) -> Timing:
        tm = _Timing()
        rc = self.lib.at_batch_run(self.h, C.byref(tm))
        if rc:
            raise AtError(rc, self.al.last_error())
        return Timing(tm.fill_ms, tm.traceback_ms, tm.device_ms, tm.cells, tm.launches, tm.ptr_bytes,
                      tm.fill_kernel_ms, tm.fill_kernel_cells, tm.fill_kernel_kind, tm.fill_kernel_rows, tm.fill_kernel_flags)

    def fetch(self) -> BatchResult:
        res = BatchResult(self.n)
        no, nc = C.c_uint64(), C.c_uint64()
        rc = self.lib.at_batch_sizes(self.h, C.byref(no), C.byref(nc))
        if rc:
            raise AtError(rc, self.al.last_error())
        out = _Output()
        out.score = res.score.ctypes.data
        out.end_i, out.end_j = res.end_i.ctypes.data, res.end_j.ctypes.data
        out.beg_i, out.beg_j = res.beg_i.ctypes.data, res.beg_j.ctypes.data
        path = _has_path(self.mode, self.out_flags)
        if self.out_flags & OUT_CIGAR and path:
            res.cigar = np.zeros(no.value + 1, np.uint32)
            res.cigar_off = np.zeros(self.n + 1, np.uint64)
            out.cigar, out.cigar_cap, out.cigar_off = res.cigar.ctypes.data, no.value + 1, res.cigar_off.ctypes.data
        if self.out_flags & OUT_ALN and path:
            res.aln1 = np.zeros(nc.value + 1, np.uint8)
            res.aln2 = np.zeros(nc.value + 1, np.uint8)
            res.aln_off = np.zeros(self.n + 1, np.uint64)
            out.aln1, out.aln2, out.aln_cap, out.aln_off = res.aln1.ctypes.data, res.aln2.ctypes.data, nc.value + 1, res.aln_off.ctypes.data
        rc = self.lib.at_batch_fetch(self.h, C.byref(out))
        if rc:
            raise AtError(rc, self.al.last_error())
        return res

    def free(self):
        if self.h:
            self.lib.at_batch_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Aligner:
    """Owns an at_handle (one stream + host thread per device)."""

    def __init__(self, devices=None):
        self.lib = load_library()
        self.h = C.c_void_p()
        if devices:
            arr = (C.c_int * len(devices))(*devices)
            rc = self.lib.at_create(arr, len(devices), C.byref(self.h))
        else:
            rc = self.lib.at_create(None, 0, C.byref(self.h))
        if rc:
            raise AtError(rc, self.lib.at_strerror(rc).decode())

    def last_error(self):
        return self.lib.at_last_error(self.h).decode()

    def launch_count(self):
        return int(self.lib.at_launch_count(self.h))

    def batch(self, mode, opt, q, q_off, q_len, t, t_off, t_len, **kw) -> Batch:
        return Batch(self, mode, opt, q, q_off, q_len, t, t_off, t_len, **kw)

    def align_arrays(self, mode, opt, q, q_off, q_len, t, t_off, t_len, sites=None, site_off=None,
                     out_flags=OUT_CIGAR, encoding=SEQ_BYTES, out: BatchResult = None,
                     cigar_cap=None, aln_cap=None, band=None, scoring=None) -> BatchResult:
        """One-shot at_batch_align (host arrays in, host arrays out; large batches are pipelined
        H2D / kernels / D2H inside the library).  `out` may be a BatchResult from a previous call
        whose buffers are reused; capacities default to the worst case (l1 + l2 per pair) for
        the alignment strings and for the CIGARs (32 ops per pair once that exceeds 64 Mi ops;
        AT_E_NOSPACE tells when to pass a larger cigar_cap).  band: (lo, hi) per-pair diagonals of a banded "overlap" or
        "global" alignment (at_batch_align_banded), or None.  scoring: a 256 x 256 int8 substitution table
        (at_batch_align_scored), or None."""
        md = _mode(mode)
        n = int(len(q_len))
        res = out if out is not None else BatchResult(n)
        o = _Output()
        o.score = res.score.ctypes.data
        o.end_i, o.end_j = res.end_i.ctypes.data, res.end_j.ctypes.data
        o.beg_i, o.beg_j = res.beg_i.ctypes.data, res.beg_j.ctypes.data
        path = _has_path(md, out_flags)
        if out_flags & OUT_CIGAR and path:
            if cigar_cap is None:
                worst = int(q_len.astype(np.uint64).sum() + t_len.astype(np.uint64).sum())     # one op per column
                cigar_cap = worst if worst <= (1 << 26) else 32 * n + 1024
            cap = int(cigar_cap)
            if res.cigar is None or res.cigar.size < cap:
                res.cigar = np.zeros(cap, np.uint32)
                res.cigar_off = np.zeros(n + 1, np.uint64)
            o.cigar, o.cigar_cap, o.cigar_off = res.cigar.ctypes.data, res.cigar.size, res.cigar_off.ctypes.data
        if out_flags & OUT_ALN and path:
            cap = int(aln_cap if aln_cap is not None else int(q_len.astype(np.uint64).sum() + t_len.astype(np.uint64).sum()) + 16)
            if res.aln1 is None or res.aln1.size < cap:
                res.aln1 = np.zeros(cap, np.uint8)
                res.aln2 = np.zeros(cap, np.uint8)
                res.aln_off = np.zeros(n + 1, np.uint64)
            o.aln1, o.aln2, o.aln_cap, o.aln_off = res.aln1.ctypes.data, res.aln2.ctypes.data, res.aln1.size, res.aln_off.ctypes.data
        inp = _Input(n, encoding, q.ctypes.data, q_off.ctypes.data, q_len.ctypes.data,
                     t.ctypes.data, t_off.ctypes.data, t_len.ctypes.data,
                     sites.ctypes.data if sites is not None else None,
                     site_off.ctypes.data if site_off is not None else None)
        prm = opt.c()
        tm = _Timing()
        bnd = _band_arrays(band, n)
        mat = _scoring_matrix(scoring)
        if mat is not None:
            if bnd is not None:
                raise ValueError("scoring: a substitution matrix takes no band")
            rc = self.lib.at_batch_align_scored(self.h, md, C.byref(prm), C.byref(inp), C.byref(_Scoring(mat.ctypes.data)), out_flags,
                                                C.byref(o), C.byref(tm))
        elif bnd is None:
            rc = self.lib.at_batch_align(self.h, md, C.byref(prm), C.byref(inp), out_flags, C.byref(o), C.byref(tm))
        else:
            bd = _Band(bnd[0].ctypes.data, bnd[1].ctypes.data)
            rc = self.lib.at_batch_align_banded(self.h, md, C.byref(prm), C.byref(inp), C.byref(bd), out_flags, C.byref(o), C.byref(tm))
        if rc:
            raise AtError(rc, self.last_error())
        res.timing = Timing(tm.fill_ms, tm.traceback_ms, tm.device_ms, tm.cells, tm.launches, tm.ptr_bytes,
                            tm.fill_kernel_ms, tm.fill_kernel_cells, tm.fill_kernel_kind, tm.fill_kernel_rows, tm.fill_kernel_flags)
        return res

    def align(self, mode, reads, targets, opt: Opt = None, sites=None, out_flags=OUT_CIGAR | OUT_ALN, band=None,
              scoring=None) -> BatchResult:
        """Lists of bytes in, BatchResult out (create + run + fetch).  band: (lo, hi) diagonals, "overlap" or "global".
        scoring: a 256 x 256 int8 substitution table (see scoring_matrix), or None."""
        opt = opt or Opt()
        q, qo, ql = pack_seqs(reads)
        t, to, tl = pack_seqs(targets)
        sa = so = None
        if _mode(mode) == 2 and opt.jump:
            sites = sites if sites is not None else [opt.sites] * len(reads)
            flat = [x for s in sites for x in (s or [])]
            sa = np.array(flat + [0], dtype=np.int32)
            so = np.zeros(len(reads) + 1, np.uint64)
            np.cumsum([len(s or []) for s in sites], out=so[1:])
        b = Batch(self, mode, opt, q, qo, ql, t, to, tl, sites=sa, site_off=so, out_flags=out_flags, band=band, scoring=scoring)
        try:
            tm = b.run()
            res = b.fetch()
            res.timing = tm
        finally:
            b.free()
        return res

    def close(self):
        if self.h:
            self.lib.at_destroy(self.h)
            self.h = C.c_void_p()


_default = None


def default_aligner() -> Aligner:
    global _default
    if _default is None:
        _default = Aligner()
    return _default


# ---- reference-named single-pair operators (same argument meaning / error behaviour) ----
def _single(mode, s1, s2, opt):
    opt = opt or Opt()
    if s1 is None or s2 is None:
        raise ValueError("align: parameter error")            # die() at :419
    if mode == "fit" and len(s1) > len(s2):
        raise ValueError("first sequence must be shorter than the second to do fitting alignment")  # :599
    res = default_aligner().align(mode, [bytes(s1)], [bytes(s2)], opt,
                                  out_flags=0 if mode == "edit" else OUT_CIGAR | OUT_ALN)
    if mode == "edit":
        return int(res.score[0])
    r1, r2 = res.aln(0)
    return float(res.score[0]), r1, r2


def align_gla(s1, s2, opt: Opt = None):
    """align_gla (src/alignment.h:417-473): (score, r1, r2)."""
    return _single("global", s1, s2, opt)


def align_local_affine(s1, s2, opt: Opt = None):
    """align_local_affine (src/alignment.h:805-847)."""
    return _single("local", s1, s2, opt)


def align_fit_affine_jump(s1, s2, opt: Opt = None):
    """align_fit_affine_jump (src/alignment.h:596-694); opt.jump / opt.sites as `-s`."""
    return _single("fit", s1, s2, opt)


def align_overlap(s1, s2, opt: Opt = None):
    """align_overlap (src/alignment.h:926-964)."""
    return _single("overlap", s1, s2, opt)


def edit_dist(s1, s2, opt: Opt = None):
    """edit_dist (src/alignment.h:291-315)."""
    return _single("edit", s1, s2, opt)
