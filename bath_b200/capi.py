"""ctypes binding of the C ABI in include/bathgpu.h (the calls a bathsearch build would make)."""
import ctypes as C
import os

import numpy as np

from .build import library_path

OK, EMEM, EINVAL, ERANGE, ENODEVICE, ECUDA = 0, 5, 11, 16, 100, 101
KP = 29

EXPORTS = [
    "bathgpu_create", "bathgpu_destroy", "bathgpu_last_error", "bathgpu_device_info", "bathgpu_set_long_models",
    "bathgpu_load_fs_profile", "bathgpu_upload_block", "bathgpu_fs_fwd_windows",
    "bathgpu_stage_windows", "bathgpu_fs_fwd_staged", "bathgpu_fetch_scores",
    "bathgpu_fs_bck_decode", "bathgpu_fs_domains", "bathgpu_last_stage_timing", "bathgpu_measure_fp32_peak",
    "bathgpu_host_alloc", "bathgpu_host_free", "bathgpu_fs_fetch_xrows",
    "bathgpu_fs_fetch_domain_matrices",
    "bathgpu_load_filter_profile", "bathgpu_upload_orfs", "bathgpu_msv_orfs", "bathgpu_ssv_windows", "bathgpu_vit_orfs",
    "bathgpu_fwd_orfs", "bathgpu_fs_fwd_bck_xrows", "bathgpu_select_slot",
    "bathgpu_orf_fwd_bck_xrows", "bathgpu_orf_domains", "bathgpu_orf_fetch_domain_matrices",
    "bathgpu_orfs_msv_screen", "bathgpu_orfs_fetch", "bathgpu_revcomp_slot", "bathgpu_fs_fwd_block", "bathgpu_fs_forward_matrices",
    "bathgpu_bias_forward", "bathgpu_orfs_stage_breakdown", "bathgpu_measure_int16_peak", "bathgpu_orf_forward_matrices",
    "bathgpu_packed4_bytes", "bathgpu_pack_dna4", "bathgpu_upload_block_packed4", "bathgpu_fs_fwd_block_packed4",
    "bathgpu_upload_block_segments", "bathgpu_load_fs_profile_set", "bathgpu_fs_set_scores",
    "bathgpu_load_filter_profile_set", "bathgpu_orfs_msv_screen_set", "bathgpu_orfs_fetch_set",
]


class Window(C.Structure):
    _fields_ = [("start", C.c_int64), ("L", C.c_int32), ("pmove", C.c_float), ("ploop", C.c_float)]


Envelope = Window

window_dtype = np.dtype([("start", "<i8"), ("L", "<i4"), ("pmove", "<f4"), ("ploop", "<f4")], align=True)
set_window_dtype = np.dtype([("start", "<i8"), ("L", "<i4"), ("pmove", "<f4"), ("ploop", "<f4"), ("profile", "<i4")], align=True)
trace_dtype = np.dtype([("i", "<i4"), ("k", "<i2"), ("st", "u1"), ("c", "u1"), ("pp", "<f4")], align=True)
domain_dtype = np.dtype([("envsc", "<f4"), ("bcksc", "<f4"), ("oasc", "<f4"), ("status", "<i4"),
                         ("trace_offset", "<i4"), ("trace_len", "<i4"), ("null2", "<f4", (KP,))], align=True)


class FilterParams(C.Structure):
    _fields_ = [("M", C.c_int32), ("tbm_b", C.c_int32), ("tec_b", C.c_int32), ("base_b", C.c_int32), ("bias_b", C.c_int32),
                ("scale_b", C.c_float), ("base_w", C.c_int32), ("ddbound_w", C.c_int32), ("xw_E_move", C.c_int32),
                ("xw_E_loop", C.c_int32), ("scale_w", C.c_float), ("cpu_lanes_u8", C.c_int32), ("cpu_lanes_i16", C.c_int32)]


orf_dtype = np.dtype([("offset", "<i8"), ("L", "<i4"), ("tjb_b", "u1"), ("ssv_thresh", "u1"), ("xw_move", "<i2"),
                      ("vit_thresh", "<i2"), ("flags", "<i2"), ("ext_thresh", "<i4")], align=True)
orf_window_dtype = np.dtype([("orf", "<i4"), ("n", "<i4"), ("k", "<i4"), ("length", "<i4"), ("score", "<f4")], align=True)
bias_item_dtype = np.dtype([("start", "<i8"), ("L", "<i4"), ("table", "<i4"), ("t00", "<f4"), ("pad_", "<i4")], align=True)
block_dtype = np.dtype([("goff", "<i8"), ("n", "<i4"), ("C", "<i4")], align=True)


class ScreenJob(C.Structure):
    """bathgpu_screen_job"""
    _fields_ = [("profile", C.c_int32), ("nblocks", C.c_int32), ("blocks", C.c_void_p), ("min_bits", C.c_double)]
orf_hit_dtype = np.dtype([("block", "<i4"), ("index", "<i4"), ("start", "<i4"), ("end", "<i4"), ("n", "<i4"), ("frame", "<i4"),
                          ("offset", "<i8"), ("usc", "<f4"), ("status", "<i4")], align=True)


class BathGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"bathgpu status {code}: {msg}")
        self.code = code


_lib = None


def load():
    """Load libbathgpu.so.  Fails loudly if it has not been built -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: build it with `python -m bath_b200.build` "
                          "(the CUDA library is the product; there is no CPU fallback)")
    L = C.CDLL(path)
    vp, fp, ip = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int32)
    L.bathgpu_create.restype = C.c_int
    L.bathgpu_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.bathgpu_destroy.restype = None
    L.bathgpu_destroy.argtypes = [vp]
    L.bathgpu_last_error.restype = C.c_char_p
    L.bathgpu_last_error.argtypes = [vp]
    L.bathgpu_device_info.restype = C.c_int
    L.bathgpu_set_long_models.restype = C.c_int
    L.bathgpu_set_long_models.argtypes = [vp, C.c_int]
    L.bathgpu_device_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_size_t)]
    L.bathgpu_load_fs_profile.restype = C.c_int
    L.bathgpu_load_fs_profile.argtypes = [vp, C.c_int, C.c_int, C.c_int, fp, fp]
    L.bathgpu_upload_block.restype = C.c_int
    L.bathgpu_upload_block.argtypes = [vp, C.POINTER(C.c_uint8), C.c_int64]
    L.bathgpu_packed4_bytes.restype = C.c_int64
    L.bathgpu_packed4_bytes.argtypes = [C.c_int64]
    L.bathgpu_pack_dna4.restype = C.c_int
    L.bathgpu_pack_dna4.argtypes = [C.POINTER(C.c_uint8), C.c_int64, C.POINTER(C.c_uint8)]
    L.bathgpu_upload_block_segments.restype = C.c_int
    L.bathgpu_upload_block_segments.argtypes = [vp, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_int64), C.c_int]
    L.bathgpu_upload_block_packed4.restype = C.c_int
    L.bathgpu_upload_block_packed4.argtypes = [vp, C.POINTER(C.c_uint8), C.c_int64]
    L.bathgpu_fs_fwd_windows.restype = C.c_int
    L.bathgpu_fs_fwd_windows.argtypes = [vp, vp, C.c_int, fp, fp, ip]
    L.bathgpu_stage_windows.restype = C.c_int
    L.bathgpu_stage_windows.argtypes = [vp, vp, C.c_int]
    L.bathgpu_fs_fwd_staged.restype = C.c_int
    L.bathgpu_fs_fwd_staged.argtypes = [vp, fp]
    L.bathgpu_fetch_scores.restype = C.c_int
    L.bathgpu_fetch_scores.argtypes = [vp, fp, ip, C.c_int]
    L.bathgpu_fs_bck_decode.restype = C.c_int
    L.bathgpu_fs_bck_decode.argtypes = [vp, vp, C.c_int, fp, fp, C.POINTER(C.c_int64), fp, fp, fp, fp, fp, ip]
    L.bathgpu_fs_domains.restype = C.c_int
    L.bathgpu_fs_domains.argtypes = [vp, vp, C.c_int, fp, vp, vp, C.c_int64]
    L.bathgpu_last_stage_timing.restype = C.c_int
    L.bathgpu_last_stage_timing.argtypes = [vp, fp, C.POINTER(C.c_int)]
    L.bathgpu_measure_fp32_peak.restype = C.c_int
    L.bathgpu_measure_fp32_peak.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.bathgpu_fs_fetch_xrows.restype = C.c_int
    L.bathgpu_fs_fetch_xrows.argtypes = [vp, C.c_int, fp, C.c_int64]
    L.bathgpu_fs_fetch_domain_matrices.restype = C.c_int
    L.bathgpu_fs_fetch_domain_matrices.argtypes = [vp, C.c_int, fp, fp, fp, fp]
    L.bathgpu_load_filter_profile.restype = C.c_int
    L.bathgpu_load_filter_profile.argtypes = [vp, C.POINTER(FilterParams), C.POINTER(C.c_uint8), C.POINTER(C.c_int16), C.POINTER(C.c_int16)]
    L.bathgpu_upload_orfs.restype = C.c_int
    L.bathgpu_upload_orfs.argtypes = [vp, C.POINTER(C.c_uint8), C.c_int64]
    L.bathgpu_msv_orfs.restype = C.c_int
    L.bathgpu_msv_orfs.argtypes = [vp, vp, C.c_int, fp, ip]
    L.bathgpu_ssv_windows.restype = C.c_int
    L.bathgpu_ssv_windows.argtypes = [vp, vp, C.c_int, vp, C.c_int, ip]
    L.bathgpu_vit_orfs.restype = C.c_int
    L.bathgpu_vit_orfs.argtypes = [vp, vp, C.c_int, fp, ip, vp, C.c_int, ip]
    L.bathgpu_fwd_orfs.restype = C.c_int
    L.bathgpu_fwd_orfs.argtypes = [vp, vp, C.c_int, C.c_float, fp, fp, ip]
    L.bathgpu_fs_fwd_bck_xrows.restype = C.c_int
    L.bathgpu_fs_fwd_bck_xrows.argtypes = [vp, vp, C.c_int, fp, fp, fp, fp, fp, ip]
    L.bathgpu_orf_fwd_bck_xrows.restype = C.c_int
    L.bathgpu_orf_fwd_bck_xrows.argtypes = [vp, vp, C.c_int, C.c_float, fp, fp, fp, fp, fp, ip]
    L.bathgpu_orf_domains.restype = C.c_int
    L.bathgpu_orf_domains.argtypes = [vp, vp, C.c_int, fp, vp, vp, C.c_int64]
    L.bathgpu_orf_fetch_domain_matrices.restype = C.c_int
    L.bathgpu_orf_fetch_domain_matrices.argtypes = [vp, C.c_int, fp, fp, fp, fp]
    L.bathgpu_orfs_msv_screen.restype = C.c_int
    L.bathgpu_orfs_msv_screen.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(C.c_uint8), C.c_int, C.POINTER(C.c_uint8), fp, C.c_int, C.c_double,
                                          C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.bathgpu_orfs_fetch.restype = C.c_int
    L.bathgpu_orfs_fetch.argtypes = [vp, vp, C.POINTER(C.c_uint8)]
    L.bathgpu_load_filter_profile_set.restype = C.c_int
    L.bathgpu_load_filter_profile_set.argtypes = [vp, C.c_int, vp, C.POINTER(C.POINTER(C.c_uint8))]
    L.bathgpu_orfs_msv_screen_set.restype = C.c_int
    L.bathgpu_orfs_msv_screen_set.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(C.c_uint8), C.c_int, C.POINTER(C.c_uint8), fp, C.c_int,
                                              C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.bathgpu_orfs_fetch_set.restype = C.c_int
    L.bathgpu_orfs_fetch_set.argtypes = [vp, vp, C.POINTER(C.c_uint8)]
    L.bathgpu_revcomp_slot.restype = C.c_int
    L.bathgpu_revcomp_slot.argtypes = [vp, C.c_int, C.c_int]
    L.bathgpu_fs_fwd_block.restype = C.c_int
    L.bathgpu_fs_fwd_block.argtypes = [vp, C.POINTER(C.c_uint8), C.c_int64, vp, C.c_int, fp, fp, ip]
    L.bathgpu_fs_fwd_block_packed4.restype = C.c_int
    L.bathgpu_fs_fwd_block_packed4.argtypes = [vp, C.POINTER(C.c_uint8), C.c_int64, vp, C.c_int, fp, fp, ip]
    L.bathgpu_fs_forward_matrices.restype = C.c_int
    L.bathgpu_fs_forward_matrices.argtypes = [vp, vp, C.c_int, fp, fp, fp, C.c_int64, fp, ip]
    L.bathgpu_select_slot.restype = C.c_int
    L.bathgpu_select_slot.argtypes = [vp, C.c_int]
    L.bathgpu_orf_forward_matrices.restype = C.c_int
    L.bathgpu_orf_forward_matrices.argtypes = [vp, vp, C.c_int, fp, fp, fp, C.c_int64, fp, ip]
    L.bathgpu_measure_int16_peak.restype = C.c_int
    L.bathgpu_measure_int16_peak.argtypes = [vp, C.POINTER(C.c_double)]
    L.bathgpu_orfs_stage_breakdown.restype = C.c_int
    L.bathgpu_orfs_stage_breakdown.argtypes = [vp, fp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.bathgpu_bias_forward.restype = C.c_int
    L.bathgpu_bias_forward.argtypes = [vp, C.c_int, vp, C.c_int, fp, C.c_int, C.c_float, C.c_float, C.POINTER(C.c_uint8), fp]
    L.bathgpu_load_fs_profile_set.restype = C.c_int
    L.bathgpu_load_fs_profile_set.argtypes = [vp, C.c_int, C.c_int, ip, ip, C.POINTER(fp), C.POINTER(fp)]
    L.bathgpu_fs_set_scores.restype = C.c_int
    L.bathgpu_fs_set_scores.argtypes = [vp, C.c_int, vp, C.c_int, fp, fp, ip]
    L.bathgpu_host_alloc.restype = vp
    L.bathgpu_host_alloc.argtypes = [C.c_size_t]
    L.bathgpu_host_free.restype = None
    L.bathgpu_host_free.argtypes = [vp]
    _lib = L
    return L


def pinned_array(shape, dtype):
    """numpy array over page-locked memory from bathgpu_host_alloc (kept alive by the returned array's base)."""
    dt = np.dtype(dtype)
    n = int(np.prod(shape)) * dt.itemsize
    L = load()
    p = L.bathgpu_host_alloc(max(n, 1))
    if not p:
        raise MemoryError(f"bathgpu_host_alloc({n}) failed")

    class _Owner:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            try:
                L.bathgpu_host_free(self.ptr)
            except Exception:
                pass

    buf = (C.c_uint8 * max(n, 1)).from_address(p)
    buf._owner = _Owner(p)
    return np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)


def _f(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _i(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


class Context:
    """One device context (one stream).  Mirrors the per-worker P7_PIPELINE ownership of the
    reference (src/bathsearch.c:814-844): one context per worker thread / per GPU."""

    def __init__(self, device=0, long_models=False):
        """long_models: take profiles of up to 2048 nodes (bathgpu_set_long_models); without it the context refuses profiles past 1024"""
        self.lib = load()
        h = C.c_void_p()
        st = self.lib.bathgpu_create(device, C.byref(h))
        if st != OK:
            raise BathGpuError(st, "bathgpu_create failed (no usable CUDA device?)")
        self.h = h
        if long_models:
            self._check(self.lib.bathgpu_set_long_models(self.h, 1))

    def close(self):
        if getattr(self, "h", None):
            self.lib.bathgpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st):
        if st != OK:
            raise BathGpuError(st, self.lib.bathgpu_last_error(self.h).decode())

    def device_info(self):
        sm, khz, mem = C.c_int(), C.c_int(), C.c_size_t()
        self._check(self.lib.bathgpu_device_info(self.h, C.byref(sm), C.byref(khz), C.byref(mem)))
        return {"sm_count": sm.value, "clock_khz": khz.value, "total_mem": mem.value}

    def load_fs_profile(self, which, rfv, tfv):
        rfv = np.ascontiguousarray(rfv, dtype=np.float32)
        tfv = np.ascontiguousarray(tfv, dtype=np.float32)
        nrows, ld = rfv.shape
        assert tfv.shape == (8, ld)
        self._check(self.lib.bathgpu_load_fs_profile(self.h, which, ld - 1, nrows, _f(rfv), _f(tfv)))

    def load_fs_profile_set(self, which, profiles):
        """bathgpu_load_fs_profile_set: profiles = [(rfv [nrows][M+1], tfv [8][M+1]), ...] of one codon length"""
        rf = [np.ascontiguousarray(r, dtype=np.float32) for r, _ in profiles]
        tf = [np.ascontiguousarray(t, dtype=np.float32) for _, t in profiles]
        n = len(rf)
        assert all(t.shape == (8, r.shape[1]) for r, t in zip(rf, tf))
        M = np.array([r.shape[1] - 1 for r in rf], np.int32)
        nrows = np.array([r.shape[0] for r in rf], np.int32)
        fp = C.POINTER(C.c_float)
        self._check(self.lib.bathgpu_load_fs_profile_set(self.h, which, n, _i(M), _i(nrows), (fp * n)(*[_f(r) for r in rf]),
                                                         (fp * n)(*[_f(t) for t in tf])))

    @staticmethod
    def make_set_windows(starts, lengths, profiles, nj=1.0):
        """bathgpu_set_window descriptors: make_windows' length model, window w scored with profile profiles[w] of the set"""
        w = np.zeros(len(starts), dtype=set_window_dtype)
        base = Context.make_windows(starts, lengths, nj)
        for f in ("start", "L", "pmove", "ploop"):
            w[f] = base[f]
        w["profile"] = profiles
        return w

    def fs_set_scores(self, which, wins, xfE):
        """bathgpu_fs_set_scores over the loaded set of this codon length: xfE [n_profiles][2]; returns (scores, status)"""
        wins = np.ascontiguousarray(wins, set_window_dtype)
        n = len(wins)
        sc, st = np.empty(n, np.float32), np.empty(n, np.int32)
        xf = np.ascontiguousarray(xfE, np.float32)
        self._check(self.lib.bathgpu_fs_set_scores(self.h, which, wins.ctypes.data, n, _f(xf), _f(sc), _i(st)))
        return sc, st

    def select_slot(self, slot):
        self._check(self.lib.bathgpu_select_slot(self.h, slot))

    def upload_block(self, dsq):
        dsq = np.ascontiguousarray(dsq, dtype=np.uint8)
        self._check(self.lib.bathgpu_upload_block(self.h, dsq.ctypes.data_as(C.POINTER(C.c_uint8)), len(dsq) - 2))

    def upload_block_segments(self, pieces):
        """bathgpu_upload_block_segments: arrays of nucleotide codes (no sentinels) that follow one another in the resident block"""
        pieces = [np.ascontiguousarray(p, dtype=np.uint8) for p in pieces]
        ptrs = (C.POINTER(C.c_uint8) * len(pieces))(*[p.ctypes.data_as(C.POINTER(C.c_uint8)) for p in pieces])
        lens = (C.c_int64 * len(pieces))(*[len(p) for p in pieces])
        self._check(self.lib.bathgpu_upload_block_segments(self.h, ptrs, lens, len(pieces)))

    def upload_block_packed4(self, packed, n):
        """bathgpu_upload_block_packed4: a block already packed two nucleotides per byte (pack_dna4)"""
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        assert len(packed) >= (n + 1) // 2
        self._check(self.lib.bathgpu_upload_block_packed4(self.h, packed.ctypes.data_as(C.POINTER(C.c_uint8)), n))

    def fs_fwd_block_packed4_into(self, packed, n, wins, xfE, sc, st):
        """bathgpu_fs_fwd_block_packed4: upload (half the bytes, no packing kernel) and score in one call, into caller-owned arrays"""
        xf = np.asarray(xfE, np.float32)
        self._check(self.lib.bathgpu_fs_fwd_block_packed4(self.h, packed.ctypes.data_as(C.POINTER(C.c_uint8)), n, wins.ctypes.data, len(wins),
                                                          _f(xf), _f(sc), _i(st)))

    @staticmethod
    def make_windows(starts, lengths, nj=1.0):
        """Window descriptors with the length model of p7_fs_oprofile_ReconfigLength(om, L/3)
        (src/impl_sse/p7_fs_oprofile.c:636-651), computed in float32 as the reference does."""
        w = np.zeros(len(starts), dtype=window_dtype)
        w["start"] = starts
        w["L"] = lengths
        La = (np.asarray(lengths) // 3).astype(np.float32)
        njf = np.float32(nj)
        pmove = (np.float32(2.0) + njf) / (La + np.float32(2.0) + njf)
        w["pmove"] = pmove.astype(np.float32)
        w["ploop"] = (np.float32(1.0) - pmove).astype(np.float32)
        return w

    def fs_fwd_windows(self, wins, xfE=(0.5, 0.5)):
        n = len(wins)
        sc = np.empty(n, np.float32)
        st = np.empty(n, np.int32)
        xf = np.asarray(xfE, np.float32)
        self._check(self.lib.bathgpu_fs_fwd_windows(self.h, wins.ctypes.data, n, _f(xf), _f(sc), _i(st)))
        return sc, st

    def fs_fwd_windows_into(self, wins, xfE, sc, st):
        """Same call writing into caller-owned (e.g. pinned) score/status arrays."""
        xf = np.asarray(xfE, np.float32)
        self._check(self.lib.bathgpu_fs_fwd_windows(self.h, wins.ctypes.data, len(wins), _f(xf), _f(sc), _i(st)))

    def fs_fwd_block_into(self, dsq, wins, xfE, sc, st):
        """bathgpu_fs_fwd_block: upload and score in one call (upload overlapped with the kernel), into caller-owned arrays"""
        xf = np.asarray(xfE, np.float32)
        d = np.ascontiguousarray(dsq, np.uint8)
        self._check(self.lib.bathgpu_fs_fwd_block(self.h, d.ctypes.data_as(C.POINTER(C.c_uint8)), len(d) - 2, wins.ctypes.data, len(wins),
                                                  _f(xf), _f(sc), _i(st)))

    def stage_windows(self, wins):
        self._check(self.lib.bathgpu_stage_windows(self.h, wins.ctypes.data, len(wins)))

    def fs_fwd_staged(self, xfE=(0.5, 0.5)):
        xf = np.asarray(xfE, np.float32)
        self._check(self.lib.bathgpu_fs_fwd_staged(self.h, _f(xf)))

    def fetch_scores(self, n):
        sc = np.empty(n, np.float32)
        st = np.empty(n, np.int32)
        self._check(self.lib.bathgpu_fetch_scores(self.h, _f(sc), _i(st), n))
        return sc, st

    def last_stage_timing(self):
        ms, nl = C.c_float(), C.c_int()
        self._check(self.lib.bathgpu_last_stage_timing(self.h, C.byref(ms), C.byref(nl)))
        return ms.value, nl.value

    def measure_fp32_peak(self):
        tf, mhz = C.c_double(), C.c_double()
        self._check(self.lib.bathgpu_measure_fp32_peak(self.h, C.byref(tf), C.byref(mhz)))
        return tf.value, mhz.value

    def fs_bck_decode(self, wins, xfE, xf5_loop):
        n = len(wins)
        Ls = wins["L"].astype(np.int64)
        off = np.zeros(n, np.int64)
        off[1:] = np.cumsum(Ls[:-1] + 1)
        tot = int((Ls + 1).sum())
        mocc, btot, etot = (np.zeros(tot, np.float32) for _ in range(3))
        fsc, bsc, st = np.empty(n, np.float32), np.empty(n, np.float32), np.empty(n, np.int32)
        xf = np.asarray(xfE, np.float32)
        x5 = np.asarray(xf5_loop, np.float32)
        self._check(self.lib.bathgpu_fs_bck_decode(self.h, wins.ctypes.data, n, _f(xf), _f(x5),
                                                   off.ctypes.data_as(C.POINTER(C.c_int64)),
                                                   _f(mocc), _f(btot), _f(etot), _f(fsc), _f(bsc), _i(st)))
        split = lambda a: [a[off[w]: off[w] + Ls[w] + 1] for w in range(n)]
        return split(mocc), split(btot), split(etot), fsc, bsc, st

    def fs_fetch_xrows(self, which, wins):
        """X rows of the Forward (0) / Backward (1) parser for the windows of the last fs_bck_decode call -> list of [L+1][6]"""
        Ls = wins["L"].astype(np.int64)
        tot = int((Ls + 1).sum())
        out = np.empty((tot, 6), np.float32)
        self._check(self.lib.bathgpu_fs_fetch_xrows(self.h, which, _f(out), tot))
        off = np.concatenate([[0], np.cumsum(Ls + 1)])
        return [out[off[w]: off[w + 1]] for w in range(len(wins))]

    def fs_fetch_domain_matrices(self, e, M, L):
        pp = np.empty((L + 1, M + 1, 8), np.float32)
        oa = np.empty((L + 1, M + 1, 3), np.float32)
        ppx = np.empty((L + 1, 6), np.float32)
        oax = np.empty((L + 1, 6), np.float32)
        self._check(self.lib.bathgpu_fs_fetch_domain_matrices(self.h, e, _f(pp), _f(oa), _f(ppx), _f(oax)))
        return pp, oa, ppx, oax

    def load_filter_profile(self, params, rbv, rwv, twv):
        """params: dict with the FilterParams fields; rbv [29][M+1] u8, rwv [29][M+1] i16, twv [8][M+1] i16"""
        prm = FilterParams(**params)
        rbv = np.ascontiguousarray(rbv, np.uint8)
        rwv = np.ascontiguousarray(rwv, np.int16)
        twv = np.ascontiguousarray(twv, np.int16)
        self._check(self.lib.bathgpu_load_filter_profile(self.h, C.byref(prm), rbv.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                         rwv.ctypes.data_as(C.POINTER(C.c_int16)),
                                                         twv.ctypes.data_as(C.POINTER(C.c_int16))))

    def upload_orfs(self, residues):
        residues = np.ascontiguousarray(residues, np.uint8)
        self._check(self.lib.bathgpu_upload_orfs(self.h, residues.ctypes.data_as(C.POINTER(C.c_uint8)), len(residues)))

    def msv_orfs(self, orfs):
        n = len(orfs)
        sc, st = np.empty(n, np.float32), np.empty(n, np.int32)
        self._check(self.lib.bathgpu_msv_orfs(self.h, orfs.ctypes.data, n, _f(sc), _i(st)))
        return sc, st

    def ssv_windows(self, orfs, max_wins=None):
        max_wins = max_wins or (16 * len(orfs) + 64)
        w = np.zeros(max_wins, orf_window_dtype)
        nw = C.c_int32()
        self._check(self.lib.bathgpu_ssv_windows(self.h, orfs.ctypes.data, len(orfs), w.ctypes.data, max_wins, C.byref(nw)))
        return w[: nw.value]

    def vit_orfs(self, orfs, max_wins=None):
        n = len(orfs)
        max_wins = max_wins or (16 * n + 64)
        sc, st = np.empty(n, np.float32), np.empty(n, np.int32)
        w = np.zeros(max_wins, orf_window_dtype)
        nw = C.c_int32()
        self._check(self.lib.bathgpu_vit_orfs(self.h, orfs.ctypes.data, n, _f(sc), _i(st), w.ctypes.data, max_wins, C.byref(nw)))
        return sc, st, w[: nw.value]

    def fwd_orfs(self, orfs, nj=1.0, xfE=(0.5, 0.5)):
        n = len(orfs)
        sc, st = np.empty(n, np.float32), np.empty(n, np.int32)
        xf = np.asarray(xfE, np.float32)
        self._check(self.lib.bathgpu_fwd_orfs(self.h, orfs.ctypes.data, n, nj, _f(xf), _f(sc), _i(st)))
        return sc, st

    def fs_fwd_bck_xrows(self, wins, xfE=(0.5, 0.5)):
        n = len(wins)
        Ls = wins["L"].astype(np.int64)
        tot = int((Ls + 1).sum())
        fx, bx = np.empty((tot, 6), np.float32), np.empty((tot, 6), np.float32)
        fsc, bsc, st = np.empty(n, np.float32), np.empty(n, np.float32), np.empty(n, np.int32)
        xf = np.asarray(xfE, np.float32)
        self._check(self.lib.bathgpu_fs_fwd_bck_xrows(self.h, wins.ctypes.data, n, _f(xf), _f(fx), _f(bx), _f(fsc), _f(bsc), _i(st)))
        off = np.concatenate([[0], np.cumsum(Ls + 1)])
        return [fx[off[w]: off[w + 1]] for w in range(n)], [bx[off[w]: off[w + 1]] for w in range(n)], fsc, bsc, st

    def revcomp_slot(self, src, dst):
        self._check(self.lib.bathgpu_revcomp_slot(self.h, int(src), int(dst)))

    def orf_forward_matrices(self, regs, M, xfE=(0.5, 0.5)):
        """bathgpu_orf_forward_matrices: per region the matrix [(L+1)][(M+1)][4] {M, D, I, 0} and the X rows [(L+1)][6]; scores; status"""
        n = len(regs)
        Ls = regs["L"].astype(np.int64)
        off = np.concatenate([[0], np.cumsum(Ls + 1)])
        mx = np.zeros((int(off[-1]), M + 1, 4), np.float32)
        xr = np.zeros((int(off[-1]), 6), np.float32)
        sc, st = np.empty(n, np.float32), np.empty(n, np.int32)
        xf = np.asarray(xfE, np.float32)
        self._check(self.lib.bathgpu_orf_forward_matrices(self.h, regs.ctypes.data, n, _f(xf), _f(mx), _f(xr), int(off[-1]), _f(sc), _i(st)))
        return [mx[off[r]: off[r + 1]] for r in range(n)], [xr[off[r]: off[r + 1]] for r in range(n)], sc, st

    def measure_int16_peak(self):
        t = C.c_double(0)
        self._check(self.lib.bathgpu_measure_int16_peak(self.h, C.byref(t)))
        return float(t.value)

    def orfs_stage_breakdown(self):
        """(ms of [classes, count pass, emit pass, MSV, screen], ORFs found, residues scored) of the last orfs_msv_screen call"""
        ms = np.zeros(5, np.float32)
        no, nr = C.c_int64(0), C.c_int64(0)
        self._check(self.lib.bathgpu_orfs_stage_breakdown(self.h, _f(ms), C.byref(no), C.byref(nr)))
        return ms, int(no.value), int(nr.value)

    def bias_forward(self, kind, items, tables, t10, t11, gcode=None):
        """bathgpu_bias_forward: items = bias_item_dtype array; tables [ntab][29][2]; returns n (kind 0) or n x 3 (kind 1) scores"""
        items = np.ascontiguousarray(items, bias_item_dtype)
        tables = np.ascontiguousarray(tables, np.float32).reshape(-1, KP, 2)
        out = np.zeros(len(items) * (3 if kind == 1 else 1), np.float32)
        g = np.ascontiguousarray(gcode if gcode is not None else np.zeros(64), np.uint8)
        self._check(self.lib.bathgpu_bias_forward(self.h, int(kind), items.ctypes.data_as(C.c_void_p), len(items), _f(tables), len(tables),
                                                  float(t10), float(t11), g.ctypes.data_as(C.POINTER(C.c_uint8)), _f(out)))
        return out.reshape(-1, 3) if kind == 1 else out

    def orfs_msv_screen(self, blocks, complement, gcode, min_len, tjb_of, null_of, min_bits):
        """bathgpu_orfs_msv_screen + bathgpu_orfs_fetch: (ORFs found per block, survivors, their residues)"""
        nb = len(blocks)
        gcode = np.ascontiguousarray(gcode, np.uint8)
        tjb_of = np.ascontiguousarray(tjb_of, np.uint8)
        null_of = np.ascontiguousarray(null_of, np.float32)
        per = np.zeros(nb, np.int64)
        nh, nr = C.c_int64(), C.c_int64()
        u8 = C.POINTER(C.c_uint8)
        self._check(self.lib.bathgpu_orfs_msv_screen(self.h, blocks.ctypes.data, nb, int(complement), gcode.ctypes.data_as(u8), int(min_len),
                                                     tjb_of.ctypes.data_as(u8), _f(null_of), len(tjb_of) - 1, float(min_bits),
                                                     per.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(nh), C.byref(nr)))
        hits = np.zeros(max(nh.value, 1), orf_hit_dtype)
        res = np.zeros(max(nr.value, 1), np.uint8)
        self._check(self.lib.bathgpu_orfs_fetch(self.h, hits.ctypes.data, res.ctypes.data_as(u8)))
        return per, hits[: nh.value], res[: nr.value]

    def load_filter_profile_set(self, profiles):
        """bathgpu_load_filter_profile_set: profiles = [(params dict with the FilterParams fields, rbv [29][M+1] u8), ...]"""
        n = len(profiles)
        prm = (FilterParams * n)(*[FilterParams(**p) for p, _ in profiles])
        rbv = [np.ascontiguousarray(r, np.uint8) for _, r in profiles]
        u8 = C.POINTER(C.c_uint8)
        self._check(self.lib.bathgpu_load_filter_profile_set(self.h, n, C.cast(prm, C.c_void_p), (u8 * n)(*[r.ctypes.data_as(u8) for r in rbv])))

    def orfs_msv_screen_set(self, jobs, complement, gcode, min_len, tjb_of, null_of):
        """bathgpu_orfs_msv_screen_set + bathgpu_orfs_fetch_set over jobs = [(profile, blocks (block_dtype array), min_bits), ...]:
        per job (ORFs found per block, survivors, the residues each survivor's offset indexes -- one buffer shared by all jobs)"""
        n = len(jobs)
        blocks = [np.ascontiguousarray(b, block_dtype) for _, b, _ in jobs]
        jd = (ScreenJob * n)(*[ScreenJob(int(p), len(b), b.ctypes.data, float(mb)) for (p, _, mb), b in zip(jobs, blocks)])
        gcode = np.ascontiguousarray(gcode, np.uint8)
        tjb_of = np.ascontiguousarray(tjb_of, np.uint8)
        null_of = np.ascontiguousarray(null_of, np.float32)
        nblk = [len(b) for b in blocks]
        per = np.zeros(max(sum(nblk), 1), np.int64)
        nh, nr = np.zeros(n, np.int64), np.zeros(n, np.int64)
        u8, i64 = C.POINTER(C.c_uint8), C.POINTER(C.c_int64)
        self._check(self.lib.bathgpu_orfs_msv_screen_set(self.h, C.cast(jd, C.c_void_p), n, int(complement), gcode.ctypes.data_as(u8), int(min_len),
                                                         tjb_of.ctypes.data_as(u8), _f(null_of), len(tjb_of) - 1, per.ctypes.data_as(i64),
                                                         nh.ctypes.data_as(i64), nr.ctypes.data_as(i64)))
        hits = np.zeros(max(int(nh.sum()), 1), orf_hit_dtype)
        res = np.zeros(max(int(nr.sum()), 1), np.uint8)
        self._check(self.lib.bathgpu_orfs_fetch_set(self.h, hits.ctypes.data, res.ctypes.data_as(u8)))
        out, z, b0 = [], 0, 0
        for j in range(n):
            out.append((per[b0: b0 + nblk[j]], hits[z: z + nh[j]], res[: int(nr.sum())]))
            z += int(nh[j]); b0 += nblk[j]
        return out

    def orf_fwd_bck_xrows(self, orfs, nj=1.0, xfE=(0.5, 0.5)):
        n = len(orfs)
        Ls = orfs["L"].astype(np.int64)
        tot = int((Ls + 1).sum())
        fx, bx = np.empty((tot, 6), np.float32), np.empty((tot, 6), np.float32)
        fsc, bsc, st = np.empty(n, np.float32), np.empty(n, np.float32), np.empty(n, np.int32)
        xf = np.asarray(xfE, np.float32)
        self._check(self.lib.bathgpu_orf_fwd_bck_xrows(self.h, orfs.ctypes.data, n, C.c_float(nj), _f(xf), _f(fx), _f(bx), _f(fsc), _f(bsc), _i(st)))
        off = np.concatenate([[0], np.cumsum(Ls + 1)])
        return [fx[off[w]: off[w + 1]] for w in range(n)], [bx[off[w]: off[w + 1]] for w in range(n)], fsc, bsc, st

    def orf_domains(self, envs, xfE=(1.0, 0.0), max_steps=None, M=0):
        n = len(envs)
        if max_steps is None:
            max_steps = int((envs["L"].astype(np.int64) + M + 8).sum())
        res = np.zeros(n, dtype=domain_dtype)
        tr = np.zeros(max_steps, dtype=trace_dtype)
        xf = np.asarray(xfE, np.float32)
        self._check(self.lib.bathgpu_orf_domains(self.h, envs.ctypes.data, n, _f(xf), res.ctypes.data, tr.ctypes.data, C.c_int64(max_steps)))
        return res, tr

    def orf_fetch_domain_matrices(self, e, L, M):
        pp = np.empty((L + 1, M + 1, 3), np.float32)
        oa = np.empty((L + 1, M + 1, 3), np.float32)
        ppx = np.empty((L + 1, 6), np.float32)
        oax = np.empty((L + 1, 6), np.float32)
        self._check(self.lib.bathgpu_orf_fetch_domain_matrices(self.h, e, _f(pp), _f(oa), _f(ppx), _f(oax)))
        return pp, oa, ppx, oax

    def fs_forward_matrices(self, regs, M, xfE5=(0.5, 0.5)):
        """bathgpu_fs_forward_matrices: (mx [rows][(M+1)][8], xrows [rows][6], row offsets, fwdsc, status)"""
        n = len(regs)
        off = np.concatenate([[0], np.cumsum(regs["L"].astype(np.int64) + 1)])
        rows = int(off[-1])
        mx = np.empty((rows, M + 1, 8), np.float32)
        xr = np.empty((rows, 6), np.float32)
        sc = np.empty(n, np.float32)
        st = np.empty(n, np.int32)
        xf = np.asarray(xfE5, np.float32)
        self._check(self.lib.bathgpu_fs_forward_matrices(self.h, regs.ctypes.data, n, _f(xf), _f(mx), _f(xr), rows, _f(sc), _i(st)))
        return mx, xr, off, sc, st

    def fs_domains(self, envs, xfE5=(1.0, 0.0), max_steps=None):
        n = len(envs)
        if max_steps is None:
            max_steps = int((envs["L"].astype(np.int64) + 8).sum())
        res = np.zeros(n, dtype=domain_dtype)
        tr = np.zeros(max_steps, dtype=trace_dtype)
        xf = np.asarray(xfE5, np.float32)
        self._check(self.lib.bathgpu_fs_domains(self.h, envs.ctypes.data, n, _f(xf), res.ctypes.data, tr.ctypes.data,
                                                max_steps))
        return res, tr


def pack_dna4(dsq, out=None):
    """bathgpu_pack_dna4: ESL_DSQ bytes (sentinels at both ends) -> two nucleotides per byte, the form bathgpu_upload_block_packed4 and
    bathgpu_fs_fwd_block_packed4 take"""
    L = load()
    dsq = np.ascontiguousarray(dsq, np.uint8)
    n = len(dsq) - 2
    if out is None:
        out = np.empty(int(L.bathgpu_packed4_bytes(n)), np.uint8)
    st = L.bathgpu_pack_dna4(dsq.ctypes.data_as(C.POINTER(C.c_uint8)), n, out.ctypes.data_as(C.POINTER(C.c_uint8)))
    if st != 0:
        raise RuntimeError(f"bathgpu_pack_dna4: status {st}")
    return out
