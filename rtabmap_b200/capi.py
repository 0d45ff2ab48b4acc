"""ctypes binding of include/lcd_b200.h (the C ABI of liblcd_b200.so).

This is the binding a Python host would use; INTEGRATION.md shows the equivalent C++ shim
for the reference.  Every method maps 1:1 onto an ``lcd_*`` entry point and raises
:class:`LcdError` with ``lcd_last_error`` on a non-zero status.  Nothing here computes:
if the library is missing it is built (nvcc); if no CUDA device is present ``Engine()`` raises.
"""
from __future__ import annotations

import ctypes as C
import os
import sys
from pathlib import Path

import numpy as np

from . import build as _build

LCD_OK = 0
LCD_DESC_U8 = 0
LCD_DESC_F32 = 1

_lib = None


class LcdError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"lcd_b200 error {code}: {msg}")
        self.code = code


class _Config(C.Structure):
    _fields_ = [
        ("device", C.c_int),
        ("desc_type", C.c_int),
        ("desc_dim", C.c_int),
        ("max_words", C.c_int),
        ("max_signatures", C.c_int),
        ("max_queries", C.c_int),
        ("max_batch", C.c_int),
    ]


class Keypoint(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("size", C.c_float), ("angle", C.c_float), ("response", C.c_float), ("octave", C.c_int)]


class OrbParams(C.Structure):
    """lcd_orb_params (Kp/*, ORB/*, FAST/*, Mem/DepthAsMask parameters of the reference)."""
    _fields_ = [
        ("n_features", C.c_int), ("n_levels", C.c_int), ("scale_factor", C.c_float), ("edge_threshold", C.c_int),
        ("fast_threshold", C.c_int), ("patch_size", C.c_int), ("min_depth", C.c_float), ("max_depth", C.c_float),
        ("depth_as_mask", C.c_int), ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
    ]


class GfttParams(C.Structure):
    """lcd_gftt_params (GFTT/* parameters of the reference, corelib/include/rtabmap/core/Parameters.h:313-317)."""
    _fields_ = [
        ("quality_level", C.c_double), ("min_distance", C.c_double), ("block_size", C.c_int), ("use_harris", C.c_int), ("k", C.c_double),
    ]


LCD_DETECTOR_ORB = 2
LCD_DETECTOR_GFTT_ORB = 8


class VerifyParams(C.Structure):
    """lcd_verify_params (Vis/* parameters of the reference, corelib/include/rtabmap/core/Parameters.h:713-754)."""
    _fields_ = [
        ("nndr", C.c_float),
        ("min_inliers", C.c_int),
        ("iterations", C.c_int),
        ("reproj_error", C.c_float),
        ("refine_iterations", C.c_int),
        ("refine_sigma", C.c_float),
        ("fx", C.c_double),
        ("fy", C.c_double),
        ("cx", C.c_double),
        ("cy", C.c_double),
        ("var_median_ratio", C.c_int),
        ("max_variance", C.c_float),
        ("split_linear_cov", C.c_int),
        ("image_width", C.c_int),
        ("image_height", C.c_int),
        ("repeat_once", C.c_int),
        ("guess_win_size", C.c_int),
    ]


class VerifyResult(C.Structure):
    _fields_ = [
        ("ok", C.c_int),
        ("n_matches", C.c_int),
        ("n_inliers", C.c_int),
        ("iterations_run", C.c_int),
        ("rvec", C.c_double * 3),
        ("tvec", C.c_double * 3),
        ("transform", C.c_float * 12),
        ("covariance", C.c_double * 36),
    ]


def library_path() -> Path:
    return _build.LIB


_P = C.c_void_p
_I = C.c_int
_F = C.c_float
_IP = C.POINTER(C.c_int)
_FP = C.POINTER(C.c_float)

# name -> (restype, argtypes); kept in the order of include/lcd_b200.h
SIGNATURES = {
    "lcd_create": (_P, [C.POINTER(_Config)]),
    "lcd_destroy": (None, [_P]),
    "lcd_last_error": (C.c_char_p, [_P]),
    "lcd_abi_version": (_I, []),
    "lcd_build_arch": (C.c_char_p, []),
    "lcd_launch_count": (C.c_longlong, [_P]),
    "lcd_orb_detect_describe": (_I, [_P, _I, _P, _I, _I, _I, _P, _I, _P, _I, _P, _P, _P, _P]),
    "lcd_orb_detect_describe_dev": (_I, [_P, _I, _P, _I, _I, _I, _P, _I, _P, _I, _P, _P, _P, _P, _P, _P]),
    "lcd_orb_overflow": (_I, [_P]),
    "lcd_orb_last_path": (_I, [_P]),
    "lcd_set_detector": (_I, [_P, _I, _P]),
    "lcd_dict_add_words": (_I, [_P, _P, _P, _I]),
    "lcd_dict_remove_words": (_I, [_P, _P, _I]),
    "lcd_dict_update": (_I, [_P]),
    "lcd_dict_clear": (_I, [_P]),
    "lcd_dict_size": (_I, [_P]),
    "lcd_dict_indexed_size": (_I, [_P]),
    "lcd_dict_not_indexed_size": (_I, [_P]),
    "lcd_dict_last_word_id": (_I, [_P]),
    "lcd_dict_set_last_word_id": (_I, [_P, _I]),
    "lcd_dict_has_word": (_I, [_P, _I]),
    "lcd_dict_get_indexed": (_I, [_P, _P, _P, _I]),
    "lcd_nn_select": (_I, [_P, _I]),
    "lcd_nn_last_kernel": (_I, [_P]),
    "lcd_nn_f32_stats": (_I, [_P, _I, _P, _P, _P]),
    "lcd_dict_knn2": (_I, [_P, _P, _I, _P, _P, _P, _P]),
    "lcd_dict_quantize": (_I, [_P, _P, _I, _I, _I, _F, _I, _P, _P]),
    "lcd_dict_find_nn": (_I, [_P, _P, _I, _I, _F, _P]),
    "lcd_index_add_refs": (_I, [_P, _I, _P, _I]),
    "lcd_index_remove_sig": (_I, [_P, _I]),
    "lcd_index_set_ni": (_I, [_P, _P, _P, _I]),
    "lcd_index_load_csr": (_I, [_P, _P, _I, _P, _P, _P]),
    "lcd_index_word_nw": (_I, [_P, _I]),
    "lcd_index_total_refs": (C.c_longlong, [_P]),
    "lcd_index_get_refs": (_I, [_P, _I, _P, _P, _I]),
    "lcd_index_score": (_I, [_P, _P, _I, _P, _I, _I, _P]),
    "lcd_adjust_likelihood": (_I, [_P, _P, _I, _I, _I, _P]),
    "lcd_adjust_likelihood_dev": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "lcd_bayes_compute_posterior": (_I, [_P, _P, _P, _I, _P, _P, _P, _P, _I, _F, _P]),
    "lcd_bayes_reset": (_I, [_P]),
    "lcd_localize_batch": (_I, [_P, _P, _I, _I, _I, _F, _I, _P, _I, _I, _P, _P]),
    "lcd_localize_batch_dev": (_I, [_P, _P, _I, _I, _I, _F, _I, _P, _I, _I, _P, _P, _P]),
    "lcd_match_pairs": (_I, [_P, _I, _I, _P, _P, _P, _P, _F, _P, _P]),
    "lcd_verify_batch": (_I, [_P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "lcd_pnp_ransac": (_I, [_P, _P, _P, _I, _P, _P, _I, _P, _P, _I, _I, _F, _I, _I, _I, _F, _P, _P]),
    "lcd_pnp_ransac_batch": (_I, [_P, _I, _I, _P, _P, _P, _P, _P, _I, _P, _P, _I, _I, _F, _I, _I, _I, _F, _P, _P, _P]),
    "lcd_match_bf": (_I, [_P, _I, _I, _P, _P, _P, _P, _I, _P, _P, _P, _P]),
    "lcd_sig_add_batch": (_I, [_P, _P, _I, _I, _P, _P, _P]),
    "lcd_sig_remove": (_I, [_P, _I]),
    "lcd_sig_count": (_I, [_P]),
    "lcd_sig_slots": (_I, [_P]),
    "lcd_process_batch": (_I, [_P, _P, _P, _I, _I, _I, _F, _I, _P, _I, _I, _P, _P, _P, _P, _P]),
    "lcd_process_batch_dev": (_I, [_P, _P, _P, _I, _I, _I, _F, _I, _P, _I, _I, _P, _P, _P, _P]),
    "lcd_process_fetch": (_I, [_P, _I, _P, _P]),
    "lcd_process_fetch_async": (_I, [_P, _I, _P, _P, _P]),
    "lcd_process_frames": (_I, [_P, _I, _P, _I, _I, _I, _P, _I, _P, _I, _F, _I, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "lcd_process_frames_submit": (_I, [_P, _I, _P, _I, _I, _I, _P, _I, _P, _I, _F, _I, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "lcd_process_frames_wait": (_I, [_P]),
    "lcd_process_frames_dev": (_I, [_P, _I, _P, _I, _I, _I, _P, _I, _P, _I, _F, _I, _P, _I, _I, _P, _P, _P, _P]),
    "lcd_map_detect_async": (_I, [_P, _P, _I, _I, _I, _P, _I, _P]),
    "lcd_map_frame": (_I, [_P, _I, _I, _F, _I, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "lcd_verify_top_dev": (_I, [_P, _P, _P, _I, _I, _P, _P, _I, _P, _P]),
    "lcd_shard_set_row_offset": (_I, [_P, _I]),
    "lcd_shard_knn2_keys_dev": (_I, [_P, _P, _I, _P, _P]),
    "lcd_shard_resolve_score_dev": (_I, [_P, _P, _I, _I, _P, _I, _P, _I, _I, _I, _F, _I, _P, _I, _I, _P, _P, _P]),
    "lcd_shard_resolve_frames_dev": (_I, [_P, _P, _I, _I, _I, _I, _P, _I, _P, _I, _I, _F, _I, _P, _P, _P]),
    "lcd_shard_score_ids_dev": (_I, [_P, _P, _I, _I, _P, _I, _I, _P, _P]),
    "lcd_shard_finalize_dev": (_I, [_P, _P, _I, _P, _P]),
    "lcd_shard_unique_id": (_I, [_P]),
    "lcd_shard_comm_init": (_I, [_P, _P, _I, _I]),
    "lcd_shard_comm_adopt": (_I, [_P, _P, _I, _I]),
    "lcd_shard_comm_destroy": (_I, [_P]),
    "lcd_shard_process_frames_dev": (_I, [_P, _I, _P, _I, _I, _I, _P, _I, _P, _I, _F, _I, _P, _I, _I, _P, _I, _P, _P, _P, _P]),
    "lcd_profile_enable": (_I, [_P, _I]),
    "lcd_profile_read": (_I, [_P, _I, _P, _P]),
    "lcd_profile_reset": (_I, [_P]),
    "lcd_debug_orb_buffer": (C.c_longlong, [_P, _I, _P, C.c_longlong]),
    "lcd_stream": (_P, [_P]),
    "lcd_synchronize": (_I, [_P]),
}


def load_library(build_if_missing: bool = True) -> C.CDLL:
    """dlopen liblcd_b200.so (building it with nvcc first if needed) and set prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if build_if_missing and _build.needs_build():
        # one process may rebuild a stale library in place; the ranks of a multi-process job must not race each other on the same file
        if not path.exists() or int(os.environ.get("WORLD_SIZE", "1")) <= 1:
            _build.build()
        else:
            print(f"rtabmap_b200: {path} is older than its sources; not rebuilding inside a {os.environ.get('WORLD_SIZE')}-process job", file=sys.stderr)
    if not path.exists():
        raise LcdError(-2, f"{path} is missing: the CUDA extension must be built (python -m rtabmap_b200.build)")
    lib = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.int32)


class Engine:
    """One device-resident dictionary + inverted index (``lcd_engine``)."""

    def __init__(self, device: int = 0, desc_type: int = LCD_DESC_U8, desc_dim: int = 32, max_words: int = 65536,
                 max_signatures: int = 16384, max_queries: int = 1024, max_batch: int = 64):
        self._lib = load_library()
        cfg = _Config(device, desc_type, desc_dim, max_words, max_signatures, max_queries, max_batch)
        self._h = self._lib.lcd_create(C.byref(cfg))
        if not self._h:
            raise LcdError(-2, self._lib.lcd_last_error(None).decode())
        self.desc_type = desc_type
        self.desc_dim = desc_dim
        self.device = device

    # -- plumbing ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.lcd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise LcdError(rc, self._lib.lcd_last_error(self._h).decode())

    def _desc(self, d) -> np.ndarray:
        dt = np.uint8 if self.desc_type == LCD_DESC_U8 else np.float32
        d = np.ascontiguousarray(d, dtype=dt)
        if d.ndim != 2 or d.shape[1] != self.desc_dim:
            raise LcdError(-1, f"descriptors must be [n,{self.desc_dim}] {dt.__name__}, got {d.shape}")
        return d

    @property
    def handle(self):
        return self._h

    @property
    def launch_count(self) -> int:
        return int(self._lib.lcd_launch_count(self._h))

    @property
    def stream(self) -> int:
        return int(self._lib.lcd_stream(self._h) or 0)

    def synchronize(self):
        self._check(self._lib.lcd_synchronize(self._h))

    def profile_enable(self, on: bool = True):
        self._check(self._lib.lcd_profile_enable(self._h, int(on)))

    def profile_reset(self):
        self._check(self._lib.lcd_profile_reset(self._h))

    def profile_read(self, which: int):
        ms = C.c_double(0)
        n = C.c_longlong(0)
        self._check(self._lib.lcd_profile_read(self._h, which, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    # -- detect (ORB) ----------------------------------------------------------------------------
    @staticmethod
    def orb_params(K4=(525.0, 525.0, 320.0, 240.0), n_features=1000, n_levels=3, scale_factor=2.0, edge_threshold=19, fast_threshold=20,
                   patch_size=31, min_depth=0.0, max_depth=0.0, depth_as_mask=True):
        return OrbParams(n_features, n_levels, scale_factor, edge_threshold, fast_threshold, patch_size, min_depth, max_depth, int(depth_as_mask),
                         *[float(k) for k in K4])

    @staticmethod
    def gftt_params(quality_level=0.001, min_distance=7.0, block_size=3, use_harris=False, k=0.04):
        return GfttParams(float(quality_level), float(min_distance), int(block_size), int(use_harris), float(k))

    def set_detector(self, strategy: int, gftt: "GfttParams" = None):
        """Kp/DetectorStrategy of every later detection: LCD_DETECTOR_ORB (2) or LCD_DETECTOR_GFTT_ORB (8, needs ``gftt``)."""
        self._check(self._lib.lcd_set_detector(self._h, int(strategy), C.byref(gftt) if gftt is not None else None))

    def orb_detect_describe(self, images, depth, params: "OrbParams", cap: int = 0):
        """images [n,h,w] (gray) or [n,h,w,3] (BGR) uint8; depth [n,h,w] uint16 (mm) / float32 (m) / None.
        Returns per frame: (keypoints [k,6] float32 = x,y,size,angle,response,octave; desc [k,32]; xyz [k,3])."""
        img = np.ascontiguousarray(images, np.uint8)
        assert img.ndim in (3, 4)
        n, h, w = img.shape[:3]
        ch = 1 if img.ndim == 3 else img.shape[3]
        dtype = 0
        dptr = None
        if depth is not None:
            if depth.dtype == np.uint16:
                dtype, depth = 1, np.ascontiguousarray(depth)
            else:
                dtype, depth = 2, np.ascontiguousarray(depth, np.float32)
            dptr = _ptr(depth)
        cap = cap or (params.n_features + 256)
        kp = (Keypoint * (n * cap))()
        desc = np.zeros((n, cap, 32), np.uint8)
        xyz = np.zeros((n, cap, 3), np.float32)
        cnt = np.zeros(n, np.int32)
        self._check(self._lib.lcd_orb_detect_describe(self._h, n, _ptr(img), w, h, ch, dptr, dtype, C.byref(params), cap, kp, _ptr(desc), _ptr(xyz), _ptr(cnt)))
        kpa = np.frombuffer(kp, dtype=np.dtype([("x", "f4"), ("y", "f4"), ("size", "f4"), ("angle", "f4"), ("response", "f4"), ("octave", "i4")])).reshape(n, cap)
        out = []
        for i in range(n):
            k = kpa[i, :cnt[i]]
            arr = np.stack([k["x"], k["y"], k["size"], k["angle"], k["response"], k["octave"].astype(np.float32)], 1) if cnt[i] else np.zeros((0, 6), np.float32)
            out.append((arr, desc[i, :cnt[i]].copy(), xyz[i, :cnt[i]].copy()))
        return out

    def debug_orb_buffer(self, which: int, nbytes: int, dtype=np.uint8) -> np.ndarray:
        buf = np.zeros(nbytes, np.uint8)
        n = self._lib.lcd_debug_orb_buffer(self._h, which, _ptr(buf), nbytes)
        if n < 0:
            self._check(int(n))
        return buf[:n].view(dtype)

    # -- dictionary --------------------------------------------------------------------------
    def add_words(self, ids, desc):
        ids = _i32(ids)
        desc = self._desc(desc)
        assert len(ids) == len(desc)
        self._check(self._lib.lcd_dict_add_words(self._h, _ptr(ids), _ptr(desc), len(ids)))

    def remove_words(self, ids):
        ids = _i32(ids)
        self._check(self._lib.lcd_dict_remove_words(self._h, _ptr(ids), len(ids)))

    def update(self):
        self._check(self._lib.lcd_dict_update(self._h))

    def clear(self):
        self._check(self._lib.lcd_dict_clear(self._h))

    def size(self) -> int:
        return self._lib.lcd_dict_size(self._h)

    def indexed_size(self) -> int:
        return self._lib.lcd_dict_indexed_size(self._h)

    def not_indexed_size(self) -> int:
        return self._lib.lcd_dict_not_indexed_size(self._h)

    @property
    def last_word_id(self) -> int:
        return self._lib.lcd_dict_last_word_id(self._h)

    @last_word_id.setter
    def last_word_id(self, v: int):
        self._check(self._lib.lcd_dict_set_last_word_id(self._h, int(v)))

    def has_word(self, word_id: int) -> bool:
        return bool(self._lib.lcd_dict_has_word(self._h, int(word_id)))

    def get_indexed(self):
        n = self.indexed_size()
        ids = np.zeros(n, np.int32)
        dt = np.uint8 if self.desc_type == LCD_DESC_U8 else np.float32
        desc = np.zeros((n, self.desc_dim), dt)
        if n:
            r = self._lib.lcd_dict_get_indexed(self._h, _ptr(ids), _ptr(desc), n)
            if r < 0:
                self._check(r)
        return ids, desc

    def nn_select(self, kernel: int):
        """0 = XOR/POPC kernel, 1 = tensor-core kernel (default for 32-byte descriptors)."""
        self._check(self._lib.lcd_nn_select(self._h, int(kernel)))

    def nn_f32_stats(self, nq: int):
        """(queries redone by the exact fallback, candidate rows re-ranked, dictionary rows converted to fp16 so far) of the last float search."""
        fb = C.c_int(0)
        cand = C.c_longlong(0)
        conv = C.c_longlong(0)
        self._check(self._lib.lcd_nn_f32_stats(self._h, int(nq), C.byref(fb), C.byref(cand), C.byref(conv)))
        return fb.value, cand.value, conv.value

    @property
    def nn_last_kernel(self) -> int:
        return int(self._lib.lcd_nn_last_kernel(self._h))

    def knn2(self, queries):
        q = self._desc(queries)
        n = len(q)
        id1 = np.zeros(n, np.int32)
        id2 = np.zeros(n, np.int32)
        d1 = np.zeros(n, np.float32)
        d2 = np.zeros(n, np.float32)
        self._check(self._lib.lcd_dict_knn2(self._h, _ptr(q), n, _ptr(id1), _ptr(d1), _ptr(id2), _ptr(d2)))
        return id1, d1, id2, d2

    def quantize(self, queries, sig_id: int, incremental: bool = True, nndr: float = 0.8, cmp_new: bool = True):
        q = self._desc(queries)
        out = np.zeros(len(q), np.int32)
        n_new = C.c_int(0)
        self._check(self._lib.lcd_dict_quantize(self._h, _ptr(q), len(q), int(sig_id), int(incremental), float(nndr),
                                                 int(cmp_new), _ptr(out), C.byref(n_new)))
        return out, n_new.value

    def find_nn(self, queries, incremental: bool = True, nndr: float = 0.8):
        q = self._desc(queries)
        out = np.zeros(len(q), np.int32)
        self._check(self._lib.lcd_dict_find_nn(self._h, _ptr(q), len(q), int(incremental), float(nndr), _ptr(out)))
        return out

    # -- inverted index ----------------------------------------------------------------------
    def add_refs(self, sig_id: int, word_ids):
        w = _i32(word_ids)
        self._check(self._lib.lcd_index_add_refs(self._h, int(sig_id), _ptr(w), len(w)))

    def remove_sig(self, sig_id: int):
        self._check(self._lib.lcd_index_remove_sig(self._h, int(sig_id)))

    def set_ni(self, sig_ids, ni):
        s = _i32(sig_ids)
        n = _i32(ni)
        self._check(self._lib.lcd_index_set_ni(self._h, _ptr(s), _ptr(n), len(s)))

    def load_csr(self, word_ids, row_ptr, sig, cnt):
        w = _i32(word_ids)
        rp = np.ascontiguousarray(row_ptr, dtype=np.int64)
        s = _i32(sig)
        c = _i32(cnt)
        assert len(rp) == len(w) + 1 and len(s) == len(c) == rp[-1]
        self._check(self._lib.lcd_index_load_csr(self._h, _ptr(w), len(w), _ptr(rp), _ptr(s), _ptr(c)))

    def word_nw(self, word_id: int) -> int:
        return self._lib.lcd_index_word_nw(self._h, int(word_id))

    def total_refs(self) -> int:
        return int(self._lib.lcd_index_total_refs(self._h))

    def get_refs(self, word_id: int):
        n = self.word_nw(word_id)
        s = np.zeros(max(n, 1), np.int32)
        c = np.zeros(max(n, 1), np.int32)
        r = self._lib.lcd_index_get_refs(self._h, int(word_id), _ptr(s), _ptr(c), len(s))
        if r < 0:
            self._check(r)
        return s[:r], c[:r]

    def score(self, query_word_ids, sig_ids, n_total: int):
        w = _i32(query_word_ids)
        s = _i32(sig_ids)
        out = np.zeros(len(s), np.float32)
        self._check(self._lib.lcd_index_score(self._h, _ptr(w), len(w), _ptr(s), len(s), int(n_total), _ptr(out)))
        return out

    # -- batched localisation ------------------------------------------------------------------
    def adjust_likelihood(self, likelihood, virtual_place_ratio: int = 0) -> np.ndarray:
        """Rtabmap::adjustLikelihood of rows [n_frames, ns] (or one row): returns [n_frames, ns + 1], column 0 = virtual place."""
        l = np.ascontiguousarray(likelihood, np.float32)
        one = l.ndim == 1
        l2 = l.reshape(1, -1) if one else l
        out = np.zeros((l2.shape[0], l2.shape[1] + 1), np.float32)
        self._check(self._lib.lcd_adjust_likelihood(self._h, _ptr(l2), l2.shape[0], l2.shape[1], int(virtual_place_ratio), _ptr(out)))
        return out[0] if one else out

    def bayes_reset(self):
        self._check(self._lib.lcd_bayes_reset(self._h))

    def bayes_compute_posterior(self, ids, likelihood, col_ptr, nbr_row, nbr_level, prediction_lc, virtual_place_prior: float = 0.9) -> np.ndarray:
        """BayesFilter::computePosterior with the prediction in sparse form (see lcd_b200.h)."""
        i = _i32(ids)
        l = np.ascontiguousarray(likelihood, np.float32)
        cp = np.ascontiguousarray(col_ptr, np.int64)
        r = _i32(nbr_row)
        lv = _i32(nbr_level)
        lc = np.ascontiguousarray(prediction_lc, np.float64)
        out = np.zeros(len(i), np.float32)
        self._check(self._lib.lcd_bayes_compute_posterior(self._h, _ptr(i), _ptr(l), len(i), _ptr(cp), _ptr(r), _ptr(lv), _ptr(lc), len(lc),
                                                           float(virtual_place_prior), _ptr(out)))
        return out

    def localize_batch(self, queries, n_frames: int, sig_ids, n_total: int, incremental: bool = True, nndr: float = 0.8,
                       cmp_new: bool = True, want_words: bool = True, want_likelihood: bool = True,
                       out_words=None, out_like=None):
        q = self._desc(queries)
        assert len(q) % n_frames == 0
        nq = len(q) // n_frames
        s = _i32(sig_ids)
        words = None
        like = None
        if want_words:
            words = out_words if out_words is not None else np.zeros((n_frames, nq), np.int32)
        if want_likelihood:
            like = out_like if out_like is not None else np.zeros((n_frames, len(s)), np.float32)
        self._check(self._lib.lcd_localize_batch(self._h, _ptr(q), n_frames, nq, int(incremental), float(nndr), int(cmp_new),
                                                  _ptr(s), len(s), int(n_total), _ptr(words), _ptr(like)))
        return words, like

    def localize_batch_dev(self, d_queries: int, n_frames: int, nq: int, d_sig_ids: int, ns: int, n_total: int,
                           d_words_out: int = 0, d_like_out: int = 0, incremental: bool = True, nndr: float = 0.8,
                           cmp_new: bool = True, stream: int = 0):
        self._check(self._lib.lcd_localize_batch_dev(self._h, C.c_void_p(d_queries), n_frames, nq, int(incremental), float(nndr),
                                                      int(cmp_new), C.c_void_p(d_sig_ids), ns, int(n_total),
                                                      C.c_void_p(d_words_out or None), C.c_void_p(d_like_out or None),
                                                      C.c_void_p(stream or None)))

    # -- geometric verification -----------------------------------------------------------------
    def _pairs(self, desc_from, desc_to, n_from, n_to):
        dt = np.uint8 if self.desc_type == LCD_DESC_U8 else np.float32
        a = np.ascontiguousarray(desc_from, dtype=dt)
        b = np.ascontiguousarray(desc_to, dtype=dt)
        if a.ndim != 3 or a.shape != b.shape or a.shape[2] != self.desc_dim:
            raise LcdError(-1, f"descriptors must be [n_pairs, cap, {self.desc_dim}]")
        n_pairs, cap = a.shape[:2]
        nf = _i32(n_from if n_from is not None else np.full(n_pairs, cap))
        nt = _i32(n_to if n_to is not None else np.full(n_pairs, cap))
        return a, b, nf, nt, n_pairs, cap

    def match_pairs(self, desc_from, desc_to, n_from=None, n_to=None, nndr: float = 0.8):
        a, b, nf, nt, n_pairs, cap = self._pairs(desc_from, desc_to, n_from, n_to)
        fid = np.zeros((n_pairs, cap), np.int32)
        tid = np.zeros((n_pairs, cap), np.int32)
        self._check(self._lib.lcd_match_pairs(self._h, n_pairs, cap, _ptr(a), _ptr(nf), _ptr(b), _ptr(nt), float(nndr), _ptr(fid), _ptr(tid)))
        return fid, tid

    def verify_batch(self, desc_from, xyz_from, desc_to, uv_to, K4, n_from=None, n_to=None, nndr: float = 0.8, min_inliers: int = 20,
                     iterations: int = 300, reproj_error: float = 2.0, refine_iterations: int = 1, refine_sigma: float = 3.0, xyz_to=None,
                     var_median_ratio: int = 4, max_variance: float = 0.0, split_linear_cov: bool = False, image_size=(0, 0),
                     repeat_once: bool = False, guess_win_size: int = 40):
        """Memory::computeTransform for a batch of (FROM, TO) pairs; returns a list of dicts."""
        a, b, nf, nt, n_pairs, cap = self._pairs(desc_from, desc_to, n_from, n_to)
        xyz = np.ascontiguousarray(xyz_from, np.float32).reshape(n_pairs, cap, 3)
        uv = np.ascontiguousarray(uv_to, np.float32).reshape(n_pairs, cap, 2)
        xt = None if xyz_to is None else np.ascontiguousarray(xyz_to, np.float32).reshape(n_pairs, cap, 3)
        prm = self.verify_params(K4, nndr, min_inliers, iterations, reproj_error, refine_iterations, refine_sigma, var_median_ratio, max_variance,
                                 split_linear_cov, image_size, repeat_once, guess_win_size)
        res = (VerifyResult * n_pairs)()
        mids = np.zeros((n_pairs, cap), np.int32)
        iids = np.zeros((n_pairs, cap), np.int32)
        self._check(self._lib.lcd_verify_batch(self._h, n_pairs, cap, _ptr(a), _ptr(xyz), _ptr(nf), _ptr(b), _ptr(uv), _ptr(xt), _ptr(nt),
                                                C.byref(prm), res, _ptr(mids), _ptr(iids)))
        out = []
        for i in range(n_pairs):
            r = res[i]
            out.append({"ok": bool(r.ok), "matches": mids[i, :r.n_matches].copy(), "inliers": iids[i, :r.n_inliers].copy(),
                        "iterations_run": r.iterations_run, "rvec": np.array(r.rvec[:]), "tvec": np.array(r.tvec[:]),
                        "transform": np.array(r.transform[:], np.float32).reshape(3, 4),
                        "covariance": np.array(r.covariance[:], np.float64).reshape(6, 6)})
        return out

    def pnp_ransac(self, object_points, image_points, K4, rvec=None, tvec=None, use_guess: bool = True, iterations: int = 300,
                   reproj_error: float = 2.0, min_inliers: int = 20, flags: int = 0, refine_iterations: int = 1, refine_sigma: float = 3.0,
                   dist_coeffs=None):
        """util3d::solvePnPRansac: returns (rvec, tvec, inlier indices)."""
        X = np.ascontiguousarray(object_points, np.float32).reshape(-1, 3)
        uv = np.ascontiguousarray(image_points, np.float32).reshape(-1, 2)
        n = len(X)
        K = np.array([K4[0], 0, K4[2], 0, K4[1], K4[3], 0, 0, 1], np.float64)
        D = None if dist_coeffs is None else np.ascontiguousarray(dist_coeffs, np.float64)
        r = np.zeros(3) if rvec is None else np.array(rvec, np.float64)
        t = np.zeros(3) if tvec is None else np.array(tvec, np.float64)
        inl = np.zeros(max(n, 1), np.int32)
        n_inl = C.c_int(0)
        self._check(self._lib.lcd_pnp_ransac(self._h, _ptr(X), _ptr(uv), n, _ptr(K), _ptr(D), 0 if D is None else len(D), _ptr(r), _ptr(t),
                                              int(use_guess), int(iterations), float(reproj_error), int(min_inliers), int(flags),
                                              int(refine_iterations), float(refine_sigma), _ptr(inl), C.byref(n_inl)))
        return r, t, inl[:n_inl.value].copy()

    def pnp_ransac_batch(self, object_points, image_points, n_points, K4, iterations: int = 300, reproj_error: float = 2.0,
                         min_inliers: int = 20, refine_iterations: int = 1, refine_sigma: float = 3.0):
        X = np.ascontiguousarray(object_points, np.float32)
        uv = np.ascontiguousarray(image_points, np.float32)
        n_sets, cap = X.shape[:2]
        npts = _i32(n_points)
        K = np.array([K4[0], 0, K4[2], 0, K4[1], K4[3], 0, 0, 1], np.float64)
        r = np.zeros((n_sets, 3))
        t = np.zeros((n_sets, 3))
        inl = np.zeros((n_sets, cap), np.int32)
        n_inl = np.zeros(n_sets, np.int32)
        its = np.zeros(n_sets, np.int32)
        self._check(self._lib.lcd_pnp_ransac_batch(self._h, n_sets, cap, _ptr(X), _ptr(uv), _ptr(npts), _ptr(K), None, 0, _ptr(r), _ptr(t), 1,
                                                    int(iterations), float(reproj_error), int(min_inliers), 0, int(refine_iterations),
                                                    float(refine_sigma), _ptr(inl), _ptr(n_inl), _ptr(its)))
        return r, t, [inl[i, :n_inl[i]].copy() for i in range(n_sets)], its

    def match_bf(self, desc_query, desc_train, n_query=None, n_train=None, cross_check: bool = False):
        """cv::BFMatcher on [n_pairs, cap, dim] descriptor sets: (idx1, dist1, idx2, dist2); idx2 / dist2 are None with cross_check."""
        q, t, nq, nt, n_pairs, cap = self._pairs(desc_query, desc_train, n_query, n_train)
        i1 = np.zeros((n_pairs, cap), np.int32)
        d1 = np.zeros((n_pairs, cap), np.float32)
        i2 = None if cross_check else np.zeros((n_pairs, cap), np.int32)
        d2 = None if cross_check else np.zeros((n_pairs, cap), np.float32)
        self._check(self._lib.lcd_match_bf(self._h, n_pairs, cap, _ptr(q), _ptr(nq), _ptr(t), _ptr(nt), 1 if cross_check else 0, _ptr(i1), _ptr(d1),
                                            _ptr(i2), _ptr(d2)))
        return i1, d1, i2, d2

    # -- signature store + fused query -------------------------------------------------------------
    def sig_add_batch(self, sig_ids, desc, xyz, n=None):
        ids = _i32(sig_ids)
        dt = np.uint8 if self.desc_type == LCD_DESC_U8 else np.float32
        d = np.ascontiguousarray(desc, dtype=dt)
        assert d.ndim == 3 and d.shape[0] == len(ids) and d.shape[2] == self.desc_dim
        cap = d.shape[1]
        x = np.ascontiguousarray(xyz, np.float32).reshape(len(ids), cap, 3)
        nn = _i32(n if n is not None else np.full(len(ids), cap))
        self._check(self._lib.lcd_sig_add_batch(self._h, _ptr(ids), len(ids), cap, _ptr(d), _ptr(x), _ptr(nn)))

    def sig_remove(self, sig_id: int):
        self._check(self._lib.lcd_sig_remove(self._h, int(sig_id)))

    def sig_count(self) -> int:
        return self._lib.lcd_sig_count(self._h)

    def sig_slots(self) -> int:
        return self._lib.lcd_sig_slots(self._h)

    @property
    def orb_last_path(self) -> int:
        """bit flags of the kernels the last detection used: 1 TMA tiles, 2 shared-memory patches, 4 vectorised preparation"""
        return self._lib.lcd_orb_last_path(self._h)

    def orb_overflow(self) -> bool:
        r = self._lib.lcd_orb_overflow(self._h)
        if r < 0:
            self._check(r)
        return bool(r)

    @staticmethod
    def verify_params(K4, nndr=0.8, min_inliers=20, iterations=300, reproj_error=2.0, refine_iterations=1, refine_sigma=3.0, var_median_ratio=4,
                      max_variance=0.0, split_linear_cov=False, image_size=(0, 0), repeat_once=False, guess_win_size=40):
        return VerifyParams(nndr, min_inliers, iterations, reproj_error, refine_iterations, refine_sigma, *[float(k) for k in K4],
                            int(var_median_ratio), float(max_variance), int(bool(split_linear_cov)), int(image_size[0]), int(image_size[1]),
                            int(bool(repeat_once)), int(guess_win_size))

    @staticmethod
    def _results(res, n):
        out = []
        for i in range(n):
            r = res[i]
            out.append({"ok": bool(r.ok), "n_matches": r.n_matches, "n_inliers": r.n_inliers, "iterations_run": r.iterations_run,
                        "rvec": np.array(r.rvec[:]), "tvec": np.array(r.tvec[:]), "transform": np.array(r.transform[:], np.float32).reshape(3, 4),
                        "covariance": np.array(r.covariance[:], np.float64).reshape(6, 6)})
        return out

    def process_batch(self, queries, uv, n_frames: int, sig_ids, n_total: int, vp: "VerifyParams", incremental: bool = True, nndr: float = 0.8,
                      cmp_new: bool = True, out_words=None, out_like=None, want_words=True, want_likelihood=True):
        q = self._desc(queries)
        nq = len(q) // n_frames
        u = np.ascontiguousarray(uv, np.float32)
        s = _i32(sig_ids)
        words = (out_words if out_words is not None else np.zeros((n_frames, nq), np.int32)) if want_words else None
        like = (out_like if out_like is not None else np.zeros((n_frames, len(s)), np.float32)) if want_likelihood else None
        hyp = np.zeros(n_frames, np.int32)
        res = (VerifyResult * n_frames)()
        self._check(self._lib.lcd_process_batch(self._h, _ptr(q), _ptr(u), n_frames, nq, int(incremental), float(nndr), int(cmp_new), _ptr(s), len(s),
                                                 int(n_total), C.byref(vp), _ptr(words), _ptr(like), _ptr(hyp), res))
        return words, like, hyp, self._results(res, n_frames)

    def process_batch_dev(self, d_queries: int, d_uv: int, n_frames: int, nq: int, d_sig_ids: int, ns: int, n_total: int, vp: "VerifyParams",
                          d_words_out: int = 0, d_like_out: int = 0, incremental: bool = True, nndr: float = 0.8, cmp_new: bool = True, stream: int = 0):
        self._check(self._lib.lcd_process_batch_dev(self._h, C.c_void_p(d_queries), C.c_void_p(d_uv), n_frames, nq, int(incremental), float(nndr),
                                                     int(cmp_new), C.c_void_p(d_sig_ids), ns, int(n_total), C.byref(vp),
                                                     C.c_void_p(d_words_out or None), C.c_void_p(d_like_out or None), C.c_void_p(stream or None)))

    def process_frames(self, images, depth, op: "OrbParams", sig_ids, n_total: int, vp: "VerifyParams" = None, incremental: bool = True,
                       nndr: float = 0.8, cmp_new: bool = True, out_words=None, out_like=None):
        """The whole hot path from host images: returns (n_kp, words, likelihood, hypothesis, results)."""
        img = np.ascontiguousarray(images, np.uint8)
        n, h, w = img.shape[:3]
        ch = 1 if img.ndim == 3 else img.shape[3]
        dtype, dptr = 0, None
        if depth is not None:
            if depth.dtype == np.uint16:
                dtype, depth = 1, np.ascontiguousarray(depth)
            else:
                dtype, depth = 2, np.ascontiguousarray(depth, np.float32)
            dptr = _ptr(depth)
        s = _i32(sig_ids)
        cap = op.n_features
        words = out_words if out_words is not None else np.zeros((n, cap), np.int32)
        like = out_like if out_like is not None else np.zeros((n, len(s)), np.float32)
        nkp = np.zeros(n, np.int32)
        hyp = np.zeros(n, np.int32)
        res = (VerifyResult * n)()
        self._check(self._lib.lcd_process_frames(self._h, n, _ptr(img), w, h, ch, dptr, dtype, C.byref(op), int(incremental), float(nndr), int(cmp_new),
                                                  _ptr(s), len(s), int(n_total), C.byref(vp) if vp is not None else None, _ptr(nkp), _ptr(words),
                                                  _ptr(like), _ptr(hyp), res))
        return nkp, words, like, hyp, (self._results(res, n) if vp is not None else None)

    def process_frames_submit(self, images, depth, op: "OrbParams", sig_ids, n_total: int, vp: "VerifyParams", out_nkp, out_words, out_like,
                              out_hyp, out_res, incremental: bool = True, nndr: float = 0.8, cmp_new: bool = True):
        """Pipelined lcd_process_frames: queue one batch (all arrays must stay alive, ideally pinned, until process_frames_wait).
        images uint8 [n,h,w,(ch)], depth uint16/float32 [n,h,w] or None; out_* numpy arrays; out_res a (VerifyResult * n)() array."""
        n, h, w = images.shape[:3]
        ch = 1 if images.ndim == 3 else images.shape[3]
        dtype, dptr = 0, None
        if depth is not None:
            dtype = 1 if depth.dtype == np.uint16 else 2
            dptr = _ptr(depth)
        self._check(self._lib.lcd_process_frames_submit(self._h, n, _ptr(images), w, h, ch, dptr, dtype, C.byref(op), int(incremental), float(nndr),
                                                         int(cmp_new), _ptr(sig_ids), len(sig_ids), int(n_total),
                                                         C.byref(vp) if vp is not None else None, _ptr(out_nkp), _ptr(out_words), _ptr(out_like),
                                                         _ptr(out_hyp), out_res))

    def process_frames_wait(self):
        self._check(self._lib.lcd_process_frames_wait(self._h))

    def process_frames_dev(self, d_images: int, n_frames: int, w: int, h: int, ch: int, d_depth: int, depth_type: int, op: "OrbParams", d_sig_ids: int,
                           ns: int, n_total: int, vp: "VerifyParams", d_words_out: int = 0, d_like_out: int = 0, incremental: bool = True,
                           nndr: float = 0.8, cmp_new: bool = True, stream: int = 0):
        self._check(self._lib.lcd_process_frames_dev(self._h, n_frames, C.c_void_p(d_images), w, h, ch, C.c_void_p(d_depth or None), depth_type,
                                                      C.byref(op), int(incremental), float(nndr), int(cmp_new), C.c_void_p(d_sig_ids), ns, int(n_total),
                                                      C.byref(vp) if vp is not None else None, C.c_void_p(d_words_out or None),
                                                      C.c_void_p(d_like_out or None), C.c_void_p(stream or None)))

    def map_detect_async(self, image, depth, op: "OrbParams"):
        """Queue the upload + ORB of ONE frame (image [h,w] or [h,w,3] uint8, depth [h,w] or None); buffers must stay alive until map_frame."""
        img = np.ascontiguousarray(image, np.uint8)
        h, w = img.shape[:2]
        ch = 1 if img.ndim == 2 else img.shape[2]
        dtype, dptr = 0, None
        if depth is not None:
            if depth.dtype == np.uint16:
                dtype, depth = 1, np.ascontiguousarray(depth)
            else:
                dtype, depth = 2, np.ascontiguousarray(depth, np.float32)
            dptr = _ptr(depth)
        self._map_keep = getattr(self, "_map_keep", [])[-1:] + [(img, depth)]
        self._map_cap = op.n_features
        self._check(self._lib.lcd_map_detect_async(self._h, _ptr(img), w, h, ch, dptr, dtype, C.byref(op)))

    def map_frame(self, sig_id: int, wm_sig_ids=None, n_total: int = 0, incremental: bool = True, nndr: float = 0.8, cmp_new: bool = True,
                  want_features: bool = False):
        """Memory::update + computeLikelihood of the oldest detected frame: (n_kp, word ids [n_kp], n_new, likelihood or None[, kp, desc, xyz])."""
        cap = getattr(self, "_map_cap", 1)
        words = np.zeros(cap, np.int32)
        n_kp = C.c_int(0)
        n_new = C.c_int(0)
        s = None if wm_sig_ids is None or len(wm_sig_ids) == 0 else _i32(wm_sig_ids)
        like = None if s is None else np.zeros(len(s), np.float32)
        kp = (Keypoint * cap)() if want_features else None
        desc = np.zeros((cap, 32), np.uint8) if want_features else None
        xyz = np.zeros((cap, 3), np.float32) if want_features else None
        self._check(self._lib.lcd_map_frame(self._h, int(sig_id), int(incremental), float(nndr), int(cmp_new), _ptr(s), 0 if s is None else len(s),
                                             int(n_total), C.byref(n_kp), kp, _ptr(desc), _ptr(xyz), _ptr(words), C.byref(n_new), _ptr(like)))
        n = n_kp.value
        if want_features:
            return n, words[:n], n_new.value, like, kp, desc[:n], xyz[:n]
        return n, words[:n], n_new.value, like

    def verify_top_dev(self, d_queries: int, d_uv: int, n_frames: int, nq: int, d_like: int, d_sig_ids: int, ns: int, vp: "VerifyParams", stream: int = 0):
        self._check(self._lib.lcd_verify_top_dev(self._h, C.c_void_p(d_queries), C.c_void_p(d_uv), n_frames, nq, C.c_void_p(d_like),
                                                  C.c_void_p(d_sig_ids), ns, C.byref(vp), C.c_void_p(stream or None)))

    def process_fetch(self, n_frames: int):
        hyp = np.zeros(n_frames, np.int32)
        res = (VerifyResult * n_frames)()
        self._check(self._lib.lcd_process_fetch(self._h, n_frames, _ptr(hyp), res))
        return hyp, self._results(res, n_frames)

    def process_fetch_async(self, n_frames: int, hyp_ptr: int, res_ptr: int, stream: int = 0):
        """queue the download of the last step's hypotheses (int32[n]) and results (lcd_verify_result[n]) into pinned host memory at the given
        addresses, behind that step on `stream`; nothing is synchronised — read them after an event recorded behind this call"""
        self._check(self._lib.lcd_process_fetch_async(self._h, n_frames, C.c_void_p(hyp_ptr), C.c_void_p(res_ptr), C.c_void_p(stream)))

    @staticmethod
    def results_from_buffer(buf: np.ndarray, n_frames: int):
        """lcd_verify_result records written by process_fetch_async into a uint8 array -> the dictionaries process_fetch returns"""
        res = (VerifyResult * n_frames).from_buffer_copy(buf[: n_frames * C.sizeof(VerifyResult)].tobytes())
        return Engine._results(res, n_frames)

    # -- word-range sharding ----------------------------------------------------------------------
    @staticmethod
    def shard_unique_id() -> bytes:
        """ncclGetUniqueId through the library (rank 0); broadcast the 128 bytes to the other ranks."""
        buf = C.create_string_buffer(128)
        rc = load_library().lcd_shard_unique_id(buf)
        if rc != LCD_OK:
            raise LcdError(rc, (load_library().lcd_last_error(None) or b"").decode())
        return buf.raw

    def shard_comm_init(self, unique_id: bytes, rank: int, n_ranks: int):
        self._check(self._lib.lcd_shard_comm_init(self._h, C.create_string_buffer(unique_id, 128), int(rank), int(n_ranks)))

    def shard_comm_destroy(self):
        self._check(self._lib.lcd_shard_comm_destroy(self._h))

    def shard_process_frames_dev(self, d_images: int, n_frames: int, w: int, h: int, ch: int, d_depth: int, depth_type: int, op: "OrbParams", d_sig_ids: int,
                                 ns: int, n_total: int, d_row_ids_global: int, last_word_id: int, vp: "VerifyParams", d_words_out: int, d_like_out: int,
                                 incremental: bool = True, nndr: float = 0.8, cmp_new: bool = True, stream: int = 0):
        self._check(self._lib.lcd_shard_process_frames_dev(self._h, n_frames, C.c_void_p(d_images), w, h, ch, C.c_void_p(d_depth or None), depth_type,
                                                            C.byref(op), int(incremental), float(nndr), int(cmp_new), C.c_void_p(d_sig_ids), ns, int(n_total),
                                                            C.c_void_p(d_row_ids_global), int(last_word_id), C.byref(vp) if vp is not None else None,
                                                            C.c_void_p(d_words_out or None), C.c_void_p(d_like_out), C.c_void_p(stream or None)))

    def shard_set_row_offset(self, off: int):
        self._check(self._lib.lcd_shard_set_row_offset(self._h, int(off)))

    def shard_knn2_keys_dev(self, d_queries: int, nq: int, d_keys_out: int, stream: int = 0):
        self._check(self._lib.lcd_shard_knn2_keys_dev(self._h, C.c_void_p(d_queries), nq, C.c_void_p(d_keys_out), C.c_void_p(stream or None)))

    def shard_resolve_score_dev(self, d_queries: int, n_frames: int, nq: int, d_keys_gathered: int, n_ranks: int, d_row_ids: int,
                                total_rows: int, last_word_id: int, d_sig_ids: int, ns: int, n_total: int, d_words_out: int,
                                d_scores_out: int, incremental: bool = True, nndr: float = 0.8, cmp_new: bool = True, stream: int = 0):
        self._check(self._lib.lcd_shard_resolve_score_dev(
            self._h, C.c_void_p(d_queries), n_frames, nq, C.c_void_p(d_keys_gathered), n_ranks, C.c_void_p(d_row_ids), total_rows,
            last_word_id, int(incremental), float(nndr), int(cmp_new), C.c_void_p(d_sig_ids), ns, int(n_total),
            C.c_void_p(d_words_out or None), C.c_void_p(d_scores_out or None), C.c_void_p(stream or None)))

    def shard_resolve_frames_dev(self, d_queries_all: int, frame0: int, n_frames: int, n_frames_total: int, nq: int, d_keys_gathered: int,
                                 n_ranks: int, d_row_ids: int, last_word_id: int, d_n_per_frame: int, d_words_out: int, incremental: bool = True,
                                 nndr: float = 0.8, cmp_new: bool = True, stream: int = 0):
        self._check(self._lib.lcd_shard_resolve_frames_dev(
            self._h, C.c_void_p(d_queries_all), frame0, n_frames, n_frames_total, nq, C.c_void_p(d_keys_gathered), n_ranks, C.c_void_p(d_row_ids),
            last_word_id, int(incremental), float(nndr), int(cmp_new), C.c_void_p(d_n_per_frame or None), C.c_void_p(d_words_out),
            C.c_void_p(stream or None)))

    def shard_score_ids_dev(self, d_word_ids_all: int, n_frames: int, nq: int, d_sig_ids: int, ns: int, n_total: int, d_scores_out: int,
                            stream: int = 0):
        self._check(self._lib.lcd_shard_score_ids_dev(self._h, C.c_void_p(d_word_ids_all), n_frames, nq, C.c_void_p(d_sig_ids), ns, int(n_total),
                                                       C.c_void_p(d_scores_out), C.c_void_p(stream or None)))

    def shard_finalize_dev(self, d_scores: int, n: int, d_like_out: int, stream: int = 0):
        self._check(self._lib.lcd_shard_finalize_dev(self._h, C.c_void_p(d_scores), n, C.c_void_p(d_like_out), C.c_void_p(stream or None)))
