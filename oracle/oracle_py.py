"""ctypes binding of oracle/liboracle.so (restatement) and oracle/_ref/libref_flann.so
(the reference's own rtflann, compiled from /root/reference by oracle/Makefile).

TEST INFRASTRUCTURE ONLY: checker for tests/, smoke() and bench.py's CPU baseline.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "liboracle.so"
REF_LIB = HERE / "_ref" / "libref_flann.so"
REFERENCE_ROOT = Path("/root/reference")

_lib = None
_ref = None
_P = C.c_void_p
_I = C.c_int
_F = C.c_float


def _reference_readable() -> bool:
    """Whether the reference sources can be read: a user without access to them still builds and tests, without _ref."""
    try:
        return REFERENCE_ROOT.is_dir()
    except OSError:
        return False


def build(with_ref: bool = True) -> None:
    """Compile liboracle.so (always) and _ref/libref_flann.so (when the reference sources are readable)."""
    srcs = [HERE / "oracle.cpp", HERE / "oracle_verify.cpp", HERE / "pnp_math.h"]
    if not LIB.exists() or LIB.stat().st_mtime < max(s.stat().st_mtime for s in srcs):
        subprocess.run(["make", "-C", str(HERE), "liboracle.so"], check=True, capture_output=True)
    if with_ref and _reference_readable() and not REF_LIB.exists():
        subprocess.run(["make", "-C", str(HERE), "ref"], check=True, capture_output=True)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build(with_ref=False)
        L = C.CDLL(str(LIB))
        L.orc_create.restype = _P
        L.orc_create.argtypes = [_I, _I, _I, _F, _I]
        L.orc_destroy.argtypes = [_P]
        L.orc_set_params.argtypes = [_P, _I, _F, _I]
        L.orc_add_words.argtypes = [_P, _P, _P, _I]
        L.orc_remove_words.argtypes = [_P, _P, _I]
        L.orc_update.argtypes = [_P]
        for f in ("orc_size", "orc_indexed_size", "orc_not_indexed_size", "orc_last_word_id"):
            getattr(L, f).argtypes = [_P]
            getattr(L, f).restype = _I
        L.orc_set_last_word_id.argtypes = [_P, _I]
        L.orc_total_refs.argtypes = [_P]
        L.orc_total_refs.restype = C.c_longlong
        L.orc_get_indexed_ids.argtypes = [_P, _P, _I]
        L.orc_get_indexed_ids.restype = _I
        L.orc_knn2.argtypes = [_P, _P, _I, _P, _P, _P, _P]
        L.orc_knn2_raw.argtypes = [_I, _I, _P, _I, _P, _I, _P, _P]
        L.orc_add_new_words.argtypes = [_P, _P, _I, _I, _P]
        L.orc_add_new_words.restype = _I
        L.orc_find_nn.argtypes = [_P, _P, _I, _P]
        L.orc_add_refs.argtypes = [_P, _I, _P, _I]
        L.orc_remove_sig.argtypes = [_P, _I]
        L.orc_set_ni.argtypes = [_P, _P, _P, _I]
        L.orc_load_csr.argtypes = [_P, _P, _I, _P, _P, _P]
        L.orc_get_refs.argtypes = [_P, _I, _P, _P, _I]
        L.orc_get_refs.restype = _I
        L.orc_likelihood.argtypes = [_P, _P, _I, _P, _I, _I, _P]
        L.orc_localize.argtypes = [_P, _P, _I, _I, _P, _I, _I, _P, _P]
        L.orc_localize.restype = _I
        L.orc_localize_ro.argtypes = [_P, _P, _I, _P, _I, _I, _P, _P]
        L.orc_localize_ro.restype = _I
        L.orc_localize_ro_knn.argtypes = [_P, _P, _I, _P, _P, _P, _I, _I, _P, _P]
        L.orc_localize_ro_knn.restype = _I
        L.orc_adjust_likelihood.argtypes = [_P, _I, _I]
        _lib = L
    return _lib


def ref_lib():
    """The reference's compiled rtflann, or None when it has not been built and its sources cannot be read."""
    global _ref
    if _ref is None:
        if not REF_LIB.exists():
            if _reference_readable():
                build(with_ref=True)
            else:
                return None
        R = C.CDLL(str(REF_LIB))
        R.ref_flann_knn2_hamming.argtypes = [_P, _I, _I, _P, _I, _P, _P]
        R.ref_flann_knn2_l2.argtypes = [_P, _I, _I, _P, _I, _P, _P]
        _ref = R
    return _ref


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def ref_knn2(data: np.ndarray, queries: np.ndarray):
    """2-NN through the reference's rtflann LinearIndex: (idx[nq,2] int64, dist[nq,2] float32)."""
    R = ref_lib()
    if R is None:
        raise RuntimeError("oracle/_ref/libref_flann.so is not built")
    nq = len(queries)
    idx = np.zeros((nq, 2), np.int64)
    dist = np.zeros((nq, 2), np.float32)
    if data.dtype == np.uint8:
        data = np.ascontiguousarray(data)
        queries = np.ascontiguousarray(queries)
        R.ref_flann_knn2_hamming(_p(data), len(data), data.shape[1], _p(queries), nq, _p(idx), _p(dist))
    else:
        data = np.ascontiguousarray(data, np.float32)
        queries = np.ascontiguousarray(queries, np.float32)
        R.ref_flann_knn2_l2(_p(data), len(data), data.shape[1], _p(queries), nq, _p(idx), _p(dist))
    return idx, dist


def knn2_raw(data: np.ndarray, queries: np.ndarray):
    L = lib()
    t = 0 if data.dtype == np.uint8 else 1
    data = np.ascontiguousarray(data)
    queries = np.ascontiguousarray(queries)
    nq = len(queries)
    idx = np.zeros((nq, 2), np.int32)
    dist = np.zeros((nq, 2), np.float32)
    L.orc_knn2_raw(t, data.shape[1], _p(data), len(data), _p(queries), nq, _p(idx), _p(dist))
    return idx, dist


def adjust_likelihood(lik: np.ndarray, virtual_place_ratio: int = 0) -> np.ndarray:
    out = np.ascontiguousarray(lik, np.float32).copy()
    lib().orc_adjust_likelihood(_p(out), len(out), virtual_place_ratio)
    return out


class OracleDictionary:
    """Restated rtabmap::VWDictionary (+ Memory::computeLikelihood) on the CPU."""

    def __init__(self, desc_type: int = 0, dim: int = 32, incremental: bool = True, nndr: float = 0.8, cmp_new: bool = True):
        self.L = lib()
        self.h = self.L.orc_create(desc_type, dim, int(incremental), nndr, int(cmp_new))
        self.dt = np.uint8 if desc_type == 0 else np.float32
        self.dim = dim

    def __del__(self):
        if getattr(self, "h", None):
            self.L.orc_destroy(self.h)
            self.h = None

    def _d(self, x):
        x = np.ascontiguousarray(x, self.dt)
        assert x.ndim == 2 and x.shape[1] == self.dim
        return x

    def set_params(self, incremental, nndr, cmp_new):
        self.L.orc_set_params(self.h, int(incremental), nndr, int(cmp_new))

    def add_words(self, ids, desc):
        ids = _i32(ids)
        self.L.orc_add_words(self.h, _p(ids), _p(self._d(desc)), len(ids))

    def remove_words(self, ids):
        ids = _i32(ids)
        self.L.orc_remove_words(self.h, _p(ids), len(ids))

    def update(self):
        self.L.orc_update(self.h)

    def size(self):
        return self.L.orc_size(self.h)

    def indexed_size(self):
        return self.L.orc_indexed_size(self.h)

    def not_indexed_size(self):
        return self.L.orc_not_indexed_size(self.h)

    @property
    def last_word_id(self):
        return self.L.orc_last_word_id(self.h)

    @last_word_id.setter
    def last_word_id(self, v):
        self.L.orc_set_last_word_id(self.h, int(v))

    def indexed_ids(self):
        n = self.indexed_size()
        ids = np.zeros(n, np.int32)
        self.L.orc_get_indexed_ids(self.h, _p(ids), n)
        return ids

    def knn2(self, q):
        q = self._d(q)
        n = len(q)
        id1 = np.zeros(n, np.int32)
        id2 = np.zeros(n, np.int32)
        d1 = np.zeros(n, np.float32)
        d2 = np.zeros(n, np.float32)
        self.L.orc_knn2(self.h, _p(q), n, _p(id1), _p(d1), _p(id2), _p(d2))
        return id1, d1, id2, d2

    def add_new_words(self, desc, sig_id):
        desc = self._d(desc)
        out = np.zeros(len(desc), np.int32)
        n = self.L.orc_add_new_words(self.h, _p(desc), len(desc), int(sig_id), _p(out))
        return out[:n]

    def find_nn(self, desc):
        desc = self._d(desc)
        out = np.zeros(len(desc), np.int32)
        self.L.orc_find_nn(self.h, _p(desc), len(desc), _p(out))
        return out

    def add_refs(self, sig_id, word_ids):
        w = _i32(word_ids)
        self.L.orc_add_refs(self.h, int(sig_id), _p(w), len(w))

    def remove_sig(self, sig_id):
        self.L.orc_remove_sig(self.h, int(sig_id))

    def set_ni(self, sig_ids, ni):
        s, n = _i32(sig_ids), _i32(ni)
        self.L.orc_set_ni(self.h, _p(s), _p(n), len(s))

    def load_csr(self, word_ids, row_ptr, sig, cnt):
        w = _i32(word_ids)
        rp = np.ascontiguousarray(row_ptr, np.int64)
        s, c = _i32(sig), _i32(cnt)
        self.L.orc_load_csr(self.h, _p(w), len(w), _p(rp), _p(s), _p(c))

    def get_refs(self, word_id, cap=1 << 16):
        s = np.zeros(cap, np.int32)
        c = np.zeros(cap, np.int32)
        n = self.L.orc_get_refs(self.h, int(word_id), _p(s), _p(c), cap)
        return s[:n], c[:n]

    def total_refs(self):
        return int(self.L.orc_total_refs(self.h))

    def likelihood(self, qwords, sig_ids, n_total):
        w, s = _i32(qwords), _i32(sig_ids)
        out = np.zeros(len(s), np.float32)
        self.L.orc_likelihood(self.h, _p(w), len(w), _p(s), len(s), int(n_total), _p(out))
        return out

    def localize(self, desc, sig_id, sig_ids, n_total, want_like=True):
        desc = self._d(desc)
        s = _i32(sig_ids)
        words = np.zeros(len(desc), np.int32)
        like = np.zeros(len(s), np.float32) if want_like else None
        n = self.L.orc_localize(self.h, _p(desc), len(desc), int(sig_id), _p(s), len(s), int(n_total), _p(words), _p(like))
        return words[:n], like

    def localize_ro(self, desc, sig_ids, n_total, want_like=True):
        """Thread-safe read-only variant of localize() (ctypes releases the GIL during the call)."""
        desc = self._d(desc)
        s = _i32(sig_ids)
        words = np.zeros(len(desc), np.int32)
        like = np.zeros(len(s), np.float32) if want_like else None
        n = self.L.orc_localize_ro(self.h, _p(desc), len(desc), _p(s), len(s), int(n_total), _p(words), _p(like))
        return words[:n], like

    def localize_ro_knn(self, desc, knn_idx, knn_dist, sig_ids, n_total, want_like=True):
        """localize_ro with the index search done by the caller (bench.py: the reference's own compiled rtflann, ref_knn2)."""
        desc = self._d(desc)
        s = _i32(sig_ids)
        ki = np.ascontiguousarray(knn_idx, np.int64)
        kd = np.ascontiguousarray(knn_dist, np.float32)
        words = np.zeros(len(desc), np.int32)
        like = np.zeros(len(s), np.float32) if want_like else None
        n = self.L.orc_localize_ro_knn(self.h, _p(desc), len(desc), _p(ki), _p(kd), _p(s), len(s), int(n_total), _p(words), _p(like))
        return words[:n], like


# ---------------------------------------------------------------- verification stage (oracle_verify.cpp)
def _vlib():
    L = lib()
    if not getattr(L, "_verify_ready", False):
        L.orcv_solve_pnp_epnp.argtypes = [_P, _P, _I, _P, _P, _P]
        L.orcv_solve_pnp_epnp.restype = _I
        L.orcv_solve_pnp_iterative.argtypes = [_P, _P, _I, _P, _P, _P]
        L.orcv_project.argtypes = [_P, _I, _P, _P, _P, _P]
        L.orcv_rodrigues.argtypes = [_P, _P]
        L.orcv_sym_eigen.argtypes = [_P, _I, _I, _P, _P]
        L.orcv_rodrigues_inv.argtypes = [_P, _P]
        L.orcv_rng_draws.argtypes = [_I, _I, _P]
        L.orcv_pnp_ransac.argtypes = [_P, _P, _I, _P, _I, _F, _I, _I, _F, _P, _P, _P, _P, _P, _P]
        L.orcv_pnp_ransac.restype = _I
        L.orcv_match_pair.argtypes = [_I, _I, _P, _I, _P, _I, _F, _P, _P]
        L.orcv_verify_pair.argtypes = [_I, _I, _P, _P, _I, _P, _P, _I, _P, _F, _I, _I, _F, _I, _P, _P, _P, _P, _P, _P, _P]
        L.orcv_verify_pair.restype = _I
        L.orcv_verify_pair_cov.argtypes = [_I, _I, _P, _P, _I, _P, _P, _P, _I, _P, _F, _I, _I, _F, _I, _I, _I, _I, _F, _I, _P, _P, _P, _P, _P, _P,
                                           _P, _P]
        L.orcv_verify_pair_cov.restype = _I
        L.orcv_verify_pair_repeat.argtypes = [_I, _I, _P, _P, _I, _P, _P, _P, _I, _P, _F, _I, _I, _F, _I, _I, _I, _I, _F, _I, _I, _F, _P, _P, _P, _P, _P,
                                              _P, _P, _P, _P]
        L.orcv_verify_pair_repeat.restype = _I
        L.orcv_guess_match.argtypes = [_I, _I, _P, _P, _I, _P, _P, _I, _P, _P, _P, _I, _I, _F, _F, _P]
        L.orcv_guess_match.restype = _I
        L._verify_ready = True
    return L


def sym_eigen(a, method=0):
    """Eigenvalues (descending) and eigenvectors (rows) of a symmetric matrix; method 0 = Householder+QL, 1 = Jacobi."""
    a = np.ascontiguousarray(a, np.float64)
    n = a.shape[0]
    w = np.zeros(n)
    vt = np.zeros((n, n))
    _vlib().orcv_sym_eigen(_p(a), n, method, _p(w), _p(vt))
    return w, vt


def solve_pnp_epnp(X, uv, K4):
    L = _vlib()
    X = np.ascontiguousarray(X, np.float32)
    uv = np.ascontiguousarray(uv, np.float32)
    K4 = np.ascontiguousarray(K4, np.float64)
    r = np.zeros(3)
    t = np.zeros(3)
    ok = L.orcv_solve_pnp_epnp(_p(X), _p(uv), len(X), _p(K4), _p(r), _p(t))
    return bool(ok), r, t


def solve_pnp_iterative(X, uv, K4, rvec0, tvec0):
    L = _vlib()
    X = np.ascontiguousarray(X, np.float32)
    uv = np.ascontiguousarray(uv, np.float32)
    K4 = np.ascontiguousarray(K4, np.float64)
    r = np.array(rvec0, np.float64).copy()
    t = np.array(tvec0, np.float64).copy()
    L.orcv_solve_pnp_iterative(_p(X), _p(uv), len(X), _p(K4), _p(r), _p(t))
    return r, t


def pnp_ransac(X, uv, K4, iterations=300, reproj=2.0, min_inliers=20, refine_iterations=1, refine_sigma=3.0, guess=None):
    """util3d::solvePnPRansac (cv3::solvePnPRansac + refinement): ok, rvec, tvec, inlier indices, iterations run."""
    L = _vlib()
    X = np.ascontiguousarray(X, np.float32)
    uv = np.ascontiguousarray(uv, np.float32)
    K4 = np.ascontiguousarray(K4, np.float64)
    r = np.zeros(3)
    t = np.zeros(3)
    inl = np.zeros(len(X), np.int32)
    n_inl = C.c_int(0)
    it = C.c_int(0)
    g = None if guess is None else np.ascontiguousarray(guess, np.float64)
    ok = L.orcv_pnp_ransac(_p(X), _p(uv), len(X), _p(K4), iterations, reproj, min_inliers, refine_iterations, refine_sigma,
                           _p(g), _p(r), _p(t), _p(inl), C.byref(n_inl), C.byref(it))
    return bool(ok), r, t, inl[:n_inl.value].copy(), it.value


def match_pair(desc_from, desc_to, nndr=0.8):
    """RegistrationVis global matching through a temporary dictionary: (from word ids, to word ids)."""
    L = _vlib()
    t = 0 if desc_from.dtype == np.uint8 else 1
    a = np.ascontiguousarray(desc_from)
    b = np.ascontiguousarray(desc_to)
    fi = np.zeros(max(len(a), 1), np.int32)
    ti = np.zeros(max(len(b), 1), np.int32)
    L.orcv_match_pair(t, a.shape[1], _p(a), len(a), _p(b), len(b), nndr, _p(fi), _p(ti))
    return fi[:len(a)], ti[:len(b)]


def verify_pair(desc_from, xyz_from, desc_to, uv_to, K4, nndr=0.8, min_inliers=20, iterations=300, reproj=2.0, refine_iterations=1):
    """Memory::computeTransform for one pair (global matching + PnP RANSAC).  Returns a dict."""
    L = _vlib()
    t = 0 if desc_from.dtype == np.uint8 else 1
    a = np.ascontiguousarray(desc_from)
    b = np.ascontiguousarray(desc_to)
    xa = np.ascontiguousarray(xyz_from, np.float32)
    ub = np.ascontiguousarray(uv_to, np.float32)
    K4 = np.ascontiguousarray(K4, np.float64)
    cap = max(len(a), len(b), 1)
    mids = np.zeros(cap, np.int32)
    iids = np.zeros(cap, np.int32)
    nm = C.c_int(0)
    ni = C.c_int(0)
    r = np.zeros(3)
    tv = np.zeros(3)
    T = np.zeros(12, np.float32)
    ok = L.orcv_verify_pair(t, a.shape[1], _p(a), _p(xa), len(a), _p(b), _p(ub), len(b), _p(K4), nndr, min_inliers, iterations, reproj,
                            refine_iterations, _p(mids), C.byref(nm), _p(iids), C.byref(ni), _p(r), _p(tv), _p(T))
    return {"ok": bool(ok), "matches": mids[:nm.value].copy(), "inliers": iids[:ni.value].copy(), "rvec": r, "tvec": tv,
            "transform": T.reshape(3, 4)}


def verify_pair_cov(desc_from, xyz_from, desc_to, uv_to, K4, xyz_to=None, nndr=0.8, min_inliers=20, iterations=300, reproj=2.0, refine_iterations=1,
                    image_size=(0, 0), var_median_ratio=4, max_variance=0.0, split_linear_cov=False):
    """verify_pair plus RegistrationInfo::covariance (util3d_motion_estimation.cpp:156-266)."""
    L = _vlib()
    t = 0 if desc_from.dtype == np.uint8 else 1
    a = np.ascontiguousarray(desc_from)
    b = np.ascontiguousarray(desc_to)
    xa = np.ascontiguousarray(xyz_from, np.float32)
    ub = np.ascontiguousarray(uv_to, np.float32)
    xb = None if xyz_to is None else np.ascontiguousarray(xyz_to, np.float32)
    K4 = np.ascontiguousarray(K4, np.float64)
    cap = max(len(a), len(b), 1)
    mids = np.zeros(cap, np.int32)
    iids = np.zeros(cap, np.int32)
    nm = C.c_int(0)
    ni = C.c_int(0)
    r = np.zeros(3)
    tv = np.zeros(3)
    T = np.zeros(12, np.float32)
    cov = np.zeros(36)
    ok = L.orcv_verify_pair_cov(t, a.shape[1], _p(a), _p(xa), len(a), _p(b), _p(ub), _p(xb), len(b), _p(K4), nndr, int(min_inliers),
                                int(iterations), reproj, int(refine_iterations), int(image_size[0]), int(image_size[1]), int(var_median_ratio),
                                max_variance, int(bool(split_linear_cov)), _p(mids), C.byref(nm), _p(iids), C.byref(ni), _p(r), _p(tv), _p(T),
                                _p(cov))
    return {"ok": bool(ok), "matches": mids[:nm.value].copy(), "inliers": iids[:ni.value].copy(), "rvec": r, "tvec": tv,
            "transform": T.reshape(3, 4), "covariance": cov.reshape(6, 6)}


def verify_pair_repeat(desc_from, xyz_from, desc_to, uv_to, K4, xyz_to=None, nndr=0.8, min_inliers=20, iterations=300, reproj=2.0, refine_iterations=1,
                       image_size=(640, 480), var_median_ratio=4, max_variance=0.0, split_linear_cov=False, repeat_once=True, guess_win_size=40):
    """Memory::computeTransform as Registration::computeTransformationMod runs it by default: global matching pass, then (Reg/RepeatOnce) the
    pass with the first result as the guess.  Returns the dict of verify_pair_cov plus "second_pass" (bool)."""
    L = _vlib()
    t = 0 if desc_from.dtype == np.uint8 else 1
    a = np.ascontiguousarray(desc_from)
    b = np.ascontiguousarray(desc_to)
    xa = np.ascontiguousarray(xyz_from, np.float32)
    ub = np.ascontiguousarray(uv_to, np.float32)
    xb = None if xyz_to is None else np.ascontiguousarray(xyz_to, np.float32)
    K4 = np.ascontiguousarray(K4, np.float64)
    cap = max(len(a), len(b), 1)
    mids = np.zeros(cap, np.int32)
    iids = np.zeros(cap, np.int32)
    nm = C.c_int(0)
    ni = C.c_int(0)
    sp = C.c_int(0)
    r = np.zeros(3)
    tv = np.zeros(3)
    T = np.zeros(12, np.float32)
    cov = np.zeros(36)
    ok = L.orcv_verify_pair_repeat(t, a.shape[1], _p(a), _p(xa), len(a), _p(b), _p(ub), _p(xb), len(b), _p(K4), nndr, int(min_inliers), int(iterations),
                                   reproj, int(refine_iterations), int(image_size[0]), int(image_size[1]), int(var_median_ratio), max_variance,
                                   int(bool(split_linear_cov)), int(bool(repeat_once)), float(guess_win_size), _p(mids), C.byref(nm), _p(iids),
                                   C.byref(ni), _p(r), _p(tv), _p(T), _p(cov), C.byref(sp))
    return {"ok": bool(ok), "matches": mids[:nm.value].copy(), "inliers": iids[:ni.value].copy(), "rvec": r, "tvec": tv, "transform": T.reshape(3, 4),
            "covariance": cov.reshape(6, 6), "second_pass": bool(sp.value)}
