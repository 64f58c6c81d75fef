"""ctypes binding of libvsom_b200.so (include/vsom_b200.h).  Product code: never imports oracle/."""
from __future__ import annotations

import ctypes as C
import os
import re

import numpy as np

from . import build as _build

STANDARD, MEDIAN, CLR = 0, 1, 2
EXPONENTIAL, INVERSE_PROPORTIONAL = 0, 1
ORDER_REFERENCE, ORDER_LANES, ORDER_EIGEN_SSE = 0, 1, 2
CLUSTER_UNIFORM, CLUSTER_HITS = 0, 1

_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)
_i32p = C.POINTER(C.c_int32)
_vp = C.c_void_p

_PROTOS = {
    "vsom_create": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "vsom_destroy": (None, [_vp]),
    "vsom_create_sharded": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "vsom_peer_export": (C.c_int, [_vp, C.c_char_p]),
    "vsom_peer_import": (C.c_int, [_vp, C.c_int, C.c_char_p]),
    "vsom_peer_export_planes": (C.c_int, [_vp, C.c_char_p]),
    "vsom_peer_import_planes": (C.c_int, [_vp, C.c_int, C.c_char_p]),
    "vsom_peer_attach": (C.c_int, [_vp, C.c_int, _vp]),
    "vsom_shard_rows": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vsom_last_error": (C.c_char_p, [_vp]),
    "vsom_model_length": (C.c_int, [C.c_int, C.c_int]),
    "vsom_depth": (C.c_int, [_vp]),
    "vsom_node_count": (C.c_int, [_vp]),
    "vsom_stream": (_vp, [_vp]),
    "vsom_synchronize": (C.c_int, [_vp]),
    "vsom_launch_count": (C.c_uint64, [_vp]),
    "vsom_planes_resident": (C.c_int, [_vp]),
    "vsom_debug_profile": (C.c_int, [_vp, C.c_int]),
    "vsom_debug_last_train_fast": (C.c_int, [_vp]),
    "vsom_debug_phase_cycles_raw": (C.c_int, [_vp, _f64p]),
    "vsom_debug_die_aware": (C.c_int, [_vp]),
    "vsom_debug_measure_peaks": (C.c_int, [_vp, _f64p]),
    "vsom_debug_phase_cycles": (C.c_int, [_vp, _f64p]),
    "vsom_upload_state": (C.c_int, [_vp, _f32p, _f32p, _f32p, _f32p, _u64p]),
    "vsom_download_state": (C.c_int, [_vp, _f32p, _f32p, _f32p, _f32p, _u64p]),
    "vsom_get_node": (C.c_int, [_vp, C.c_size_t, _f32p, _f32p]),
    "vsom_linear_init": (C.c_int, [_vp, _f32p, C.c_size_t, _f64p, _f64p, _f64p]),
    "vsom_debug_linear_init_phases": (C.c_int, [_vp, _f64p]),
    "vsom_debug_cluster_phases": (C.c_int, [_vp, _f64p]),
    "vsom_cluster_nodes": (C.c_int, [_vp, C.c_int, C.c_uint64, C.c_int, C.c_int, _i32p, _f64p, _f64p, _f64p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vsom_train_chunk": (C.c_int, [_vp, _f32p, C.c_size_t, C.c_double, C.c_double, C.c_int, _u64p, _u32p, _f32p, _f32p]),
    "vsom_train_chunk_device": (C.c_int, [_vp, _vp, C.c_size_t, C.c_double, C.c_double, C.c_int, _vp, _vp]),
    "vsom_batch_epoch": (C.c_int, [_vp, _f32p, C.c_size_t, C.c_double, C.c_int, _u64p, _f32p]),
    "vsom_find_bmu": (C.c_int, [_vp, _f32p, C.c_size_t, C.c_uint64, _u32p, _f32p]),
    "vsom_find_bmu_device": (C.c_int, [_vp, _vp, C.c_size_t, C.c_uint64, _vp, _vp]),
    "vsom_find_bmu_exact": (C.c_int, [_vp, _f32p, C.c_size_t, C.c_uint64, _u32p, _f32p]),
    "vsom_find_bmu_exact_device": (C.c_int, [_vp, _vp, C.c_size_t, C.c_uint64, _vp, _vp]),
    "vsom_debug_last_score_tc": (C.c_int, [_vp]),
    "vsom_debug_last_score_pair": (C.c_int, [_vp]),
    "vsom_debug_tc_stats": (C.c_int, [_vp, _u64p]),
    "vsom_find_bmu_batch": (C.c_int, [_vp, _f32p, C.c_size_t, C.c_uint64, _u32p, _f32p, _u64p]),
    "vsom_find_bmu_batch_device": (C.c_int, [_vp, _vp, C.c_size_t, C.c_uint64, _vp, _vp, _u64p]),
    "vsom_find_bmu2": (C.c_int, [_vp, _f32p, C.c_size_t, C.c_uint64, _u32p, _f32p, _u32p, _f32p, _u64p]),
    "vsom_find_bmu2_device": (C.c_int, [_vp, _vp, C.c_size_t, C.c_uint64, _vp, _vp, _vp, _vp, _u64p]),
    "vsom_find_bmu2_exact": (C.c_int, [_vp, _f32p, C.c_size_t, C.c_uint64, _u32p, _f32p, _u32p, _f32p]),
    "vsom_evaluate": (C.c_int, [_vp, _f32p, C.c_size_t, _f64p]),
    "vsom_measure_similarity": (C.c_int, [_vp, _f32p, C.c_size_t, C.c_uint64, C.c_int, _u32p, _f32p]),
    "vsom_soft_assign": (C.c_int, [_vp, _f32p, C.c_size_t, C.c_uint64, _f64p]),
    "vsom_all_dists": (C.c_int, [_vp, _f32p, _f64p]),
    "vsom_update_umatrix": (C.c_int, [_vp, _f64p]),
    "vsom_build_index_device": (C.c_int, [_vp, _vp, C.c_size_t, _vp, _vp, _vp]),
    "vsom_build_index": (C.c_int, [_vp, _u32p, C.c_size_t, _u64p, _u64p, _u32p]),
}

_lib = None


class VsomError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"vsom_b200 error {code}: {msg}")
        self.code = code


def lib_path() -> str:
    return _build.LIB


def header_symbols():
    """Every function include/vsom_b200.h declares."""
    hdr = os.path.join(_build.REPO, "include", "vsom_b200.h")
    return sorted(set(re.findall(r"VSOM_API[^;(]*?\b(vsom_\w+)\s*\(", open(hdr).read())))


def lib():
    """Load libvsom_b200.so (building it first when the sources are newer).  Fails loudly when it cannot."""
    global _lib
    if _lib is None:
        path = _build.build()
        L = C.CDLL(path)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def exported_symbols():
    L = lib()
    return [s for s in header_symbols() if hasattr(L, s)]


def model_length(d_in: int, transform: int) -> int:
    return int(lib().vsom_model_length(d_in, transform))


def _p(a, t):
    return C.cast(None, t) if a is None else a.ctypes.data_as(t)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


class VsomContext:
    """One map on one B200.  Method names follow the C-ABI; arrays are numpy (host entry points) or anything
    with a ``data_ptr()`` (torch CUDA tensors; ``*_device`` entry points)."""

    def __init__(self, width, height, d_in, transform=STANDARD, order=ORDER_REFERENCE, device=0, rank=0, world=1):
        L = lib()
        h = _vp()
        if world > 1:
            rc = L.vsom_create_sharded(C.byref(h), device, width, height, d_in, transform, order, rank, world)
        else:
            rc = L.vsom_create(C.byref(h), device, width, height, d_in, transform, order)
        if rc != 0:
            raise VsomError(rc, (L.vsom_last_error(None) or b"").decode())
        self._h = h
        self.W, self.H, self.N, self.Din = width, height, width * height, d_in
        self.transform, self.order, self.device = transform, order, device
        self.rank, self.world = rank, world
        self.Dm = L.vsom_depth(h)

    def close(self):
        if getattr(self, "_h", None):
            lib().vsom_destroy(self._h)
            self._h = None

    __del__ = close

    def _check(self, rc):
        if rc != 0:
            raise VsomError(rc, (lib().vsom_last_error(self._h) or b"").decode())

    # ---- state
    def upload_state(self, mean=None, S=None, sigma=None, weight=None, hits=None):
        mean = None if mean is None else _f32(mean)
        S = None if S is None else _f32(S)
        sigma = None if sigma is None else _f32(sigma)
        weight = None if weight is None else _f32(weight)
        hits = None if hits is None else np.ascontiguousarray(hits, dtype=np.uint64)
        for a in (mean, S, sigma):
            if a is not None and a.size != self.N * self.Dm:
                raise ValueError("plane must be N x Dm")
        self._check(lib().vsom_upload_state(self._h, _p(mean, _f32p), _p(S, _f32p), _p(sigma, _f32p), _p(weight, _f32p), _p(hits, _u64p)))

    def download_state(self):
        mean = np.empty((self.N, self.Dm), np.float32)
        S = np.empty_like(mean)
        sigma = np.empty_like(mean)
        weight = np.empty(self.N, np.float32)
        hits = np.empty(self.N, np.uint64)
        self._check(lib().vsom_download_state(self._h, _p(mean, _f32p), _p(S, _f32p), _p(sigma, _f32p), _p(weight, _f32p), _p(hits, _u64p)))
        return dict(mean=mean, S=S, sigma=sigma, weight=weight, hits=hits)

    def download_state_zero_filled(self):
        """Sharded contexts: full-size arrays with this rank's band filled in and zeros elsewhere."""
        mean = np.zeros((self.N, self.Dm), np.float32)
        S = np.zeros_like(mean)
        sigma = np.zeros_like(mean)
        weight = np.zeros(self.N, np.float32)
        hits = np.zeros(self.N, np.uint64)
        self._check(lib().vsom_download_state(self._h, _p(mean, _f32p), _p(S, _f32p), _p(sigma, _f32p), _p(weight, _f32p), _p(hits, _u64p)))
        return dict(mean=mean, S=S, sigma=sigma, weight=weight, hits=hits)

    def get_node(self, node):
        """Som::getNeuron / Som::getSigmaNeuron: (mean, sigma) rows of one node, Dm floats each."""
        mean = np.empty(self.Dm, np.float32)
        sigma = np.empty(self.Dm, np.float32)
        self._check(lib().vsom_get_node(self._h, node, _p(mean, _f32p), _p(sigma, _f32p)))
        return mean, sigma

    def linear_init(self, x):
        """Linear initialisation along the rows' two principal components (vsom_linear_init): sets the mean plane, zeroes S, sigma,
        weight and hits; returns (mean[Din], lambda[2], axes[2, Din]) in f64."""
        x = _f32(x).reshape(-1, self.Din)
        mean = np.empty(self.Din, np.float64)
        lam = np.empty(2, np.float64)
        axes = np.empty((2, self.Din), np.float64)
        self._check(lib().vsom_linear_init(self._h, _p(x, _f32p), x.shape[0], _p(mean, _f64p), _p(lam, _f64p), _p(axes, _f64p)))
        return mean, lam, axes

    def linear_init_host_ptr(self, x_ptr: int, n: int):
        """vsom_linear_init on raw HOST rows (e.g. a pinned torch tensor); no outputs."""
        self._check(lib().vsom_linear_init(self._h, C.cast(x_ptr, _f32p), n, None, None, None))

    def linear_init_phases(self):
        """Host wall time (ms) of the last linear_init: co-moment pass (with the row copies), eigen step, fill; and its iterations."""
        out = np.zeros(4, np.float64)
        self._check(lib().vsom_debug_linear_init_phases(self._h, _p(out, _f64p)))
        return {"pass_ms": out[0], "eigen_ms": out[1], "fill_ms": out[2], "iterations": int(out[3])}

    def cluster_nodes(self, k, seed=0, weighting=CLUSTER_UNIFORM, max_iter=300):
        """k-means over the map's nodes (vsom_cluster_nodes): k-means++ seeding from `seed`, then Lloyd iterations over the mean plane,
        each node weighted by 1 (CLUSTER_UNIFORM) or its hit count (CLUSTER_HITS).  Returns (labels[N] int32, centroids[k, Dm] f64,
        weight[k] f64, inertia, iterations, converged)."""
        labels = np.empty(self.N, np.int32)
        centroids = np.empty((k, self.Dm), np.float64)
        weight = np.empty(k, np.float64)
        inertia, iterations, converged = C.c_double(0), C.c_int(0), C.c_int(0)
        self._check(lib().vsom_cluster_nodes(self._h, int(k), int(seed), int(weighting), int(max_iter), _p(labels, _i32p), _p(centroids, _f64p),
                                             _p(weight, _f64p), C.byref(inertia), C.byref(iterations), C.byref(converged)))
        return labels, centroids, weight, inertia.value, iterations.value, bool(converged.value)

    def cluster_phases(self):
        """Device time (ms) of the last cluster_nodes call's phases: seeding, all assignments, all updates, the outputs; and its number
        of assignments (updates: one fewer)."""
        out = np.zeros(5, np.float64)
        self._check(lib().vsom_debug_cluster_phases(self._h, _p(out, _f64p)))
        return {"seeding_ms": out[0], "assign_ms": out[1], "update_ms": out[2], "outputs_ms": out[3], "assignments": int(out[4])}

    # ---- online training
    def train_chunk(self, x, eta, sigma, decay=EXPONENTIAL, last_bmu=None):
        x = _f32(x).reshape(-1, self.Din)
        n = x.shape[0]
        bmu = np.empty(n, np.uint32)
        dist = np.empty(n, np.float32)
        resid2 = np.empty(n, np.float32)
        last = np.zeros(n, np.uint64) if last_bmu is None else np.ascontiguousarray(last_bmu, dtype=np.uint64)
        self._check(lib().vsom_train_chunk(self._h, _p(x, _f32p), n, eta, sigma, decay, _p(last, _u64p), _p(bmu, _u32p), _p(dist, _f32p),
                                           _p(resid2, _f32p)))
        return bmu, dist, resid2, last

    def train_chunk_device(self, x_dev, n, eta, sigma, decay=EXPONENTIAL, out_bmu_dev=None, out_dist_dev=None):
        self._check(lib().vsom_train_chunk_device(self._h, x_dev.data_ptr(), n, eta, sigma, decay,
                                                  out_bmu_dev.data_ptr() if out_bmu_dev is not None else None,
                                                  out_dist_dev.data_ptr() if out_dist_dev is not None else None))

    def batch_epoch(self, x, sigma, is_first, last_bmu=None):
        """One chunk-epoch of the batch-map trainer; returns (mse, last_bmu)."""
        x = _f32(x).reshape(-1, self.Din)
        n = x.shape[0]
        last = np.zeros(n, np.uint64) if last_bmu is None else np.ascontiguousarray(last_bmu, dtype=np.uint64).copy()
        mse = C.c_float(0)
        self._check(lib().vsom_batch_epoch(self._h, _p(x, _f32p), n, sigma, int(bool(is_first)), _p(last, _u64p), C.byref(mse)))
        return float(np.float32(mse.value)), last

    # ---- scoring
    def find_bmu(self, x, min_hits=0):
        x = _f32(x).reshape(-1, self.Din)
        n = x.shape[0]
        bmu = np.empty(n, np.uint32)
        dist = np.empty(n, np.float32)
        self._check(lib().vsom_find_bmu(self._h, _p(x, _f32p), n, min_hits, _p(bmu, _u32p), _p(dist, _f32p)))
        return bmu, dist

    def find_bmu_device(self, x_dev, n, out_bmu_dev=None, out_dist_dev=None, min_hits=0):
        self._check(lib().vsom_find_bmu_device(self._h, x_dev.data_ptr(), n, min_hits,
                                               out_bmu_dev.data_ptr() if out_bmu_dev is not None else None,
                                               out_dist_dev.data_ptr() if out_dist_dev is not None else None))

    def find_bmu_exact(self, x, min_hits=0):
        """Always the exact scan (K3), whatever the batch size."""
        x = _f32(x).reshape(-1, self.Din)
        n = x.shape[0]
        bmu = np.empty(n, np.uint32)
        dist = np.empty(n, np.float32)
        self._check(lib().vsom_find_bmu_exact(self._h, _p(x, _f32p), n, min_hits, _p(bmu, _u32p), _p(dist, _f32p)))
        return bmu, dist

    def find_bmu_exact_device(self, x_dev, n, out_bmu_dev=None, out_dist_dev=None, min_hits=0):
        self._check(lib().vsom_find_bmu_exact_device(self._h, x_dev.data_ptr(), n, min_hits,
                                                     out_bmu_dev.data_ptr() if out_bmu_dev is not None else None,
                                                     out_dist_dev.data_ptr() if out_dist_dev is not None else None))

    def find_bmu_host_ptr(self, x_ptr: int, n: int, bmu_ptr: int, dist_ptr: int, min_hits=0):
        """vsom_find_bmu on raw HOST addresses (e.g. pinned torch tensors): no numpy conversion in the way."""
        self._check(lib().vsom_find_bmu(self._h, C.cast(x_ptr, _f32p), n, min_hits, C.cast(bmu_ptr, _u32p), C.cast(dist_ptr, _f32p)))

    @property
    def last_score_tc(self) -> int:
        """0 when the last scoring call ran the exact scan, else the precision tier (1 or 2) of K2 (tcgen05 candidate search +
        exact rescore)."""
        return int(lib().vsom_debug_last_score_tc(self._h))

    @property
    def last_score_pair(self) -> int:
        """1 when the last K2 search ran as CTA pairs (cta_group::2), 0 for the single-CTA kernel."""
        return int(lib().vsom_debug_last_score_pair(self._h))

    def tc_stats(self):
        out = np.zeros(3, np.uint64)
        self._check(lib().vsom_debug_tc_stats(self._h, _p(out, _u64p)))
        return {"list_overflow": int(out[0]), "nan_or_none": int(out[1]), "certificate": int(out[2])}

    def find_bmu_batch(self, x, min_hits=0):
        """Tensor-core candidate search + exact rescore; returns (bmu, dist, rows that took the exact full scan)."""
        x = _f32(x).reshape(-1, self.Din)
        n = x.shape[0]
        bmu = np.empty(n, np.uint32)
        dist = np.empty(n, np.float32)
        fb = C.c_uint64(0)
        self._check(lib().vsom_find_bmu_batch(self._h, _p(x, _f32p), n, min_hits, _p(bmu, _u32p), _p(dist, _f32p), C.byref(fb)))
        return bmu, dist, int(fb.value)

    def find_bmu_batch_device(self, x_dev, n, out_bmu_dev=None, out_dist_dev=None, min_hits=0):
        fb = C.c_uint64(0)
        self._check(lib().vsom_find_bmu_batch_device(self._h, x_dev.data_ptr(), n, min_hits,
                                                     out_bmu_dev.data_ptr() if out_bmu_dev is not None else None,
                                                     out_dist_dev.data_ptr() if out_dist_dev is not None else None, C.byref(fb)))
        return int(fb.value)

    def find_bmu2(self, x, min_hits=0):
        """Best and second-best matching node of every row: (bmu, dist, bmu2, dist2, rows that took the exact full scan).
        bmu2 is 0xFFFFFFFF and dist2 NaN where a row has no runner-up."""
        x = _f32(x).reshape(-1, self.Din)
        n = x.shape[0]
        bmu, bmu2 = np.empty(n, np.uint32), np.empty(n, np.uint32)
        dist, dist2 = np.empty(n, np.float32), np.empty(n, np.float32)
        fb = C.c_uint64(0)
        self._check(lib().vsom_find_bmu2(self._h, _p(x, _f32p), n, min_hits, _p(bmu, _u32p), _p(dist, _f32p), _p(bmu2, _u32p), _p(dist2, _f32p),
                                         C.byref(fb)))
        return bmu, dist, bmu2, dist2, int(fb.value)

    def find_bmu2_device(self, x_dev, n, out_bmu_dev=None, out_dist_dev=None, out_bmu2_dev=None, out_dist2_dev=None, min_hits=0):
        """vsom_find_bmu2 on device arrays; returns the rows that took the exact full scan."""
        fb = C.c_uint64(0)
        ptr = lambda t: t.data_ptr() if t is not None else None
        self._check(lib().vsom_find_bmu2_device(self._h, x_dev.data_ptr(), n, min_hits, ptr(out_bmu_dev), ptr(out_dist_dev), ptr(out_bmu2_dev),
                                                ptr(out_dist2_dev), C.byref(fb)))
        return int(fb.value)

    def find_bmu2_exact(self, x, min_hits=0):
        """find_bmu2 through the exact scan (K3) whatever the batch size: (bmu, dist, bmu2, dist2)."""
        x = _f32(x).reshape(-1, self.Din)
        n = x.shape[0]
        bmu, bmu2 = np.empty(n, np.uint32), np.empty(n, np.uint32)
        dist, dist2 = np.empty(n, np.float32), np.empty(n, np.float32)
        self._check(lib().vsom_find_bmu2_exact(self._h, _p(x, _f32p), n, min_hits, _p(bmu, _u32p), _p(dist, _f32p), _p(bmu2, _u32p), _p(dist2, _f32p)))
        return bmu, dist, bmu2, dist2

    def measure_similarity(self, x, number_of_sigmas, min_hits=0):
        """Per-row pass of Som::measureSimilarity: (restricted BMU, largest normalised deviation from it) for every row."""
        x = _f32(x).reshape(-1, self.Din)
        n = x.shape[0]
        bmu = np.empty(n, np.uint32)
        row_max = np.empty(n, np.float32)
        self._check(lib().vsom_measure_similarity(self._h, _p(x, _f32p), n, min_hits, int(number_of_sigmas), _p(bmu, _u32p), _p(row_max, _f32p)))
        return bmu, row_max

    def measure_similarity_host_ptr(self, x_ptr: int, n: int, number_of_sigmas: int, bmu_ptr: int, row_max_ptr: int, min_hits=0):
        """vsom_measure_similarity on raw HOST addresses (e.g. pinned torch tensors)."""
        self._check(lib().vsom_measure_similarity(self._h, C.cast(x_ptr, _f32p), n, min_hits, int(number_of_sigmas), C.cast(bmu_ptr, _u32p), C.cast(row_max_ptr, _f32p)))

    def evaluate(self, x):
        x = _f32(x).reshape(-1, self.Din)
        out = C.c_double(0)
        self._check(lib().vsom_evaluate(self._h, _p(x, _f32p), x.shape[0], C.byref(out)))
        return out.value

    def soft_assign(self, x, min_hits=0):
        """Som::findRestrictedBmd per row: (n, N) probabilities."""
        x = _f32(x).reshape(-1, self.Din)
        out = np.empty((x.shape[0], self.N), np.float64)
        self._check(lib().vsom_soft_assign(self._h, _p(x, _f32p), x.shape[0], min_hits, _p(out, _f64p)))
        return out

    def all_dists(self, v):
        v = _f32(v).reshape(self.Din)
        out = np.empty(self.N, np.float64)
        self._check(lib().vsom_all_dists(self._h, _p(v, _f32p), _p(out, _f64p)))
        return out

    # ---- U-matrix / index
    def update_umatrix(self):
        out = np.zeros(self.N, np.float64)  # a sharded context fills in its own grid rows only
        self._check(lib().vsom_update_umatrix(self._h, _p(out, _f64p)))
        return out

    def build_index(self, bmu):
        bmu = np.ascontiguousarray(bmu, dtype=np.uint32)
        n = bmu.shape[0]
        counts = np.empty(self.N, np.uint64)
        offsets = np.empty(self.N + 1, np.uint64)
        rows = np.empty(n, np.uint32)
        self._check(lib().vsom_build_index(self._h, _p(bmu, _u32p), n, _p(counts, _u64p), _p(offsets, _u64p), _p(rows, _u32p)))
        return counts, offsets, rows

    def build_index_device(self, bmu_dev, n, counts_dev, offsets_dev, row_ids_dev):
        self._check(lib().vsom_build_index_device(self._h, bmu_dev.data_ptr(), n, counts_dev.data_ptr(), offsets_dev.data_ptr(),
                                                  row_ids_dev.data_ptr() if row_ids_dev is not None else None))

    # ---- node sharding across GPUs
    def peer_export(self) -> bytes:
        """Both IPC handles of this rank (exchange slots + mean plane), 128 bytes, for an all-gather by the caller."""
        a, b = C.create_string_buffer(64), C.create_string_buffer(64)
        self._check(lib().vsom_peer_export(self._h, a))
        self._check(lib().vsom_peer_export_planes(self._h, b))
        return a.raw + b.raw

    def peer_import(self, rank: int, handle: bytes):
        self._check(lib().vsom_peer_import(self._h, rank, handle[:64]))
        self._check(lib().vsom_peer_import_planes(self._h, rank, handle[64:128]))

    def peer_attach(self, rank: int, peer: "VsomContext"):
        """Ranks living in the same process attach each other directly (no IPC handles)."""
        self._check(lib().vsom_peer_attach(self._h, rank, peer._h))

    def shard_rows(self):
        """(rows per block, global grid row of every local row)."""
        blk, cnt = C.c_int(0), C.c_int(0)
        self._check(lib().vsom_shard_rows(self._h, C.byref(blk), C.byref(cnt), None))
        rows = (C.c_int * max(cnt.value, 1))()
        self._check(lib().vsom_shard_rows(self._h, C.byref(blk), C.byref(cnt), rows))
        return blk.value, np.array(rows[: cnt.value], dtype=np.int64)

    # ---- diagnostics
    def debug_profile(self, enable=True):
        self._check(lib().vsom_debug_profile(self._h, int(enable)))

    def debug_phase_cycles(self):
        out = np.zeros(5, np.float64)
        self._check(lib().vsom_debug_phase_cycles(self._h, _p(out, _f64p)))
        return dict(zip(("wait_sample", "scan_min", "exchange", "broadcast", "update"), out.tolist()))

    def debug_phase_cycles_raw(self):
        out = np.zeros(8, np.float64)
        self._check(lib().vsom_debug_phase_cycles_raw(self._h, _p(out, _f64p)))
        if self.last_train_fast:
            names = ("chain", "cta_min", "exchange", "coefficients", "barrier1", "update", "barrier2")
        else:
            names = ("wait_sample", "scan_min", "exchange", "broadcast", "update")
        return dict(zip(names, out.tolist()))

    def measure_peaks(self):
        """Measured on-chip read bandwidths of this device (GB/s): shared memory (all SMs / per SM) and L2."""
        out = np.zeros(4, np.float64)
        self._check(lib().vsom_debug_measure_peaks(self._h, _p(out, _f64p)))
        return {"smem_gbs": out[0], "smem_gbs_per_sm": out[1], "l2_gbs": out[2], "l2_set_mib": out[3]}

    @property
    def die_aware(self) -> bool:
        return bool(lib().vsom_debug_die_aware(self._h))

    @property
    def last_train_fast(self) -> bool:
        """True when the last train_chunk ran K1F (online_step_fast.cu) rather than the generic online-step kernel."""
        return bool(lib().vsom_debug_last_train_fast(self._h))

    # ---- plumbing
    def synchronize(self):
        self._check(lib().vsom_synchronize(self._h))

    @property
    def stream(self) -> int:
        return int(lib().vsom_stream(self._h) or 0)

    @property
    def launch_count(self) -> int:
        return int(lib().vsom_launch_count(self._h))

    @property
    def planes_resident(self) -> bool:
        return bool(lib().vsom_planes_resident(self._h))
