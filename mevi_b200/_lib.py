"""ctypes binding of libmevi_b200.so (include/mevi_b200.h).

PyTorch is used only for device memory and streams: tensors are handed to the
library as raw pointers + extents + the current cudaStream_t.  Nothing here
computes; if the shared library is missing the import of any compute path fails
loudly (no fallback).
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Dict, Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libmevi_b200.so"

METRIC_L2, METRIC_IP = 0, 1
MODE_AUTO, MODE_EXACT, MODE_TENSOR = 0, 1, 2
_MODES = {"auto": MODE_AUTO, "exact": MODE_EXACT, "tensor": MODE_TENSOR}
_METRICS = {"l2": METRIC_L2, "ip": METRIC_IP}
_MULTICLUS_AGGR = {"add": 0, "max": 1}  # MEVI_MULTICLUS_ADD / _MAX

# every symbol include/mevi_b200.h declares: (restype, argtypes)
_vp, _i, _i64, _f, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double
SYMBOLS = {
    "mevi_abi_version": (_i, []),
    "mevi_ctx_create": (_i, [_i, C.POINTER(_vp)]),
    "mevi_ctx_destroy": (None, [_vp]),
    "mevi_last_error": (C.c_char_p, [_vp]),
    "mevi_device_info": (_i, [_vp, C.POINTER(_i64)]),
    "mevi_ctx_check": (_i, [_vp, _vp]),
    "mevi_rq_encode": (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "mevi_rq_encode_host": (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _i, _i, _vp, _i64, _vp]),
    "mevi_kmeans_step": (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _vp, _i64, _vp, _vp, _vp]),
    "mevi_kmeans_step_fused": (_i, [_vp, _vp, _i64, _i, _vp, _i, _vp, _i64, _vp, _i64, _vp, _vp, _vp]),
    "mevi_kmeans_step_delta": (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "mevi_kmeans_update": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "mevi_residual_update": (_i, [_vp, _vp, _i64, _i, _vp, _i, _vp, _i64, _vp]),
    "mevi_accumulate_by_code": (_i, [_vp, _vp, _i64, _i, _vp, _i64, _i, _vp, _vp]),
    "mevi_pq_encode": (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _i, _vp, _vp]),
    "mevi_rq_beam_search": (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "mevi_build_inverted_lists": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp]),
    "mevi_leaf_lookup": (_i, [_vp, _vp, _i64, _i, _i, _vp, _i64, _vp, _vp]),
    "mevi_occurrence_table": (_i, [_vp, _vp, _i64, _vp, _i64, _i, _vp, C.POINTER(C.c_int32), _vp]),
    "mevi_cluster_rerank": (_i, [_vp, _vp, _i, _vp, _i64, _i, _i, _vp, _i64, _vp, _vp, _i, _i, _i64, _vp, _vp, _vp, _vp]),
    "mevi_cluster_rerank_multiclus": (_i, [_vp, _vp, _i, _vp, _i64, _i, _vp, _i64, _vp, _vp, _i, _vp, _i, _i, _i, _i64, _vp, _vp,
                                           _vp, _vp]),
    "mevi_cluster_rerank_prefix": (_i, [_vp, _vp, _i, _vp, _i64, _i, _vp, _i64, _vp, _vp, _i, _i, _i64, _vp, _vp, _vp, _vp]),
    "mevi_cluster_rerank_all": (_i, [_vp, _vp, _i, _vp, _i64, _i, _vp, _i64, _vp, _vp, _i, _i64, _vp, _vp, _vp, _vp, _vp]),
    "mevi_cluster_rerank_all_grouped": (_i, [_vp, _vp, _i, _vp, _i64, _i, _vp, _i64, _vp, _vp, _i, _i64, _vp, _vp, _vp, _vp,
                                             _vp]),
    "mevi_sort_candidates": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mevi_rerank_grouped_image": (_i, [_vp, _vp, _i64, _i, _vp, _i64, _vp, C.POINTER(_f), C.POINTER(_f), _vp]),
    "mevi_rerank_grouped_begin": (_i, [_vp, _vp, _i, _i, _f, _f, _vp, _vp]),
    "mevi_rerank_grouped_round": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _i, _i, _vp]),
    "mevi_rerank_grouped_plan": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i64, C.POINTER(C.c_int32), _i, _i, _i, _i, _i, _i, _vp, _vp,
                                      C.POINTER(_i64), _vp]),
    "mevi_rerank_grouped_plan_fill": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "mevi_rerank_grouped_thresholds": (_i, [_vp, _i, _i, _vp, _i, _vp]),
    "mevi_rerank_grouped_finish": (_i, [_vp, _vp, _i, _vp, _i, _i, _vp, _vp, _vp, C.POINTER(_i), _vp]),
    "mevi_rerank_grouped_multiclus": (_i, [_vp, _i, _i, _vp, _i, _vp, _i64, _vp, _i, _vp, _i, _vp, _vp, _vp]),
    "mevi_rerank_grouped_finish_multiclus": (_i, [_vp, _vp, _i, _vp, _i, _i, _vp, _i64, _vp, _vp, _vp, C.POINTER(_i), _vp]),
    "mevi_gather_rows": (_i, [_vp, _vp, _i64, _i, _vp, _i64, _vp, _vp]),
    "mevi_flat_ip_topk": (_i, [_vp, _vp, _i, _vp, _i64, _i, _i, _i64, _i, _vp, _vp, _vp]),
    "mevi_flat_index_create": (_i, [_vp, _vp, _i64, _i, C.POINTER(_vp), _vp]),
    "mevi_flat_index_search": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i, _vp, _vp, _vp]),
    "mevi_flat_index_destroy": (None, [_vp, _vp]),
    "mevi_topk_merge": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "mevi_merge_sorted_runs": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "mevi_dense_scores": (_i, [_vp, _vp, _i, _vp, _i64, _i, _vp, _vp]),
    "mevi_ensemble_cluster_ranks": (_i, [_vp, _vp, _vp, _i, _i, _vp, _i64, _i, _vp, _i, _vp, _vp, _vp]),
    "mevi_ensemble_fuse": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _d, _d, _d, _i, _vp, _vp, _vp, _vp]),
    "mevi_ensemble_positions": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "mevi_ensemble_first_hit": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _i64, _vp, _vp, _vp]),
}


class MeviError(RuntimeError):
    pass


def library_path() -> str:
    return os.environ.get("MEVI_B200_LIB", os.path.join(_HERE, _LIB_NAME))


_lib = None
_lib_lock = threading.Lock()


def load_library():
    """Load libmevi_b200.so and bind every declared symbol.  Raises MeviError if
    the library has not been built (`python -c 'import __graft_entry__ as g; g.build()'`
    or `make -C mevi_b200/csrc`)."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if not os.path.isfile(path):
            raise MeviError(
                f"{path} not found: the CUDA extension is not built. Run `make -C mevi_b200/csrc` "
                "(needs nvcc; cross-compiles for sm_100a). There is no CPU fallback."
            )
        lib = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        if lib.mevi_abi_version() != 1:
            raise MeviError(f"ABI version mismatch: library reports {lib.mevi_abi_version()}, binding expects 1")
        _lib = lib
        return lib


def _ptr(t) -> Optional[int]:
    if t is None:
        return None
    return t.data_ptr()


class Context:
    """One library context per CUDA device (owns scratch memory)."""

    def __init__(self, device: int):
        import torch

        if not torch.cuda.is_available():
            raise MeviError("no CUDA device visible: mevi_b200 has no CPU path")
        self.lib = load_library()
        self.device = int(device)
        h = _vp()
        rc = self.lib.mevi_ctx_create(self.device, C.byref(h))
        if rc != 0 or not h.value:
            raise MeviError(f"mevi_ctx_create(device={device}) failed with {rc}")
        self.handle = h
        info = (C.c_int64 * 8)()
        self._check(self.lib.mevi_device_info(self.handle, info))
        self.sm_count, self.cc = int(info[0]), (int(info[1]), int(info[2]))
        self.total_mem, self.tensor_path, self.l2_bytes = int(info[3]), bool(info[4]), int(info[5])

    @property
    def launches(self) -> int:
        """Kernels this context has launched so far (mevi_device_info info[6])."""
        info = (C.c_int64 * 8)()
        self._check(self.lib.mevi_device_info(self.handle, info))
        return int(info[6])

    def check(self):
        """Synchronise the current stream and raise MeviError if a kernel of an earlier asynchronous call reported a
        pipeline time-out (mevi_ctx_check)."""
        with self._device_guard():
            self._check(self.lib.mevi_ctx_check(self.handle, self._stream()))

    def _device_guard(self):
        import torch

        return torch.cuda.device(self.device)

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            self.lib.mevi_ctx_destroy(self.handle)
            self.handle = _vp()

    def _check(self, rc: int):
        if rc != 0:
            msg = self.lib.mevi_last_error(self.handle)
            raise MeviError(f"libmevi_b200 error {rc}: {msg.decode() if msg else '?'}")

    def _stream(self) -> int:
        import torch

        return torch.cuda.current_stream(self.device).cuda_stream

    # ---- helpers ----------------------------------------------------------
    def _dev(self, t, dtype, name):
        import torch

        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.device.index != self.device:
            raise MeviError(f"{name} must be a CUDA tensor on device {self.device}")
        if t.dtype != dtype:
            raise MeviError(f"{name} must have dtype {dtype}, got {t.dtype}")
        if not t.is_contiguous():
            raise MeviError(f"{name} must be contiguous")
        return t

    # ---- RQ encode --------------------------------------------------------
    def rq_encode(self, X, codebook, metric="l2", mode="auto", codes=None, residual=None, return_stats=False):
        """X [n,d] fp32 cuda, codebook [M,K,d] fp32 cuda -> codes [n,M] int32 cuda."""
        import torch

        X = self._dev(X, torch.float32, "X")
        cb = self._dev(codebook, torch.float32, "codebook")
        n, d = X.shape
        M, K, d2 = cb.shape
        if d2 != d:
            raise MeviError(f"codebook width {d2} != embedding width {d}")
        if codes is None:
            codes = torch.empty((n, M), dtype=torch.int32, device=X.device)
        else:
            self._dev(codes, torch.int32, "codes")
        if residual is not None:
            self._dev(residual, torch.float32, "residual")
        stats = torch.zeros(8, dtype=torch.int64, device=X.device) if return_stats else None
        with torch.cuda.device(self.device):
            self._check(
                self.lib.mevi_rq_encode(self.handle, _ptr(X), n, d, _ptr(cb), M, K, _METRICS[metric], _MODES[mode],
                                        _ptr(codes), _ptr(residual), _ptr(stats), self._stream())
            )
        return (codes, stats) if return_stats else codes

    def rq_encode_host(self, X_host, codebook_host, codes_host, metric="l2", mode="auto", chunk_rows=0):
        """numpy fp32 [n,d] (any host memory, pinned is faster) -> numpy int32 [n,M], streamed through the GPU."""
        import numpy as np

        assert X_host.dtype == np.float32 and X_host.flags.c_contiguous
        assert codebook_host.dtype == np.float32 and codebook_host.flags.c_contiguous
        assert codes_host.dtype == np.int32 and codes_host.flags.c_contiguous
        n, d = X_host.shape
        M, K, _ = codebook_host.shape
        stats = np.zeros(8, dtype=np.int64)
        self._check(
            self.lib.mevi_rq_encode_host(self.handle, X_host.ctypes.data, n, d, codebook_host.ctypes.data, M, K,
                                         _METRICS[metric], _MODES[mode], codes_host.ctypes.data, int(chunk_rows),
                                         stats.ctypes.data)
        )
        return stats

    def rq_encode_host_ptr(self, x_ptr, n, d, cb_ptr, M, K, codes_ptr, metric="l2", mode="auto", chunk_rows=0, stats_ptr=None):
        self._check(
            self.lib.mevi_rq_encode_host(self.handle, x_ptr, n, d, cb_ptr, M, K, _METRICS[metric], _MODES[mode],
                                         codes_ptr, int(chunk_rows), stats_ptr)
        )

    # ---- k-means ----------------------------------------------------------
    def kmeans_step(self, R, centroids, sums_counts, assign=None, assign_stride=1, inertia=None, mode="auto"):
        import torch

        R = self._dev(R, torch.float32, "R")
        c = self._dev(centroids, torch.float32, "centroids")
        self._dev(sums_counts, torch.float32, "sums_counts")
        n, d = R.shape
        K = c.shape[0]
        assert sums_counts.numel() == K * d + K
        if assign is not None:
            assert assign.dtype == torch.int32 and assign.is_cuda
        if inertia is not None:
            assert inertia.dtype == torch.float64 and inertia.is_cuda
        with torch.cuda.device(self.device):
            self._check(
                self.lib.mevi_kmeans_step(self.handle, _ptr(R), n, d, _ptr(c), K, _MODES[mode], _ptr(assign),
                                          int(assign_stride), _ptr(sums_counts), _ptr(inertia), self._stream())
            )

    def kmeans_step_fused(self, R, centroids, prev_assign, assign, sums_counts_prev, prev_stride=1, assign_stride=1, inertia=None):
        """One pass: `assign` = nearest centroid now, `sums_counts_prev` = per-centroid sums|counts of the rows under
        `prev_assign` (mevi_kmeans_step_fused).  Raises MeviError (MEVI_ERR_UNSUPPORTED) for shapes it does not take."""
        import torch

        R = self._dev(R, torch.float32, "R")
        c = self._dev(centroids, torch.float32, "centroids")
        self._dev(sums_counts_prev, torch.float32, "sums_counts_prev")
        n, d = R.shape
        K = c.shape[0]
        assert sums_counts_prev.numel() == K * d + K
        assert prev_assign.dtype == torch.int32 and prev_assign.is_cuda and assign.dtype == torch.int32 and assign.is_cuda
        assert prev_assign.data_ptr() != assign.data_ptr()
        if inertia is not None:
            assert inertia.dtype == torch.float64 and inertia.is_cuda
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_kmeans_step_fused(self.handle, _ptr(R), n, d, _ptr(c), K, _ptr(prev_assign), int(prev_stride),
                                                        _ptr(assign), int(assign_stride), _ptr(sums_counts_prev), _ptr(inertia),
                                                        self._stream()))

    def kmeans_step_delta(self, R, centroids, prev_assign, assign, master, sums_counts, prev_stride=1, assign_stride=1,
                          n_changed=None, inertia=None, mode="auto"):
        """One pass: `assign` = nearest centroid now; `master` (float64 [K*d+K], sums|counts under `prev_assign` on entry)
        is corrected by the rows whose assignment changed and describes `assign` on return; `sums_counts` = its fp32
        rounding (mevi_kmeans_step_delta).  Raises MeviError (MEVI_ERR_UNSUPPORTED) for shapes it does not take."""
        import torch

        R = self._dev(R, torch.float32, "R")
        c = self._dev(centroids, torch.float32, "centroids")
        self._dev(sums_counts, torch.float32, "sums_counts")
        self._dev(master, torch.float64, "master")
        n, d = R.shape
        K = c.shape[0]
        assert sums_counts.numel() == K * d + K and master.numel() == K * d + K
        assert prev_assign.dtype == torch.int32 and prev_assign.is_cuda and assign.dtype == torch.int32 and assign.is_cuda
        assert prev_assign.data_ptr() != assign.data_ptr()
        if inertia is not None:
            assert inertia.dtype == torch.float64 and inertia.is_cuda
        if n_changed is not None:
            assert n_changed.dtype == torch.int32 and n_changed.is_cuda
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_kmeans_step_delta(self.handle, _ptr(R), n, d, _ptr(c), K, _MODES[mode], _ptr(prev_assign),
                                                        int(prev_stride), _ptr(assign), int(assign_stride), _ptr(master),
                                                        _ptr(sums_counts), _ptr(n_changed), _ptr(inertia), self._stream()))

    def kmeans_update(self, sums_counts, centroids, n_empty=None):
        import torch

        K, d = centroids.shape
        with torch.cuda.device(self.device):
            self._check(
                self.lib.mevi_kmeans_update(self.handle, _ptr(sums_counts), K, d, _ptr(centroids), _ptr(n_empty),
                                            self._stream())
            )

    def residual_update(self, R, centroids, assign, assign_stride=1):
        import torch

        n, d = R.shape
        K = centroids.shape[0]
        with torch.cuda.device(self.device):
            self._check(
                self.lib.mevi_residual_update(self.handle, _ptr(R), n, d, _ptr(centroids), K, _ptr(assign),
                                              int(assign_stride), self._stream())
            )

    def accumulate_by_code(self, X, assign, K, sums_counts=None, assign_stride=1):
        """Per-centroid sums|counts [K*d+K] of the rows of X under a given assignment (int32, strided)."""
        import torch

        X = self._dev(X, torch.float32, "X")
        n, d = X.shape
        assert assign.dtype == torch.int32 and assign.is_cuda
        if sums_counts is None:
            sums_counts = torch.empty(K * d + K, dtype=torch.float32, device=X.device)
        else:
            self._dev(sums_counts, torch.float32, "sums_counts")
            assert sums_counts.numel() == K * d + K
        with torch.cuda.device(self.device):
            self._check(
                self.lib.mevi_accumulate_by_code(self.handle, _ptr(X), n, d, _ptr(assign), int(assign_stride), int(K),
                                                 _ptr(sums_counts), self._stream())
            )
        return sums_counts

    # ---- product quantiser / beam search -------------------------------------
    def pq_encode(self, X, codebook, metric="l2", codes=None):
        """X [n,d] fp32 cuda, codebook [M,K,d/M] fp32 cuda -> codes [n,M] int32 cuda (pq.py:249-279)."""
        import torch

        X = self._dev(X, torch.float32, "X")
        cb = self._dev(codebook, torch.float32, "codebook")
        n, d = X.shape
        M, K, dsub = cb.shape
        if dsub * M != d:
            raise MeviError(f"codebook [{M},{K},{dsub}] does not tile embedding width {d}")
        if codes is None:
            codes = torch.empty((n, M), dtype=torch.int32, device=X.device)
        else:
            self._dev(codes, torch.int32, "codes")
        with torch.cuda.device(self.device):
            self._check(
                self.lib.mevi_pq_encode(self.handle, _ptr(X), n, d, _ptr(cb), M, K, _METRICS[metric], _ptr(codes),
                                        self._stream())
            )
        return codes

    def rq_beam_search(self, X, codebook, num_beams, metric="l2", prod=True):
        """X [bs,d], codebook [M,K,d] -> (labels int32 [bs,num_beams,M], scores fp32 [bs,num_beams]) (pq.py:613-713)."""
        import torch

        X = self._dev(X, torch.float32, "X")
        cb = self._dev(codebook, torch.float32, "codebook")
        bs, d = X.shape
        M, K, d2 = cb.shape
        if d2 != d:
            raise MeviError(f"codebook width {d2} != embedding width {d}")
        labels = torch.empty((bs, num_beams, M), dtype=torch.int32, device=X.device)
        scores = torch.empty((bs, num_beams), dtype=torch.float32, device=X.device)
        with torch.cuda.device(self.device):
            self._check(
                self.lib.mevi_rq_beam_search(self.handle, _ptr(X), bs, d, _ptr(cb), M, K, _METRICS[metric],
                                             int(num_beams), 1 if prod else 0, _ptr(labels), _ptr(scores),
                                             self._stream())
            )
        return labels, scores

    # ---- inverted lists / re-rank ------------------------------------------
    def build_inverted_lists(self, codes, K):
        import torch

        codes = self._dev(codes, torch.int32, "codes")
        n, M = codes.shape
        docids = torch.empty(n, dtype=torch.int32, device=codes.device)
        keys = torch.empty(n, dtype=torch.int64, device=codes.device)
        with torch.cuda.device(self.device):
            self._check(
                self.lib.mevi_build_inverted_lists(self.handle, _ptr(codes), n, M, int(K), _ptr(docids), _ptr(keys),
                                                   self._stream())
            )
        return docids, keys

    def gather_rows(self, D, rows, out=None):
        """out[i] = D[rows[i]] (rows int32 on the device); `out`: a preallocated [>= len(rows), d] fp32 buffer to fill."""
        import torch

        D = self._dev(D, torch.float32, "D")
        rows = self._dev(rows, torch.int32, "rows")
        if out is None:
            out = torch.empty((rows.numel(), D.shape[1]), dtype=torch.float32, device=D.device)
        else:
            assert out.shape[0] >= rows.numel() and out.shape[1] == D.shape[1]
            out = self._dev(out, torch.float32, "out")[: rows.numel()]
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_gather_rows(self.handle, _ptr(D), D.shape[0], D.shape[1], _ptr(rows), rows.numel(),
                                                  _ptr(out), self._stream()))
        return out

    def cluster_rerank(self, Q, D, leaf_offsets, leaf_docids, query_leaves, k, id_base=0, leaf_ordered=False):
        """`leaf_ordered=True`: D is the CSR-ordered copy (`gather_rows(D, leaf_docids)`) — the fast path."""
        import torch

        Q = self._dev(Q, torch.float32, "Q")
        D = self._dev(D, torch.float32, "D")
        lo = self._dev(leaf_offsets, torch.int64, "leaf_offsets")
        ld = self._dev(leaf_docids, torch.int32, "leaf_docids")
        ql = self._dev(query_leaves, torch.int32, "query_leaves")
        nq, d = Q.shape
        n = D.shape[0]
        L = ql.shape[1]
        scores = torch.empty((nq, k), dtype=torch.float32, device=Q.device)
        ids = torch.empty((nq, k), dtype=torch.int64, device=Q.device)
        ncand = torch.empty((nq,), dtype=torch.int32, device=Q.device)
        with torch.cuda.device(self.device):
            self._check(
                self.lib.mevi_cluster_rerank(self.handle, _ptr(Q), nq, _ptr(D), n, d, 1 if leaf_ordered else 0, _ptr(lo),
                                             lo.numel() - 1, _ptr(ld),
                                             _ptr(ql), L, int(k), int(id_base), _ptr(scores), _ptr(ids), _ptr(ncand),
                                             self._stream())
            )
        return scores, ids, ncand

    def occurrence_table(self, leaf_offsets, leaf_docids):
        """Inverted lists that may list a document under several leaves -> (occ int32 [n, C-1], C): row p holds the CSR
        leaf indices of the other positions of the document at CSR position p, -1 padded (-2 - leaf for an earlier
        position in the same leaf); C = the largest number of
        positions of any document (1 for an empty or single-cluster index)."""
        import torch

        lo = self._dev(leaf_offsets, torch.int64, "leaf_offsets")
        ld = self._dev(leaf_docids, torch.int32, "leaf_docids")
        n = ld.numel()
        c = C.c_int32(0)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_occurrence_table(self.handle, _ptr(lo), lo.numel() - 1, _ptr(ld), n, 0, None, C.byref(c),
                                                       self._stream()))
            n_occ = max(int(c.value), 1)
            # 16 B of slack: mevi_cluster_rerank_multiclus copies the table in 16-byte aligned pieces
            occ = torch.empty(n * (n_occ - 1) + 4, dtype=torch.int32, device=ld.device)[: n * (n_occ - 1)].view(n, n_occ - 1)
            if n_occ > 1:
                self._check(self.lib.mevi_occurrence_table(self.handle, _ptr(lo), lo.numel() - 1, _ptr(ld), n, n_occ - 1,
                                                           _ptr(occ), C.byref(c), self._stream()))
        return occ, n_occ

    def cluster_rerank_multiclus(self, Q, D_leaf, leaf_offsets, leaf_docids, occ, n_occ, query_leaves, k, aggr, id_base=0):
        """Top-k of a multi-cluster index (`--doc_multiclus > 1`): one entry per document, its score aggregated over the
        query's leaves that list it (aggr 'add' / 'max'); occ, n_occ from occurrence_table."""
        import torch

        Q = self._dev(Q, torch.float32, "Q")
        D = self._dev(D_leaf, torch.float32, "D_leaf")
        lo = self._dev(leaf_offsets, torch.int64, "leaf_offsets")
        ld = self._dev(leaf_docids, torch.int32, "leaf_docids")
        ql = self._dev(query_leaves, torch.int32, "query_leaves")
        occ = self._dev(occ, torch.int32, "occ")
        nq, d = Q.shape
        scores = torch.empty((nq, k), dtype=torch.float32, device=Q.device)
        ids = torch.empty((nq, k), dtype=torch.int64, device=Q.device)
        ncand = torch.empty((nq,), dtype=torch.int32, device=Q.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_cluster_rerank_multiclus(
                self.handle, _ptr(Q), nq, _ptr(D), D.shape[0], d, _ptr(lo), lo.numel() - 1, _ptr(ld),
                _ptr(occ) if occ.numel() else None, int(n_occ), _ptr(ql), ql.shape[1], int(k), _MULTICLUS_AGGR[aggr],
                int(id_base), _ptr(scores), _ptr(ids), _ptr(ncand), self._stream()))
        return scores, ids, ncand

    def cluster_rerank_all(self, Q, D_leaf, leaf_offsets, leaf_docids, query_leaves, id_base=0, grouped=False):
        """Scores of ALL candidates of every query, in the reference's concatenation order (unsorted):
        -> (offsets int64 [nq+1], scores fp32 [total], ids int64 [total], n_candidates int32 [nq]).
        grouped=True: mevi_cluster_rerank_all_grouped (every leaf read once for all the queries that chose it), the same
        arrays byte for byte."""
        import torch

        Q = self._dev(Q, torch.float32, "Q")
        D = self._dev(D_leaf, torch.float32, "D_leaf")
        lo = self._dev(leaf_offsets, torch.int64, "leaf_offsets")
        ld = self._dev(leaf_docids, torch.int32, "leaf_docids")
        ql = self._dev(query_leaves, torch.int32, "query_leaves")
        nq, d = Q.shape
        sizes = lo[1:] - lo[:-1]
        cnt = torch.where(ql >= 0, sizes[ql.clamp(min=0).long()], torch.zeros((), dtype=torch.int64, device=Q.device)).sum(1)
        offsets = torch.zeros(nq + 1, dtype=torch.int64, device=Q.device)
        torch.cumsum(cnt, 0, out=offsets[1:])
        total = int(offsets[-1].item())
        scores = torch.empty(total, dtype=torch.float32, device=Q.device)
        ids = torch.empty(total, dtype=torch.int64, device=Q.device)
        ncand = cnt.clamp(max=0x7FFFFFFF).to(torch.int32)
        if total == 0:  # no query has a candidate (all its leaves are empty): nothing to score
            return offsets, scores, ids, ncand
        with torch.cuda.device(self.device):
            fn = self.lib.mevi_cluster_rerank_all_grouped if grouped else self.lib.mevi_cluster_rerank_all
            self._check(fn(self.handle, _ptr(Q), nq, _ptr(D), D.shape[0], d, _ptr(lo), lo.numel() - 1, _ptr(ld), _ptr(ql), ql.shape[1],
                           int(id_base), _ptr(offsets), _ptr(scores), _ptr(ids), _ptr(ncand), self._stream()))
        return offsets, scores, ids, ncand

    def cluster_rerank_all_grouped(self, Q, D_leaf, leaf_offsets, leaf_docids, query_leaves, id_base=0):
        """cluster_rerank_all through mevi_cluster_rerank_all_grouped: the same four tensors, bit for bit."""
        return self.cluster_rerank_all(Q, D_leaf, leaf_offsets, leaf_docids, query_leaves, id_base=id_base, grouped=True)

    def sort_candidates(self, offsets, scores, ids, out=None):
        """Every query's segment [offsets[q], offsets[q+1]) sorted by (score desc, id asc), -0.0 == +0.0, NaN first, score
        bits kept: the order of three stable torch.argsort passes.  ids must lie in [0, 2^32).  -> (scores, ids); with
        out=(scores_out, ids_out) the result goes there (it may be (scores, ids) themselves: sorted in place)."""
        import torch

        oo = self._dev(offsets, torch.int64, "offsets")
        s = self._dev(scores, torch.float32, "scores")
        i = self._dev(ids, torch.int64, "ids")
        if s.numel() != i.numel():
            raise MeviError(f"scores [{s.numel()}] and ids [{i.numel()}] differ in length")
        if out is None:
            out = (torch.empty_like(s), torch.empty_like(i))
        so = self._dev(out[0], torch.float32, "scores_out")
        io = self._dev(out[1], torch.int64, "ids_out")
        if so.numel() != s.numel() or io.numel() != i.numel():
            raise MeviError("outputs must match the inputs' length")
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_sort_candidates(self.handle, oo.numel() - 1, _ptr(oo), _ptr(s), _ptr(i), _ptr(so), _ptr(io),
                                                      self._stream()))
        return so, io

    # ---- grouped (tensor-core) re-rank ------------------------------------------
    def cluster_rerank_prefix(self, Q, D_leaf, leaf_offsets, leaf_docids, query_leaves, k, max_rows):
        """Exact top-k over the first `max_rows` candidate rows of every query (ids = rows of D_leaf)."""
        import torch

        Q = self._dev(Q, torch.float32, "Q")
        D = self._dev(D_leaf, torch.float32, "D_leaf")
        lo = self._dev(leaf_offsets, torch.int64, "leaf_offsets")
        ld = self._dev(leaf_docids, torch.int32, "leaf_docids")
        ql = self._dev(query_leaves, torch.int32, "query_leaves")
        nq, d = Q.shape
        scores = torch.empty((nq, k), dtype=torch.float32, device=Q.device)
        ids = torch.empty((nq, k), dtype=torch.int64, device=Q.device)
        ncand = torch.empty(nq, dtype=torch.int32, device=Q.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_cluster_rerank_prefix(self.handle, _ptr(Q), nq, _ptr(D), D.shape[0], d, _ptr(lo),
                                                            lo.numel() - 1, _ptr(ld), _ptr(ql), ql.shape[1], int(k),
                                                            int(max_rows), _ptr(scores), _ptr(ids), _ptr(ncand), self._stream()))
        return scores, ids, ncand

    def rerank_grouped_image(self, D_leaf, src_index, n_tiles):
        """fp16 tile image of the leaf-ordered matrix -> (image uint8 tensor, absmax, maxnorm); absmax < 0: unusable."""
        import torch

        D = self._dev(D_leaf, torch.float32, "D_leaf")
        si = self._dev(src_index, torch.int32, "src_index")
        n, d = D.shape
        assert si.numel() == n_tiles * 128
        img = torch.empty(n_tiles * 128 * d * 2, dtype=torch.uint8, device=D.device)
        a, m = C.c_float(0.0), C.c_float(0.0)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_rerank_grouped_image(self.handle, _ptr(D), n, d, _ptr(si), int(n_tiles), _ptr(img),
                                                           C.byref(a), C.byref(m), self._stream()))
        return img, float(a.value), float(m.value)

    def rerank_grouped_begin(self, Q, d_absmax, d_maxnorm, tau0=None):
        import torch

        Q = self._dev(Q, torch.float32, "Q")
        if tau0 is not None:
            self._dev(tau0, torch.float32, "tau0")
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_rerank_grouped_begin(self.handle, _ptr(Q), Q.shape[0], Q.shape[1], float(d_absmax),
                                                           float(d_maxnorm), _ptr(tau0), self._stream()))

    def leaf_lookup(self, leaves, K, leaf_keys):
        """leaves [..., M] int64 code tuples -> int32 [...] index into the ascending leaf_keys, -1 = no such leaf."""
        import torch

        leaves = self._dev(leaves, torch.int64, "leaves")
        leaf_keys = self._dev(leaf_keys, torch.int64, "leaf_keys")
        M = leaves.shape[-1]
        out = torch.empty(leaves.shape[:-1], dtype=torch.int32, device=leaves.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_leaf_lookup(self.handle, _ptr(leaves), out.numel(), M, int(K), _ptr(leaf_keys),
                                                  leaf_keys.numel(), _ptr(out), self._stream()))
        return out

    def rerank_grouped_plan(self, ql, leaf_offsets, leaf_tile0, boot_leaves, boot_min_rows, k, maxg_sample=1, maxg_last=4, pass_budget=6144):
        """Device-side round plan -> (ncand int32 [nq], weak int32 [nq], [(items, groups)] per round, n_weak)."""
        import torch

        ql = self._dev(ql, torch.int32, "ql")
        off = self._dev(leaf_offsets, torch.int64, "leaf_offsets")
        t0 = self._dev(leaf_tile0, torch.int64, "leaf_tile0")
        nq, L = ql.shape
        boot = (C.c_int32 * max(len(boot_leaves), 1))(*[int(b) for b in boot_leaves])
        sizes = (C.c_int64 * (2 * (len(boot_leaves) + 1) + 1))()
        ncand = torch.empty(nq, dtype=torch.int32, device=ql.device)
        weak = torch.empty(nq, dtype=torch.int32, device=ql.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_rerank_grouped_plan(self.handle, _ptr(ql), nq, L, _ptr(off), _ptr(t0), off.numel() - 1,
                                                          boot, len(boot_leaves), int(boot_min_rows), int(k), int(pass_budget), int(maxg_sample),
                                                          int(maxg_last), _ptr(ncand), _ptr(weak), sizes, self._stream()))
        rounds = [(int(sizes[2 * r]), int(sizes[2 * r + 1])) for r in range(len(boot_leaves) + 1)]
        return ncand, weak, rounds, int(sizes[2 * (len(boot_leaves) + 1)])

    def rerank_grouped_plan_fill(self, rnd, items, groups, device):
        """Round `rnd` of the current plan -> (item_tile, item_group, group_qid) device tensors."""
        import torch

        item_tile = torch.empty(items, dtype=torch.int32, device=device)
        item_group = torch.empty(items, dtype=torch.int32, device=device)
        group_qid = torch.empty(groups * 64, dtype=torch.int32, device=device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_rerank_grouped_plan_fill(self.handle, int(rnd), _ptr(item_tile), _ptr(item_group),
                                                               _ptr(group_qid), self._stream()))
        return item_tile, item_group, group_qid

    def rerank_grouped_round(self, Q, img, tile_row0, tile_nrows, item_tile, item_group, group_qid, k, maxg=1):
        import torch

        for name, t in (("tile_row0", tile_row0), ("tile_nrows", tile_nrows), ("item_tile", item_tile),
                        ("item_group", item_group), ("group_qid", group_qid)):
            self._dev(t, torch.int32, name)
        assert group_qid.numel() % 64 == 0 and item_tile.numel() == item_group.numel()
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_rerank_grouped_round(self.handle, _ptr(Q), Q.shape[0], Q.shape[1], _ptr(img), _ptr(tile_row0),
                                                           _ptr(tile_nrows), _ptr(item_tile), _ptr(item_group),
                                                           item_tile.numel(), _ptr(group_qid), group_qid.numel() // 64, int(maxg),
                                                           int(k), self._stream()))

    def rerank_grouped_thresholds(self, Q, tau=None):
        """tau=None: the call's current thresholds [nq] (a copy); else lift them to max(own, tau)."""
        import torch

        nq, d = Q.shape
        out = tau if tau is not None else torch.empty(nq, dtype=torch.float32, device=Q.device)
        self._dev(out, torch.float32, "tau")
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_rerank_grouped_thresholds(self.handle, nq, d, _ptr(out), 0 if tau is None else 1,
                                                                self._stream()))
        return out

    def rerank_grouped_finish(self, Q, D_leaf, k):
        """-> (scores, rows, failed int32 [nq] device mask, n_failed); n_failed == nq: the whole call is invalid."""
        import torch

        nq, d = Q.shape
        scores = torch.empty((nq, k), dtype=torch.float32, device=Q.device)
        rows = torch.empty((nq, k), dtype=torch.int64, device=Q.device)
        failed = torch.empty(nq, dtype=torch.int32, device=Q.device)
        nf = C.c_int(nq)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_rerank_grouped_finish(self.handle, _ptr(Q), nq, _ptr(D_leaf), d, int(k), _ptr(scores),
                                                            _ptr(rows), _ptr(failed), C.byref(nf), self._stream()))
        return scores, rows, failed, int(nf.value)

    def rerank_grouped_multiclus(self, Q, query_leaves, leaf_offsets, occ, n_occ, tile_leaf, aggr):
        """Attach a multi-cluster index to the grouped call begun by rerank_grouped_begin -> (query_leaves with every later
        position of a repeated leaf set to -1: the list to plan the rounds with, n_candidates int32 [nq])."""
        import torch

        ql = self._dev(query_leaves, torch.int32, "query_leaves")
        lo = self._dev(leaf_offsets, torch.int64, "leaf_offsets")
        tl = self._dev(tile_leaf, torch.int32, "tile_leaf")
        occ = self._dev(occ, torch.int32, "occ")
        nq, L = ql.shape
        masked = torch.empty_like(ql)
        ncand = torch.empty(nq, dtype=torch.int32, device=ql.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_rerank_grouped_multiclus(
                self.handle, nq, Q.shape[1], _ptr(ql), L, _ptr(lo), lo.numel() - 1, _ptr(occ) if occ.numel() else None,
                int(n_occ), _ptr(tl), _MULTICLUS_AGGR[aggr], _ptr(masked), _ptr(ncand), self._stream()))
        return masked, ncand

    def rerank_grouped_finish_multiclus(self, Q, D_leaf, k, leaf_docids, id_base=0):
        """-> (scores, ids int64 document ids, failed int32 [nq] device mask, n_failed); n_failed == nq: the call is invalid."""
        import torch

        ld = self._dev(leaf_docids, torch.int32, "leaf_docids")
        nq, d = Q.shape
        scores = torch.empty((nq, k), dtype=torch.float32, device=Q.device)
        ids = torch.empty((nq, k), dtype=torch.int64, device=Q.device)
        failed = torch.empty(nq, dtype=torch.int32, device=Q.device)
        nf = C.c_int(nq)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_rerank_grouped_finish_multiclus(self.handle, _ptr(Q), nq, _ptr(D_leaf), d, int(k), _ptr(ld),
                                                                      int(id_base), _ptr(scores), _ptr(ids), _ptr(failed),
                                                                      C.byref(nf), self._stream()))
        return scores, ids, failed, int(nf.value)

    def flat_ip_topk(self, Q, D, k, id_base=0, mode="auto"):
        import torch

        Q = self._dev(Q, torch.float32, "Q")
        D = self._dev(D, torch.float32, "D")
        nq, d = Q.shape
        n = D.shape[0]
        scores = torch.empty((nq, k), dtype=torch.float32, device=Q.device)
        ids = torch.empty((nq, k), dtype=torch.int64, device=Q.device)
        with torch.cuda.device(self.device):
            self._check(
                self.lib.mevi_flat_ip_topk(self.handle, _ptr(Q), nq, _ptr(D), n, d, int(k), int(id_base), _MODES[mode],
                                           _ptr(scores), _ptr(ids), self._stream())
            )
        return scores, ids

    def flat_index_create(self, D):
        """-> opaque handle of a persistent flat index over D [n,d] (fp16 image built once; D must stay alive)."""
        import torch

        D = self._dev(D, torch.float32, "D")
        h = _vp()
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_flat_index_create(self.handle, _ptr(D), D.shape[0], D.shape[1], C.byref(h), self._stream()))
        return h

    def flat_index_search(self, handle, Q, k, id_base=0, mode="auto"):
        import torch

        Q = self._dev(Q, torch.float32, "Q")
        nq = Q.shape[0]
        scores = torch.empty((nq, k), dtype=torch.float32, device=Q.device)
        ids = torch.empty((nq, k), dtype=torch.int64, device=Q.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_flat_index_search(self.handle, handle, _ptr(Q), nq, int(k), int(id_base), _MODES[mode],
                                                        _ptr(scores), _ptr(ids), self._stream()))
        return scores, ids

    def flat_index_destroy(self, handle):
        if handle is not None and handle.value:
            self.lib.mevi_flat_index_destroy(self.handle, handle)
            handle.value = None

    def topk_merge(self, scores_in, ids_in):
        """[S,nq,k] lists -> merged [nq,k] (score desc, id asc; -1 padded)."""
        import torch

        s = self._dev(scores_in, torch.float32, "scores_in")
        i = self._dev(ids_in, torch.int64, "ids_in")
        S, nq, k = s.shape
        scores = torch.empty((nq, k), dtype=torch.float32, device=s.device)
        ids = torch.empty((nq, k), dtype=torch.int64, device=s.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_topk_merge(self.handle, _ptr(s), _ptr(i), S, nq, k, _ptr(scores), _ptr(ids), self._stream()))
        return scores, ids

    def merge_sorted_runs(self, scores_in, ids_in, bases, run_offsets, out_offsets):
        """S runs per query, each sorted by (score desc, id asc): run r of query q is
        [bases[r] + run_offsets[r, q], bases[r] + run_offsets[r, q+1]) of scores_in / ids_in  ->  the merged CSR values
        (scores fp32 [total], ids int64 [total]) of out_offsets [nq+1].  One host sync (total, the offsets check)."""
        import torch

        s = self._dev(scores_in, torch.float32, "scores_in")
        i = self._dev(ids_in, torch.int64, "ids_in")
        b = self._dev(bases, torch.int64, "bases")
        ro = self._dev(run_offsets, torch.int64, "run_offsets")
        oo = self._dev(out_offsets, torch.int64, "out_offsets")
        S, nq1 = ro.shape
        if b.numel() != S or oo.numel() != nq1:
            raise MeviError(f"bases [{b.numel()}] and out_offsets [{oo.numel()}] must match run_offsets [{S}, {nq1}]")
        total = int(oo[-1].item())
        scores = torch.empty(max(total, 0), dtype=torch.float32, device=s.device)
        ids = torch.empty(max(total, 0), dtype=torch.int64, device=s.device)
        tmp_s, tmp_i = (torch.empty_like(scores), torch.empty_like(ids)) if S > 2 else (None, None)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_merge_sorted_runs(self.handle, _ptr(s), _ptr(i), S, nq1 - 1, _ptr(b), _ptr(ro), _ptr(oo),
                                                        total, _ptr(tmp_s), _ptr(tmp_i), _ptr(scores), _ptr(ids), self._stream()))
        return scores, ids

    def dense_scores(self, Q, P):
        import torch

        Q = self._dev(Q, torch.float32, "q_reps")
        P = self._dev(P, torch.float32, "p_reps")
        nq, d = Q.shape
        n = P.shape[0]
        out = torch.empty((nq, n), dtype=torch.float32, device=Q.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_dense_scores(self.handle, _ptr(Q), nq, _ptr(P), n, d, _ptr(out), self._stream()))
        return out

    # ---- ensemble fusion (SURVEY 8f.2) --------------------------------------
    def ensemble_cluster_ranks(self, cand_ids, cand_count, codes, query_leaves):
        """cand_ids [nq,P] int64, cand_count [nq] int32 or None, codes [N,M] int32 (the rqmapping), query_leaves
        [nq,L,M] int32 -> (cranks [nq,P] int32, num_leaves [nq] int32)."""
        import torch

        cand_ids = self._dev(cand_ids, torch.int64, "cand_ids")
        codes = self._dev(codes, torch.int32, "codes")
        leaves = self._dev(query_leaves, torch.int32, "query_leaves")
        if cand_count is not None:
            cand_count = self._dev(cand_count, torch.int32, "cand_count")
        nq, P = cand_ids.shape
        N, M = codes.shape
        if leaves.dim() != 3 or leaves.shape[0] != nq or leaves.shape[2] != M:
            raise MeviError(f"query_leaves must be [nq={nq}, L, M={M}], got {tuple(leaves.shape)}")
        cranks = torch.empty((nq, P), dtype=torch.int32, device=cand_ids.device)
        num = torch.empty((nq,), dtype=torch.int32, device=cand_ids.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_ensemble_cluster_ranks(self.handle, _ptr(cand_ids), _ptr(cand_count), nq, P,
                                                             _ptr(codes), N, M, _ptr(leaves), leaves.shape[1],
                                                             _ptr(cranks), _ptr(num), self._stream()))
        return cranks, num

    def ensemble_fuse(self, cand_ids, cand_scores, cranks, cand_count, alpha, beta, gamma, num_leaves):
        """-> (ranked ids [nq,P] int64, fused scores [nq,P] float64, distinct-document counts [nq] int32)."""
        import torch

        cand_ids = self._dev(cand_ids, torch.int64, "cand_ids")
        cand_scores = self._dev(cand_scores, torch.float64, "cand_scores")
        cranks = self._dev(cranks, torch.int32, "cranks")
        if cand_count is not None:
            cand_count = self._dev(cand_count, torch.int32, "cand_count")
        nq, P = cand_ids.shape
        if cand_scores.shape != cand_ids.shape or cranks.shape != cand_ids.shape:
            raise MeviError("cand_ids, cand_scores and cranks must have the same [nq,P] shape")
        out_ids = torch.empty((nq, P), dtype=torch.int64, device=cand_ids.device)
        out_scores = torch.empty((nq, P), dtype=torch.float64, device=cand_ids.device)
        out_count = torch.empty((nq,), dtype=torch.int32, device=cand_ids.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_ensemble_fuse(self.handle, _ptr(cand_ids), _ptr(cand_scores), _ptr(cranks),
                                                    _ptr(cand_count), nq, P, float(alpha), float(beta), float(gamma),
                                                    int(num_leaves), _ptr(out_ids), _ptr(out_scores), _ptr(out_count),
                                                    self._stream()))
        return out_ids, out_scores, out_count

    def ensemble_positions(self, ranked, ranked_count, targets, target_count):
        """positions [nq,G] int32 of targets[q,g] in ranked[q] (first occurrence), -1 if absent."""
        import torch

        ranked = self._dev(ranked, torch.int64, "ranked")
        targets = self._dev(targets, torch.int64, "targets")
        if ranked_count is not None:
            ranked_count = self._dev(ranked_count, torch.int32, "ranked_count")
        if target_count is not None:
            target_count = self._dev(target_count, torch.int32, "target_count")
        nq, P = ranked.shape
        G = targets.shape[1]
        out = torch.empty((nq, G), dtype=torch.int32, device=ranked.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_ensemble_positions(self.handle, _ptr(ranked), _ptr(ranked_count), nq, P,
                                                         _ptr(targets), _ptr(target_count), G, _ptr(out), self._stream()))
        return out

    def ensemble_first_hit(self, ranked, ranked_count, query_index, offsets, array):
        """first_hit [nq] int32: first rank whose document lists query_index[q] among its inverse answers, -1 if none."""
        import torch

        ranked = self._dev(ranked, torch.int64, "ranked")
        query_index = self._dev(query_index, torch.int64, "query_index")
        offsets = self._dev(offsets, torch.int32, "offsets")
        array = self._dev(array, torch.int32, "array")
        if ranked_count is not None:
            ranked_count = self._dev(ranked_count, torch.int32, "ranked_count")
        nq, P = ranked.shape
        out = torch.empty((nq,), dtype=torch.int32, device=ranked.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mevi_ensemble_first_hit(self.handle, _ptr(ranked), _ptr(ranked_count), nq, P,
                                                         _ptr(query_index), _ptr(offsets), offsets.numel(), _ptr(array),
                                                         _ptr(out), self._stream()))
        return out


_contexts: Dict[int, Context] = {}


def get_context(device: Optional[int] = None) -> Context:
    import torch

    if not torch.cuda.is_available():
        raise MeviError("no CUDA device visible: mevi_b200 has no CPU path")
    if device is None:
        device = torch.cuda.current_device()
    if isinstance(device, torch.device):
        device = device.index if device.index is not None else torch.cuda.current_device()
    if device not in _contexts:
        _contexts[device] = Context(device)
    return _contexts[device]
