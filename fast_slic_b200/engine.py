"""Device-side engine: one `Engine` == one fslic_ctx (fixed H, W, K, max batch) on one GPU.

Host logic only -- tensors in, tensors out; all arithmetic happens in libfslic_b200.so.
PyTorch is used for device memory and streams, nothing else.
"""
import ctypes as C
import threading

import numpy as np
import torch

from . import _lib
from ._lib import Params, check

CLUSTER_DTYPE = np.dtype(
    [("y", "<f4"), ("x", "<f4"), ("r", "<f4"), ("g", "<f4"), ("b", "<f4"), ("a", "<f4"),
     ("number", "<u2"), ("is_active", "u1"), ("is_updatable", "u1"), ("num_members", "<u4")]
)  # == Cluster, /root/reference/src/fast-slic-common.h:10-23
assert CLUSTER_DTYPE.itemsize == 32


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("fast_slic_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


class Engine:
    """A context is NOT safe for concurrent calls (shared staging buffers, streams, graph key; INTEGRATION.md).
    `lock` serialises them: every blocking entry point below holds it for the whole call, and callers that pair
    `iterate_host_async` with `wait` from several threads must hold it across the pair themselves."""

    def __init__(self, H, W, K=None, max_batch=1, device=0, cca_only=False):
        require_cuda()
        self.cca_only = bool(cca_only)
        self.H, self.W, self.K, self.max_batch = int(H), int(W), (1 if cca_only else int(K)), int(max_batch)
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self._L = _lib.lib()
        self.lock = threading.RLock()
        h = C.c_void_p()
        if cca_only:  # scratch of the connectivity stage alone; K is an argument of enforce_connectivity()
            check(self._L.fslic_b200_create_cca(self.device.index, self.H, self.W, self.max_batch, C.byref(h)))
        else:
            check(self._L.fslic_b200_create(self.device.index, self.H, self.W, self.K, self.max_batch, C.byref(h)))
        self._h = h
        self.S = self._L.fslic_b200_get_S(self._h)

    def close(self):
        with self.lock:
            if getattr(self, "_h", None):
                self._L.fslic_b200_destroy(self._h)
                self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers -------------------------------------------------------------------------------
    def _check_images(self, images):
        if images.dtype != torch.uint8 or images.dim() != 4 or images.shape[1:] != (self.H, self.W, 3):
            raise ValueError("images must be uint8 [B, %d, %d, 3]" % (self.H, self.W))
        if not images.is_contiguous():
            raise ValueError("images must be contiguous")
        if images.device != self.device:
            raise ValueError("images must live on %s" % self.device)
        if images.shape[0] > self.max_batch:
            raise ValueError("batch larger than the engine's max_batch")

    def new_clusters(self, batch):
        return torch.zeros((batch, self.K, 32), dtype=torch.uint8, device=self.device)

    @staticmethod
    def params(compactness=10.0, min_size_factor=0.25, subsample_stride=3, convert_to_lab=True, max_iter=10,
               collect_timing=0):
        return Params(float(compactness), float(min_size_factor), int(subsample_stride), int(bool(convert_to_lab)),
                      int(max_iter), int(collect_timing))

    def set_manhattan_spatial_dist(self, manhattan):
        """The spatial term of every later iterate call: L1 (True, the default) or Euclidean (False), like the reference's
        context field manhattan_spatial_dist.  It is context state: callers sharing a context set it under `lock`."""
        check(self._L.fslic_b200_set_manhattan_spatial_dist(self._h, int(bool(manhattan))))

    # -- device entry points -------------------------------------------------------------------
    def initialize_clusters(self, images, clusters=None):
        self._check_images(images)
        B = images.shape[0]
        if clusters is None:
            clusters = self.new_clusters(B)
        with self.lock:
            check(self._L.fslic_b200_initialize_clusters(self._h, images.data_ptr(), clusters.data_ptr(), B,
                                                         _stream_ptr(self.device)))
        return clusters

    def iterate(self, images, clusters, params, labels=None):
        """images u8[B,H,W,3] (cuda), clusters u8[B,K,32] (cuda, updated in place) -> labels u16 as int16[B,H,W]."""
        self._check_images(images)
        B = images.shape[0]
        if labels is None:
            labels = torch.empty((B, self.H, self.W), dtype=torch.int16, device=self.device)
        with self.lock:
            check(self._L.fslic_b200_iterate(self._h, images.data_ptr(), clusters.data_ptr(), labels.data_ptr(), B,
                                             C.byref(params), _stream_ptr(self.device)))
        return labels

    REAL_DIST_VARIANTS = {"standard": 0, "l2": 1, "noq": 2}

    def iterate_real(self, variant, images, clusters, params, labels=None):
        """Float-distance variants (fslic_b200_iterate_real): variant "standard" | "l2" | "noq"; device tensors."""
        self._check_images(images)
        B = images.shape[0]
        if labels is None:
            labels = torch.empty((B, self.H, self.W), dtype=torch.int16, device=self.device)
        with self.lock:
            check(self._L.fslic_b200_iterate_real(self._h, self.REAL_DIST_VARIANTS[variant], images.data_ptr(),
                                                  clusters.data_ptr(), labels.data_ptr(), B, C.byref(params),
                                                  _stream_ptr(self.device)))
        return labels

    def iterate_preemptive(self, images, clusters, params, preemptive_thres, labels=None):
        """`preemptive=True` of the reference (fslic_b200_iterate_preemptive); device tensors like iterate()."""
        self._check_images(images)
        B = images.shape[0]
        if labels is None:
            labels = torch.empty((B, self.H, self.W), dtype=torch.int16, device=self.device)
        with self.lock:
            check(self._L.fslic_b200_iterate_preemptive(self._h, images.data_ptr(), clusters.data_ptr(), labels.data_ptr(), B,
                                                        C.byref(params), C.c_float(preemptive_thres), _stream_ptr(self.device)))
        return labels

    def enforce_connectivity(self, labels, K, min_threshold):
        """In place on int16/uint16 labels [B,H,W] (cuda)."""
        B = labels.shape[0]
        with self.lock:
            check(self._L.fslic_b200_enforce_connectivity(self._h, labels.data_ptr(), B, int(K), int(min_threshold),
                                                          _stream_ptr(self.device)))
        return labels

    def rgb_to_quad(self, images, convert_to_lab=True):
        self._check_images(images)
        B = images.shape[0]
        quad = torch.empty((B, self.H, self.W, 4), dtype=torch.uint8, device=self.device)
        check(self._L.fslic_b200_rgb_to_quad(self._h, images.data_ptr(), quad.data_ptr(), B, int(convert_to_lab),
                                             _stream_ptr(self.device)))
        return quad

    def debug_stages(self, batch):
        quad = torch.empty((batch, self.H, self.W, 4), dtype=torch.uint8, device=self.device)
        pre = torch.empty((batch, self.H, self.W), dtype=torch.int16, device=self.device)
        check(self._L.fslic_b200_debug_stages(self._h, quad.data_ptr(), pre.data_ptr(), batch,
                                              _stream_ptr(self.device)))
        return quad, pre

    def debug_heap_select(self, area, middle):
        area = area.to(self.device, torch.int32).contiguous()
        kept = torch.empty(area.numel(), dtype=torch.uint8, device=self.device)
        check(self._L.fslic_b200_debug_heap_select(self._h, area.data_ptr(), area.numel(), int(middle),
                                                   kept.data_ptr(), _stream_ptr(self.device)))
        return kept

    # -- host entry points (numpy in / numpy out, copies inside) ---------------------------------
    def initialize_clusters_host(self, images_np):
        B = images_np.shape[0]
        clusters = np.zeros((B, self.K), CLUSTER_DTYPE)
        with self.lock:
            check(self._L.fslic_b200_initialize_clusters_host(self._h, images_np.ctypes.data, clusters.ctypes.data, B))
        return clusters

    def iterate_host(self, images_np, clusters_np, params, labels_np=None):
        B = images_np.shape[0]
        if labels_np is None:
            labels_np = np.empty((B, self.H, self.W), np.int16)
        with self.lock:
            check(self._L.fslic_b200_iterate_host(self._h, images_np.ctypes.data, clusters_np.ctypes.data,
                                                  labels_np.ctypes.data, B, C.byref(params)))
        return labels_np

    def iterate_host_async(self, images_np, clusters_np, params, labels_np):
        """Enqueue one host batch and return; `wait()` blocks until labels_np / clusters_np are filled.
        All three arrays must live in pinned memory and must not be touched in between."""
        self._inflight = (images_np, clusters_np, labels_np, params)  # keep the buffers alive
        check(self._L.fslic_b200_iterate_host_async(self._h, images_np.ctypes.data, clusters_np.ctypes.data,
                                                    labels_np.ctypes.data, images_np.shape[0], C.byref(params)))

    def wait(self):
        check(self._L.fslic_b200_wait(self._h))
        self._inflight = None

    def stage_ms(self):
        out = (C.c_float * 6)()
        check(self._L.fslic_b200_stage_ms(self._h, out, 6))
        return dict(zip(_lib.STAGE_NAMES, [float(v) for v in out]))

    def cca_stage_ms(self):
        out = (C.c_float * 6)()
        check(self._L.fslic_b200_cca_stage_ms(self._h, out, 6))
        return dict(zip(_lib.CCA_STAGE_NAMES, [float(v) for v in out]))

    def assign_kernel_time(self):
        """(total ms, launches) of the fused assign+update kernel in the last iterate (collect_timing=2)."""
        ms, n = C.c_float(), C.c_int()
        check(self._L.fslic_b200_assign_kernel_time(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def cca_counters(self, image=0):
        out = (C.c_int32 * 8)()
        check(self._L.fslic_b200_debug_cca_counters(self._h, out, image))
        return dict(zip(("ncomp", "ncand", "nkept", "sel_mode", "keep_thres", "need_sim", "heap_ops", "kth_area"), list(out)))

    def select_profile(self, image=0):
        """Clock counts of the std::partial_sort replay (needs FSLIC_SELPROF=1 when the context is created)."""
        out = (C.c_longlong * 8)()
        check(self._L.fslic_b200_debug_select_profile(self._h, out, image))
        return dict(zip(("total", "filter", "build", "replay", "trips", "queued", "chunks", "ncomp"), list(out)))

    def assign_impl(self):
        """5: TMA-staged assign kernel, 4: LDG kernel, 0: brute force (last pass of the last iterate)."""
        return int(self._L.fslic_b200_debug_assign_impl(self._h))

    def launches_last_iterate(self):
        return int(self._L.fslic_b200_launches_last_iterate(self._h))
