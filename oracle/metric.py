"""oracle/metric.py -- TEST INFRASTRUCTURE ONLY: the two CPU checkers of the spatial metric (`manhattan_spatial_dist`).

* ``MetricPort`` : oracle/liboracle_metric.so -- the plain-C restatement (oracle/spatial_metric.c)
* ``MetricRef``  : oracle/_ref/libfslic_ref_metric.so -- the unmodified reference behind oracle/ref_shim_metric.cpp

Both are built by oracle/metric.mk.  ``manhattan=True`` gives the answers of oracle.oracle.Port / Ref.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from .oracle import CLUSTER_DTYPE, Port, Ref, _p, _u8p, _u16p  # noqa: F401  (CLUSTER_DTYPE re-exported)

_HERE = os.path.dirname(os.path.abspath(__file__))


def build(force=False):
    """Compile liboracle_metric.so (always possible) and the reference door (only where /root/reference exists)."""
    if force or not os.path.exists(os.path.join(_HERE, "liboracle_metric.so")):
        subprocess.check_call(["make", "-C", _HERE, "-f", "metric.mk", "liboracle_metric.so"], stdout=subprocess.DEVNULL)
    if os.path.isdir("/root/reference/src") and (
        force or not os.path.exists(os.path.join(_HERE, "_ref", "libfslic_ref_metric.so"))
    ):
        subprocess.check_call(["make", "-C", _HERE, "-f", "metric.mk", "ref"], stdout=subprocess.DEVNULL)


class MetricPort:
    """Plain-C restatement; `initialize` is the metric-independent one of oracle.Port."""

    def __init__(self):
        build()
        self.lib = C.CDLL(os.path.join(_HERE, "liboracle_metric.so"))
        assert self.lib.orc_sizeof_cluster() == 32
        self.lib.orc_ref_hypotf.restype = C.c_float
        self._port = Port()

    def hypotf(self, a, b):
        """glibc's hypotf on integers as the restatement computes it: float(sqrt(double(a)^2 + double(b)^2))."""
        return float(self.lib.orc_ref_hypotf(int(a), int(b)))

    def spatial_patch(self, S, compactness, color_shift):
        patch = np.zeros((2 * S + 1, 2 * S + 1), np.uint16)
        self.lib.orc_spatial_patch_euclid(S, C.c_float(compactness), color_shift, _p(patch, _u16p))
        return patch

    def initialize(self, image, K):
        return self._port.initialize(image, K)

    def iterate(self, image, clusters, max_iter=10, compactness=10.0, min_size_factor=0.25, stride=3,
                convert_to_lab=True, preemptive=False, preemptive_thres=0.05, manhattan=True):
        """-> (labels, pre-CCA labels); `clusters` is updated in place."""
        image = np.ascontiguousarray(image)
        H, W, _ = image.shape
        out = np.zeros((H, W), np.uint16)
        pre = np.zeros((H, W), np.uint16)
        self.lib.orc_iterate_metric(H, W, len(clusters), _p(image, _u8p), clusters.ctypes.data_as(C.c_void_p),
                                    _p(out, _u16p), max_iter, C.c_float(compactness), C.c_float(min_size_factor), stride,
                                    int(convert_to_lab), int(bool(preemptive)), C.c_float(preemptive_thres),
                                    int(bool(manhattan)), _p(pre, _u16p))
        return out, pre

    def iterate_real(self, variant, image, clusters, max_iter=10, compactness=10.0, min_size_factor=0.25, stride=3,
                     convert_to_lab=True, manhattan=True):
        image = np.ascontiguousarray(image)
        H, W, _ = image.shape
        out = np.zeros((H, W), np.uint16)
        pre = np.zeros((H, W), np.uint16)
        self.lib.orc_iterate_real_metric(int(variant), H, W, len(clusters), _p(image, _u8p),
                                         clusters.ctypes.data_as(C.c_void_p), _p(out, _u16p), max_iter,
                                         C.c_float(compactness), C.c_float(min_size_factor), stride, int(convert_to_lab),
                                         int(bool(manhattan)), _p(pre, _u16p))
        return out, pre


class MetricRef:
    """The unmodified reference (x64/avx2 arch for the integer path), OpenMP threads = num_threads (-1: all)."""

    @staticmethod
    def available():
        return os.path.exists(os.path.join(_HERE, "_ref", "libfslic_ref_metric.so")) or os.path.isdir("/root/reference/src")

    def __init__(self):
        build()
        self._ref = Ref()
        self.lib = C.CDLL(os.path.join(_HERE, "_ref", "libfslic_ref_metric.so"))

    def initialize(self, image, K):
        return self._ref.initialize(image, K)

    def iterate(self, image, clusters, max_iter=10, compactness=10.0, min_size_factor=0.25, stride=3,
                convert_to_lab=True, preemptive=False, preemptive_thres=0.05, manhattan=True, arch="x64/avx2",
                num_threads=-1):
        image = np.ascontiguousarray(image)
        H, W, _ = image.shape
        out = np.zeros((H, W), np.uint16)
        pre = np.zeros((H, W), np.uint16)
        self.lib.refm_iterate(1 if arch == "x64/avx2" else 0, H, W, len(clusters), _p(image, _u8p),
                              clusters.ctypes.data_as(C.c_void_p), _p(out, _u16p), max_iter, C.c_float(compactness),
                              C.c_float(min_size_factor), stride, int(convert_to_lab), int(bool(preemptive)),
                              C.c_float(preemptive_thres), int(bool(manhattan)), num_threads, _p(pre, _u16p))
        return out, pre

    def iterate_real(self, variant, image, clusters, max_iter=10, compactness=10.0, min_size_factor=0.25, stride=3,
                     convert_to_lab=True, manhattan=True, num_threads=2):
        image = np.ascontiguousarray(image)
        H, W, _ = image.shape
        out = np.zeros((H, W), np.uint16)
        pre = np.zeros((H, W), np.uint16)
        self.lib.refm_iterate_real(int(variant), H, W, len(clusters), _p(image, _u8p),
                                   clusters.ctypes.data_as(C.c_void_p), _p(out, _u16p), max_iter, C.c_float(compactness),
                                   C.c_float(min_size_factor), stride, int(convert_to_lab), int(bool(manhattan)),
                                   num_threads, _p(pre, _u16p))
        return out, pre
