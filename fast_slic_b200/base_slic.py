"""Python surface of the reference, re-hosted on the CUDA engine.

Mirrors /root/reference/fast_slic/base_slic.py:3-62 (BaseSlic / Slic: same kwargs, defaults,
properties, return dtype) and the Cython ``SlicModel`` (/root/reference/cfast_slic.pyx:15-260,
attributes cfast_slic.pxd:104-120).  Implemented: the default integer-distance path of the north star, the
float-distance variants, `preemptive` and both spatial metrics (`manhattan_spatial_dist`); LSC raises NotImplementedError.
"""
import collections
import contextlib
import json
import threading

import numpy as np
import torch

from . import _lib
from .engine import CLUSTER_DTYPE, Engine, require_cuda

ARCH_NAME = "cuda/sm_100a"
_SUPPORTED_ARCHS = (ARCH_NAME,)

# Contexts are cached and reused (the reference rebuilds one per call, cfast_slic.pyx:171-197), in a small LRU:
# a data set of variable-sized images must not pin one full context (~30 B/pixel of device memory) per shape
# for ever.  Evicted contexts are closed; `Engine.lock` keeps a context another thread is using alive until
# that call returns, and the cache itself is guarded by `_cache_lock`.
ENGINE_CACHE_SIZE = 6
_engines = collections.OrderedDict()
_cache_lock = threading.Lock()


def _cached(key, make, min_batch):
    with _cache_lock:
        eng = _engines.get(key)
        stale = []
        if eng is not None and eng.max_batch < min_batch:
            stale.append(_engines.pop(key))
            eng = None
        if eng is None:
            eng = make()
            _engines[key] = eng
        _engines.move_to_end(key)
        while len(_engines) > ENGINE_CACHE_SIZE:
            stale.append(_engines.popitem(last=False)[1])
    for e in stale:
        e.close()  # takes e.lock: waits for a call in flight on another thread
    return eng


def get_engine(H, W, K, batch=1, device=0):
    key = ("slic", int(device), int(H), int(W), int(K))
    return _cached(key, lambda: Engine(H, W, K, max_batch=batch, device=device), batch)


def get_cca_engine(H, W, batch=1, device=0):
    """Connectivity-only context: keyed on the shape alone (the label range K is a call argument)."""
    key = ("cca", int(device), int(H), int(W))
    return _cached(key, lambda: Engine(H, W, max_batch=batch, device=device, cca_only=True), batch)


@contextlib.contextmanager
def _locked(getter):
    """The cached context of `getter()`, locked for the duration of the block.  If another thread evicted (and
    closed) it between the lookup and the lock, look it up again."""
    while True:
        eng = getter()
        eng.lock.acquire()
        if eng._h is not None:
            break
        eng.lock.release()
    try:
        yield eng
    finally:
        eng.lock.release()


@contextlib.contextmanager
def _spatial_metric(eng, manhattan):
    """Inside a `_locked` block: the context computes with this model's spatial metric for the duration of the call and
    is handed back with the default (Manhattan) one -- contexts are shared through the cache."""
    eng.set_manhattan_spatial_dist(manhattan)
    try:
        yield eng
    finally:
        if not manhattan:
            eng.set_manhattan_spatial_dist(True)


def clear_engine_cache():
    with _cache_lock:
        engines = list(_engines.values())
        _engines.clear()
    for e in engines:
        e.close()


def get_supported_archs():
    """== cfast_slic.get_supported_archs (cfast_slic.pyx:358-369)."""
    return list(_SUPPORTED_ARCHS)


def is_supported_arch(arch_name):
    return arch_name in _SUPPORTED_ARCHS


def _check_image(image):
    # the Cython signature `const uint8_t [:, :, ::1]` raises ValueError on dtype / ndim / contiguity
    if not isinstance(image, np.ndarray):
        image = np.asarray(image)
    if image.dtype != np.uint8:
        raise ValueError("Buffer dtype mismatch, expected 'const uint8_t' but got %r" % (image.dtype.name,))
    if image.ndim != 3:
        raise ValueError("Buffer has wrong number of dimensions (expected 3, got %d)" % image.ndim)
    if not image.flags["C_CONTIGUOUS"]:
        raise ValueError("ndarray is not C-contiguous")
    if image.shape[2] != 3:
        raise ValueError("nchan != 3")  # cfast_slic.pyx:125,153
    return image


class SlicModel(object):
    """== cfast_slic.SlicModel: owns the Cluster[K] array (host copy, 32-byte records)."""

    def __init__(self, num_components, arch_name=ARCH_NAME, real_dist=False):
        if not is_supported_arch(arch_name):
            raise NotImplementedError("Unsupported arch " + repr(arch_name))  # cfast_slic.pyx:21-22
        if num_components >= 65534:
            raise ValueError("num_components cannot exceed 65534")  # cfast_slic.pyx:24-25
        elif num_components <= 0:
            raise ValueError("num_components should be a non-negative integer")  # cfast_slic.pyx:26-27
        self._num_components = int(num_components)
        self.num_threads = -1
        self.arch_name = arch_name
        self.real_dist = real_dist
        self.real_dist_type = "standard"
        self.convert_to_lab = False
        self.float_color = True
        self.debug_mode = False
        self._clusters = np.zeros(self._num_components, CLUSTER_DTYPE)
        self.initialized = False
        self.preemptive = False
        self.preemptive_thres = 0.05
        self.manhattan_spatial_dist = True
        self.last_timing_report = None
        self.last_recorder_report = None
        self.device = 0

    @property
    def num_components(self):
        return self._num_components

    def copy(self):
        """cfast_slic.pyx:45-49 (copies the clusters and the initialized flag only)."""
        result = SlicModel(self._num_components)
        result._clusters = self._clusters.copy()
        result.initialized = self.initialized
        return result

    def to_yxmrgb(self):
        """== cfast_slic.SlicModel.to_yxmrgb (cfast_slic.pyx:100-113): float [K, 6] rows (y, x, num_members, r, g, b)."""
        c = self._clusters
        out = np.empty((self._num_components, 6), dtype=float)
        for col, name in enumerate(("y", "x", "num_members", "r", "g", "b")):
            out[:, col] = c[name]
        return out

    @property
    def clusters(self):
        """cfast_slic.pyx:51-66."""
        return [
            dict(number=int(c["number"]), yx=(float(c["y"]), float(c["x"])),
                 color=(float(c["r"]), float(c["g"]), float(c["b"])), num_members=int(c["num_members"]))
            for c in self._clusters
        ]

    @clusters.setter
    def clusters(self, clusters):
        """cfast_slic.pyx:68-98: yx -> uint16, colour -> uint8, number = index."""
        def c_uint(v, bits):  # Cython's object -> unsigned C integer conversion: truncates floats, range-checks
            v = int(v)
            if v < 0 or v >= (1 << bits):
                raise OverflowError("value too large to convert to uint%d_t" % bits)
            return v

        new = np.zeros(len(clusters), CLUSTER_DTYPE)
        for i, d in enumerate(clusters):
            y, x = d["yx"]
            r, g, b = d["color"]
            new[i]["number"] = i
            new[i]["y"] = c_uint(y, 16)
            new[i]["x"] = c_uint(x, 16)
            new[i]["r"] = c_uint(r, 8)
            new[i]["g"] = c_uint(g, 8)
            new[i]["b"] = c_uint(b, 8)
            new[i]["num_members"] = c_uint(d["num_members"], 32)
            new[i]["is_active"] = 1
            new[i]["is_updatable"] = 1
        self._clusters = new
        self._num_components = len(clusters)
        self.initialized = True

    @property
    def cluster_array(self):
        """The raw Cluster[K] records as a numpy structured array (a view, not part of the reference API)."""
        return self._clusters

    def _unsupported(self):
        if self.real_dist and self.real_dist_type not in Engine.REAL_DIST_VARIANTS:
            raise NotImplementedError("real_dist_type %r (LSC) is outside the CUDA hot path" % (self.real_dist_type,))
        if self.preemptive and self.real_dist:
            raise NotImplementedError("preemptive=True together with a float-distance variant is outside the CUDA hot path")

    def initialize(self, image):
        """cfast_slic.pyx:124-147."""
        image = _check_image(image)
        require_cuda()
        H, W, _ = image.shape
        with _locked(lambda: get_engine(H, W, self._num_components, 1, self.device)) as eng:
            self._clusters = eng.initialize_clusters_host(image[None])[0]
        self.initialized = True

    def iterate(self, image, max_iter, compactness, min_size_factor, subsample_stride):
        """cfast_slic.pyx:150-260: returns int16[H, W]."""
        if not self.initialized:
            raise RuntimeError("Slic model is not initialized")  # cfast_slic.pyx:151
        image = _check_image(image)
        self._unsupported()
        require_cuda()
        H, W, _ = image.shape
        params = Engine.params(compactness, min_size_factor, subsample_stride, self.convert_to_lab, max_iter,
                               collect_timing=1)
        if self.real_dist or self.preemptive:
            return self._iterate_real_dist(image, params)
        clusters = np.ascontiguousarray(self._clusters)[None]
        # the lock covers the timing read-out too: it belongs to this call, not to another thread's next one
        with _locked(lambda: get_engine(H, W, self._num_components, 1, self.device)) as eng:
            with _spatial_metric(eng, self.manhattan_spatial_dist):
                labels = eng.iterate_host(image[None], clusters, params)
            ms = eng.stage_ms()
            cca = eng.cca_stage_ms()
        self._clusters = clusters[0]

        def node(name, ms_value, children=()):
            return {"name": name, "duration": int(ms_value * 1000), "children": list(children)}

        # same tree as fstimer builds (context.cpp:112-192, cca.cpp:194-263); `update` is fused into `assign` here
        self.last_timing_report = json.dumps(node("iterate", ms["iterate"], [
            node("cielab_conversion", ms["cielab_conversion"]), node("assign", ms["assign"]), node("update", ms["update"]),
            node("full_assign", ms["full_assign"]),
            node("enforce_connectivity", ms["enforce_connectivity"],
                 [node("cca", ms["enforce_connectivity"], [node(n, cca[n]) for n in _lib.CCA_STAGE_NAMES])]),
        ]))
        self.last_recorder_report = b'{"snapshots":[]}'
        return labels[0]


def _iterate_real_dist(self, image, params):
    """cfast_slic.pyx:198-252: the float-distance contexts (fslic_b200_iterate_real) and the `preemptive` option
    (fslic_b200_iterate_preemptive), both through device buffers."""
    H, W, _ = image.shape
    with _locked(lambda: get_engine(H, W, self._num_components, 1, self.device)) as eng:
        with torch.cuda.device(eng.device):
            img = torch.from_numpy(image).to(eng.device)[None]
            cl = torch.from_numpy(np.ascontiguousarray(self._clusters).view(np.uint8).reshape(1, -1, 32).copy()).to(eng.device)
            with _spatial_metric(eng, self.manhattan_spatial_dist):
                if self.preemptive:  # cfast_slic.pyx:183-184
                    labels = eng.iterate_preemptive(img, cl, params, self.preemptive_thres)
                else:
                    labels = eng.iterate_real(self.real_dist_type, img, cl, params)
            ms = eng.stage_ms()
            self._clusters = cl[0].cpu().numpy().view(CLUSTER_DTYPE).reshape(-1)
            out = labels[0].cpu().numpy()
    self.last_timing_report = json.dumps({
        "name": "iterate", "duration": int(ms["iterate"] * 1000),
        "children": [{"name": n, "duration": int(ms[n] * 1000), "children": []}
                     for n in ("cielab_conversion", "assign", "update", "full_assign", "enforce_connectivity")]})
    self.last_recorder_report = b'{"snapshots":[]}'
    return out


SlicModel._iterate_real_dist = _iterate_real_dist


class NodeConnectivity(object):
    """== cfast_slic.NodeConnectivity (cfast_slic.pyx:322-345): `tolist()` -> list of neighbour lists."""

    def __init__(self, counts, neighbors):
        self._counts, self._neighbors = counts, neighbors

    def tolist(self):
        return [self._neighbors[k, :self._counts[k]].tolist() for k in range(len(self._counts))]


def _check_assignments(assignments):
    if not isinstance(assignments, np.ndarray) or assignments.dtype != np.int16 or assignments.ndim != 2 \
            or not assignments.flags["C_CONTIGUOUS"]:
        raise ValueError("assignments must be a C-contiguous int16[H, W] array")
    return assignments


def _graph_get_connectivity(self, assignments):
    """cfast_slic.pyx:262-270 -> fast_slic_get_connectivity (fast-slic.cpp:16-78) on the GPU."""
    assignments = _check_assignments(assignments)
    require_cuda()
    H, W = assignments.shape
    K = self.num_components
    dev = torch.device("cuda", self.device)
    L = _lib.lib()
    with torch.cuda.device(dev):
        lab = torch.from_numpy(assignments).to(dev)
        counts = torch.empty(K, dtype=torch.int32, device=dev)
        nb = torch.empty((K, 12), dtype=torch.int32, device=dev)
        nbytes = int(L.fslic_b200_connectivity_scratch_bytes(K))
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _lib.check(L.fslic_b200_get_connectivity(self.device, H, W, K, lab.data_ptr(), counts.data_ptr(), nb.data_ptr(),
                                                 scratch.data_ptr(), nbytes, torch.cuda.current_stream(dev).cuda_stream))
        return NodeConnectivity(counts.cpu().numpy(), nb.cpu().numpy().view(np.uint32))


def _graph_get_knn_connectivity(self, assignments, num_neighbors):
    """cfast_slic.pyx:272-281.  Not provided: the reference's fast_slic_knn_connectivity indexes its cell vector with
    a float expression that overruns it for centres low in the last cell row (fast-slic.cpp:88) -- it crashes on
    ordinary inputs, so there is no result to reproduce."""
    raise NotImplementedError("get_knn_connectivity: the reference implementation is out of bounds (fast-slic.cpp:88)")


def _graph_get_mask_density(self, mask, assignments):
    """cfast_slic.pyx:283-302 -> fast_slic_get_mask_density (fast-slic.cpp:141-155): uint8[K]."""
    assignments = _check_assignments(assignments)
    mask = np.ascontiguousarray(mask)
    if mask.dtype != np.uint8 or mask.ndim != 2:
        raise ValueError("mask must be uint8[H, W]")
    H, W = assignments.shape
    if mask.shape[0] != H or mask.shape[1] != W:
        raise ValueError("The shape of mask does not match the one of assignments")  # cfast_slic.pyx:289-290
    require_cuda()
    K = self.num_components
    dev = torch.device("cuda", self.device)
    L = _lib.lib()
    with torch.cuda.device(dev):
        lab = torch.from_numpy(assignments).to(dev)
        msk = torch.from_numpy(mask).to(dev)
        cl = torch.from_numpy(np.ascontiguousarray(self._clusters).view(np.uint8)).to(dev)
        dens = torch.empty(K, dtype=torch.uint8, device=dev)
        scratch = torch.empty(K, dtype=torch.int32, device=dev)
        _lib.check(L.fslic_b200_get_mask_density(self.device, H, W, K, cl.data_ptr(), lab.data_ptr(), msk.data_ptr(),
                                                 dens.data_ptr(), scratch.data_ptr(),
                                                 torch.cuda.current_stream(dev).cuda_stream))
        return dens.cpu().numpy()


def _graph_broadcast_density_to_mask(self, densities, assignments):
    """cfast_slic.pyx:304-320 -> fast_slic_cluster_density_to_mask (fast-slic.cpp:157-168): uint8[H, W]."""
    assignments = _check_assignments(assignments)
    densities = np.ascontiguousarray(densities)
    K = self.num_components
    if densities.dtype != np.uint8 or densities.ndim != 1:
        raise ValueError("densities must be uint8[K]")
    if densities.shape[0] != K:
        raise ValueError("The shape of densities should match the number of clusters")  # cfast_slic.pyx:309-310
    require_cuda()
    H, W = assignments.shape
    dev = torch.device("cuda", self.device)
    L = _lib.lib()
    with torch.cuda.device(dev):
        lab = torch.from_numpy(assignments).to(dev)
        dens = torch.from_numpy(densities).to(dev)
        out = torch.empty((H, W), dtype=torch.uint8, device=dev)
        _lib.check(L.fslic_b200_cluster_density_to_mask(self.device, H, W, K, lab.data_ptr(), dens.data_ptr(),
                                                        out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))
        return out.cpu().numpy()


SlicModel.get_connectivity = _graph_get_connectivity
SlicModel.get_knn_connectivity = _graph_get_knn_connectivity
SlicModel.get_mask_density = _graph_get_mask_density
SlicModel.broadcast_density_to_mask = _graph_broadcast_density_to_mask


class BaseSlic(object):
    """== fast_slic.base_slic.BaseSlic (/root/reference/fast_slic/base_slic.py:3-59)."""
    arch_name = "__TODO__"

    def __init__(self, num_components=400, slic_model=None, compactness=10, min_size_factor=0.25,
                 subsample_stride=3, convert_to_lab=True, preemptive=False, preemptive_thres=0.05,
                 manhattan_spatial_dist=True, debug_mode=False, num_threads=-1):
        self.compactness = compactness
        self.subsample_stride = subsample_stride
        self.min_size_factor = min_size_factor
        self._slic_model = slic_model and slic_model.copy() or self.make_slic_model(num_components)
        self._last_assignment = None
        self.convert_to_lab = convert_to_lab
        self._slic_model.preemptive = preemptive
        self._slic_model.preemptive_thres = preemptive_thres
        self._slic_model.manhattan_spatial_dist = manhattan_spatial_dist
        self._slic_model.num_threads = num_threads
        self._slic_model.debug_mode = debug_mode

    @property
    def convert_to_lab(self):
        return self._slic_model.convert_to_lab

    @convert_to_lab.setter
    def convert_to_lab(self, v):
        self._slic_model.convert_to_lab = v

    @property
    def slic_model(self):
        return self._slic_model

    @property
    def last_assignment(self):
        return self._last_assignment

    def iterate(self, image, max_iter=10):
        self._slic_model._unsupported()  # (before any device work: LSC etc. fail the same way with or without a GPU)
        if not self._slic_model.initialized:
            self._slic_model.initialize(image)
        assignment = self._slic_model.iterate(image, max_iter, self.compactness, self.min_size_factor,
                                              self.subsample_stride)
        self._last_assignment = assignment
        return assignment

    @property
    def num_components(self):
        return self._slic_model.num_components

    def make_slic_model(self, num_components):
        return SlicModel(num_components, self.arch_name)

    # ---- batch extension (no counterpart in the reference: it has no batch API) -------------------
    def iterate_batch(self, images, max_iter=10, clusters=None, return_clusters=False):
        """Independent images [B,H,W,3] (uint8, numpy or cuda tensor) -> int16 labels [B,H,W] of the same kind.

        Every image gets its own freshly seeded cluster set (or `clusters` to warm start, a [B,K]
        structured array / [B,K,32] uint8 cuda tensor); the single-image state of this object is untouched.
        """
        self._slic_model._unsupported()
        require_cuda()
        K = self._slic_model.num_components
        is_tensor = isinstance(images, torch.Tensor)
        B, H, W = int(images.shape[0]), int(images.shape[1]), int(images.shape[2])
        if images.shape[3] != 3:
            raise ValueError("nchan != 3")
        device = images.device.index if is_tensor else self._slic_model.device
        params = Engine.params(self.compactness, self.min_size_factor, self.subsample_stride, self.convert_to_lab,
                               max_iter)
        if not is_tensor:
            images = np.ascontiguousarray(images)
            if images.dtype != np.uint8:
                raise ValueError("images must be uint8")
        m = self._slic_model
        with _locked(lambda: get_engine(H, W, K, B, device)) as eng, _spatial_metric(eng, m.manhattan_spatial_dist):
            if m.real_dist or m.preemptive:
                # the float-distance contexts and `preemptive` have device entry points only: host batches go up and down here
                with torch.cuda.device(eng.device):
                    d_img = images if is_tensor else torch.from_numpy(images).to(eng.device)
                    if clusters is None:
                        d_cl = eng.initialize_clusters(d_img)
                    elif is_tensor:
                        d_cl = clusters
                    else:
                        d_cl = torch.from_numpy(np.ascontiguousarray(clusters).view(np.uint8).reshape(B, K, 32).copy()).to(eng.device)
                    if m.preemptive:
                        d_lab = eng.iterate_preemptive(d_img, d_cl, params, m.preemptive_thres)
                    else:
                        d_lab = eng.iterate_real(m.real_dist_type, d_img, d_cl, params)
                    if is_tensor:
                        labels, clusters = d_lab, d_cl
                    else:
                        labels = d_lab.cpu().numpy()
                        clusters = d_cl.cpu().numpy().view(CLUSTER_DTYPE).reshape(B, K)
            elif is_tensor:
                if clusters is None:
                    clusters = eng.initialize_clusters(images)
                labels = eng.iterate(images, clusters, params)
            else:
                if clusters is None:
                    clusters = eng.initialize_clusters_host(images)
                labels = eng.iterate_host(images, clusters, params)
        return (labels, clusters) if return_clusters else labels


class Slic(BaseSlic):
    """Drop-in for fast_slic.Slic / fast_slic.avx2.SlicAvx2 (identical results; base_slic.py:61-62, avx2.py:10-11)."""
    arch_name = ARCH_NAME


SlicCuda = Slic


class SlicRealDist(BaseSlic):
    """== fast_slic.base_slic.SlicRealDist (base_slic.py:64-72): float distances, float spatial term."""
    arch_name = ARCH_NAME
    real_dist_type = "standard"

    def make_slic_model(self, num_components):
        model = SlicModel(num_components, self.arch_name)
        model.real_dist = True
        model.real_dist_type = self.real_dist_type
        return model


class SlicRealDistL2(SlicRealDist):
    """== fast_slic.base_slic.SlicRealDistL2 (base_slic.py:74-76)."""
    real_dist_type = "l2"


class SlicRealDistNoQ(SlicRealDist):
    """== fast_slic.base_slic.SlicRealDistNoQ (base_slic.py:78-85): float centroids, no quantisation."""
    real_dist_type = "noq"

    def __init__(self, *args, **kwargs):
        float_color = kwargs.pop("float_color", True)
        super(SlicRealDistNoQ, self).__init__(*args, **kwargs)
        self._slic_model.float_color = float_color


class LSC(SlicRealDist):
    """== fast_slic.base_slic.LSC (base_slic.py:87-89), kept so that `from fast_slic import LSC` keeps importing: linear
    spectral clustering is a different algorithm (src/lsc.cpp) outside this engine -- iterate() raises NotImplementedError."""
    real_dist_type = "lsc"


def enforce_connectivity(assignments, min_threshold, device=0):
    """== cfast_slic.enforce_connectivity (cfast_slic.pyx:371-396): int16[H,W] in place, K = max label + 1
    (cfast_slic.pyx:377-382: the maximum over labels != -1).  K only bounds the number of kept components
    (cca.cpp:176,225), so it may exceed H*W; the context is keyed on the shape alone."""
    if not isinstance(assignments, np.ndarray) or assignments.dtype != np.int16 or assignments.ndim != 2 \
            or not assignments.flags["C_CONTIGUOUS"]:
        raise ValueError("assignments must be a C-contiguous int16[H, W] array")
    require_cuda()
    H, W = assignments.shape
    if H == 0 or W == 0:
        return assignments
    lab = assignments.view(np.uint16)
    valid = lab[lab != 0xFFFF]
    K = (int(valid.max()) if valid.size else 0) + 1
    with _locked(lambda: get_cca_engine(H, W, 1, device)) as eng:
        t = torch.from_numpy(assignments).to(eng.device, non_blocking=False)[None].contiguous()
        eng.enforce_connectivity(t, K, int(min_threshold))
        assignments[...] = t[0].cpu().numpy()
    return assignments
