"""Streaming front end over host batches (no counterpart in the reference, whose iterate() blocks).

`SlicStream` keeps `depth` contexts (default 2) and alternates between them through
fslic_b200_iterate_host_async / fslic_b200_wait: while one batch runs its kernels, the next one is on the
PCIe wire going up and the previous one is coming down.  Results are identical to `Slic.iterate_batch`
on the same images (every batch is a cold start from the grid seeding, like a fresh `Slic`).

`warm_start=True` is the reference's video use (README.md:3; cfast_slic.pyx:160 keeps `_c_clusters` between calls):
image b of every batch is the next frame of stream b and starts from the clusters its previous frame ended with --
exactly what calling `slic.iterate(frame)` again on the same `Slic` object does.

`manhattan_spatial_dist=False` selects the Euclidean spatial term, like the keyword of `Slic`.  Frame t+1 of a stream depends on
the clusters of frame t, so in this mode a submit waits for the previous batch to finish (its clusters are the
input); the upload of the new frames is still prepared while the previous batch computes.
"""
import collections

import numpy as np
import torch

from .engine import CLUSTER_DTYPE, Engine, require_cuda


def _pinned(shape, dtype):
    return torch.empty(shape, dtype=dtype).pin_memory()


class _Slot:
    def __init__(self, H, W, K, batch, device):
        self.engine = Engine(H, W, K, batch, device)
        self.images = None  # pinned staging for images that arrive in pageable memory (allocated on demand)
        self.clusters = _pinned((batch, K, 32), torch.uint8)
        self.labels = _pinned((batch, H, W), torch.int16)
        self.n = 0


class SlicStream:
    def __init__(self, height, width, num_components, batch, depth=2, device=0, compactness=10.0,
                 min_size_factor=0.25, subsample_stride=3, convert_to_lab=True, max_iter=10, warm_start=False,
                 manhattan_spatial_dist=True):
        require_cuda()
        if depth < 1:
            raise ValueError("depth must be >= 1")
        self.H, self.W, self.K, self.batch = int(height), int(width), int(num_components), int(batch)
        self._slots = [_Slot(self.H, self.W, self.K, self.batch, device) for _ in range(depth)]
        self.manhattan_spatial_dist = bool(manhattan_spatial_dist)
        for s in self._slots:  # the slots' contexts are this stream's own: the metric is set once
            s.engine.set_manhattan_spatial_dist(self.manhattan_spatial_dist)
        self._params = self._slots[0].engine.params(compactness, min_size_factor, subsample_stride, convert_to_lab,
                                                    max_iter)
        self._free = collections.deque(self._slots)
        self._busy = collections.deque()
        self._finished = collections.deque()   # warm start: batches a later submit had to wait for, not collected yet
        self._pristine = None  # grid seeding: depends on (H, W, K) only; colours are re-read from the image in pass 0
        self.warm_start = bool(warm_start)
        self._carry = None     # warm start: the clusters the previous batch ended with, [n, K, 32] bytes

    def pinned_images(self, n=None):
        """A pinned uint8 [n,H,W,3] array to fill and pass to submit() without a staging copy."""
        return _pinned((self.batch if n is None else n, self.H, self.W, 3), torch.uint8).numpy()

    def submit(self, images):
        """Enqueue uint8 [n<=batch,H,W,3]; returns immediately.  Raises if `depth` batches are already in flight."""
        if not self._free:
            raise RuntimeError("all %d slots are in flight: collect() first" % len(self._slots))
        images = np.ascontiguousarray(images)
        if images.dtype != np.uint8 or images.ndim != 4 or images.shape[1:] != (self.H, self.W, 3):
            raise ValueError("images must be uint8 [n, %d, %d, 3]" % (self.H, self.W))
        n = images.shape[0]
        if n < 1 or n > self.batch:
            raise ValueError("1 <= n <= %d images per submit" % self.batch)
        slot = self._free.popleft()
        if self._pristine is None:
            self._pristine = slot.engine.initialize_clusters_host(images[:1]).view(np.uint8).reshape(self.K, 32).copy()
        if not torch.from_numpy(images).is_pinned():
            if slot.images is None:
                slot.images = _pinned((self.batch, self.H, self.W, 3), torch.uint8)
            staged = slot.images.numpy()[:n]
            staged[...] = images
            images = staged
        cl = slot.clusters.numpy()[:n]
        cl[...] = self._pristine
        if self.warm_start:
            # the previous batch's final clusters are this batch's start (stream b <-> image b); streams that join
            # later (a larger n than before) start from the grid seeding
            while self._busy:
                self._finished.append(self._collect_one(copy=True))
            if self._carry is not None:
                m = min(n, self._carry.shape[0])
                cl[:m] = self._carry[:m]
        slot.n = n
        slot.engine.iterate_host_async(images, cl, self._params, slot.labels.numpy()[:n])
        self._busy.append(slot)

    def _collect_one(self, copy):
        slot = self._busy.popleft()
        slot.engine.wait()
        self._free.append(slot)
        labels = slot.labels.numpy()[:slot.n]
        raw = slot.clusters.numpy()[:slot.n]
        if self.warm_start:
            self._carry = raw.copy()
        clusters = raw.view(CLUSTER_DTYPE).reshape(slot.n, self.K)
        return (labels.copy(), clusters.copy()) if copy else (labels, clusters)

    def collect(self, copy=True):
        """Labels int16 [n,H,W] and clusters [n,K] of the oldest batch in flight (blocks until it is done).
        With copy=False the arrays are views of the slot's pinned buffers, valid until the slot is submitted again."""
        if self._finished:
            return self._finished.popleft()
        if not self._busy:
            raise RuntimeError("nothing in flight")
        return self._collect_one(copy)

    @property
    def in_flight(self):
        return len(self._busy) + len(self._finished)

    def map(self, batches):
        """Generator: labels of every batch of `batches`, in order, keeping the pipeline full."""
        for images in batches:
            if not self._free:
                yield self.collect()[0]
            self.submit(images)
            while self._finished:
                yield self._finished.popleft()[0]
        while self._busy or self._finished:
            yield self.collect()[0]

    def close(self):
        while self._busy:
            self._collect_one(copy=False)
        self._finished.clear()
        for s in self._slots:
            s.engine.close()
