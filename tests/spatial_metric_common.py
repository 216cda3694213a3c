"""Inputs and reference answers of the spatial-metric tests (`manhattan_spatial_dist`), shared by the CPU and GPU files.

`MetricAnswers` follows the scheme of conftest.ReferenceAnswers with a table of its own,
tests/golden/reference_digests_euclidean.json: SHA-256 digests of the compiled reference's outputs keyed by a digest of
each call's inputs.  Every call runs the plain-C restatement (oracle.metric.MetricPort), asserts that its outputs have
the digest the reference produced, and returns them.  With FSLIC_RECORD_REFERENCE_EUCLIDEAN=<file> set (and the
reference built into oracle/_ref), calls run the compiled reference instead and the session writes the extended table
to <file>.  The CPU file makes every call the GPU file makes, so the whole table can be recorded without a GPU.
"""
import json
import os

import numpy as np

from cases import make_image, split_kwargs
from conftest import ROOT, _digest, _usable_cores

TABLE = os.path.join(ROOT, "tests", "golden", "reference_digests_euclidean.json")
RECORD_ENV = "FSLIC_RECORD_REFERENCE_EUCLIDEAN"

# name, kind, H, W, K, kwargs, path: "tma" / "ldg" (W % 8 != 0) / "ldg_forced" (FSLIC_ASSIGN=4) / "generic" (S > 110) / "any"
INT_CASES = [
    ("tma_123x200_K60_msf0", "syn", 123, 200, 60, dict(min_size_factor=0.0), "tma"),
    ("tma_S16_256x256_K256", "noise", 256, 256, 256, dict(min_size_factor=0.0), "tma"),
    ("tma_S5_96x104_K350", "syn", 96, 104, 350, dict(min_size_factor=0.0), "tma"),  # list overflow: brute-force fallback
    ("tma_blocks_200x328_K150", "blocks", 200, 328, 150, dict(min_size_factor=0.0), "tma"),
    ("ldg_97x131_K37", "syn", 97, 131, 37, dict(min_size_factor=0.1), "ldg"),
    ("ldg_w33_70x33_K9", "syn", 70, 33, 9, {}, "ldg"),
    ("ldg_forced_120x160_K48", "noise", 120, 160, 48, dict(min_size_factor=0.25), "ldg_forced"),
    ("generic_300x400_K2", "syn", 300, 400, 2, {}, "generic"),
    ("edge_tiny_5x7_K3", "noise", 5, 7, 3, {}, "any"),
    ("edge_row_1x200_K7", "syn", 1, 200, 7, {}, "any"),
    ("edge_col_200x1_K7", "syn", 200, 1, 7, {}, "any"),
    ("edge_S1_20x20_K300", "noise", 20, 20, 300, dict(min_size_factor=0.0), "any"),
    ("edge_compact2000", "syn", 120, 160, 30, dict(compactness=2000.0), "any"),
    ("edge_compact0.01", "syn", 120, 160, 30, dict(compactness=0.01), "any"),
    ("stride1_it3", "syn", 90, 120, 20, dict(subsample_stride=1, max_iter=3), "any"),
    ("stride2_it1", "syn", 150, 200, 30, dict(subsample_stride=2, max_iter=1), "any"),
    ("stride5_it7", "syn", 150, 200, 60, dict(subsample_stride=5, max_iter=7), "any"),
    ("rgb_150x200_K300", "syn", 150, 200, 300, dict(convert_to_lab=False, min_size_factor=0.0), "any"),
]
# the float-distance variants: 0 SlicRealDist, 1 SlicRealDistL2, 2 SlicRealDistNoQ
REAL_CASES = [
    ("real_97x131_K37", "syn", 97, 131, 37, dict(min_size_factor=0.1), None),
    ("real_noise_120x160_K48", "noise", 120, 160, 48, dict(min_size_factor=0.0), None),
    ("real_rgb_150x200_K60", "syn", 150, 200, 60, dict(convert_to_lab=False), None),
]
PREEMPT_CASES = [
    ("preempt_180x240_K70", "syn", 180, 240, 70, dict(min_size_factor=0.1), None),
    ("preempt_noise_97x131_K37", "noise", 97, 131, 37, {}, None),
]
SEED = 17


def case_image(case):
    name, kind, H, W, K, kw, _ = case
    sigma, args = split_kwargs(kw)
    return make_image(kind, H, W, seed=SEED, sigma=sigma), K, args


# batched / streamed inputs of the GPU tests: (H, W, K, images)
def batch_inputs():
    H, W, K = 120, 160, 40
    return H, W, K, np.stack([make_image("syn" if b % 2 == 0 else "noise", H, W, seed=200 + b) for b in range(5)])


def blocking17_inputs():
    H, W, K = 96, 128, 30
    return H, W, K, np.stack([make_image("noise" if b % 3 == 0 else "syn", H, W, seed=500 + b) for b in range(17)])


def stream_inputs():
    """Three frames of two video streams: frames[t][b] is frame t of stream b."""
    H, W, K = 120, 160, 40
    base = [make_image("syn", H, W, seed=600 + b) for b in range(2)]
    frames = [np.stack([np.roll(base[b], 3 * t, axis=1) for b in range(2)]) for t in range(3)]
    return H, W, K, frames


def alternating_inputs():
    """Images of the test that alternates both metrics on one cached context (same shape, K and compactness)."""
    H, W, K = 120, 160, 40
    return H, W, K, [make_image("syn" if t % 2 else "noise", H, W, seed=700 + t) for t in range(4)]


class MetricAnswers:
    def __init__(self):
        from oracle.metric import MetricPort, MetricRef
        with open(TABLE) as f:
            self.table = json.load(f)
        self.record_to = os.environ.get(RECORD_ENV)
        if self.record_to:
            if not MetricRef.available():
                raise RuntimeError(RECORD_ENV + " needs the compiled reference (oracle/_ref)")
            self.impl = MetricRef()
            self.threads = min(8, _usable_cores())
        else:
            self.impl = MetricPort()

    def _pin(self, call, key_items, outputs):
        key, got = _digest(call, *key_items), _digest(*outputs)
        if self.record_to:
            assert self.table.setdefault(key, got) == got, "%s: the reference answers a recorded call differently" % call
            return
        assert key in self.table, "%s: no recorded reference answer for these inputs (record with %s)" % (call, RECORD_ENV)
        assert got == self.table[key], "%s: the restatement's outputs differ from the reference's" % call

    def write(self):
        with open(self.record_to, "w") as f:
            json.dump(self.table, f, indent=0, sort_keys=True)
            f.write("\n")

    def _kw(self):
        return dict(num_threads=self.threads) if self.record_to else {}

    def initialize(self, image, K):
        cl = self.impl.initialize(image, K)
        self._pin("initialize", (image, int(K)), [cl])
        return cl

    def iterate(self, image, clusters, args, manhattan, preemptive=False, preemptive_thres=0.05):
        """-> (labels, pre-CCA labels); clusters updated in place.  args: cases.split_kwargs()[1]."""
        a = (int(args["max_iter"]), float(args["compactness"]), float(args["min_size_factor"]), int(args["subsample_stride"]),
             bool(args["convert_to_lab"]))
        key = (image, clusters.copy()) + a + (bool(preemptive), float(preemptive_thres), bool(manhattan))
        out, pre = self.impl.iterate(image, clusters, *a, preemptive=preemptive, preemptive_thres=preemptive_thres,
                                     manhattan=manhattan, **self._kw())
        self._pin("iterate", key, [out, pre, clusters])
        return out, pre

    def iterate_real(self, variant, image, clusters, args, manhattan):
        a = (int(args["max_iter"]), float(args["compactness"]), float(args["min_size_factor"]), int(args["subsample_stride"]),
             bool(args["convert_to_lab"]))
        key = (int(variant), image, clusters.copy()) + a + (bool(manhattan),)
        out, pre = self.impl.iterate_real(variant, image, clusters, *a, manhattan=manhattan, **self._kw())
        self._pin("iterate_real", key, [out, pre, clusters])
        return out, pre

    def run(self, image, K, args, manhattan, kind="int", variant=None, warm=True):
        """Cold start (and, with warm, a second iterate from the clusters the first ended with), like calling
        Slic.iterate twice on one object.  -> [(init clusters, labels, pre-CCA labels, clusters) per iterate]."""
        cl = self.initialize(image, K)
        init = cl.copy()
        res = []
        for _ in range(2 if warm else 1):
            if kind == "real":
                out, pre = self.iterate_real(variant, image, cl, args, manhattan)
            else:
                out, pre = self.iterate(image, cl, args, manhattan, preemptive=(kind == "preempt"))
            res.append((init, out, pre, cl.copy()))
        return res


_answers = []


def answers():
    if not _answers:
        _answers.append(MetricAnswers())
    return _answers[0]


def finish():
    """Session end: write the table when recording."""
    if _answers and _answers[0].record_to:
        _answers[0].write()


def all_reference_calls(ans):
    """Every reference call the GPU tests make, in one place (the CPU test makes them all)."""
    out = {}
    for case in INT_CASES:
        img, K, args = case_image(case)
        out[case[0]] = ans.run(img, K, args, manhattan=False)
    for case in REAL_CASES:
        img, K, args = case_image(case)
        for v in (0, 1, 2):
            out[(case[0], v)] = ans.run(img, K, args, manhattan=False, kind="real", variant=v)
    for case in PREEMPT_CASES:
        img, K, args = case_image(case)
        out[case[0]] = ans.run(img, K, args, manhattan=False, kind="preempt")
    _, args = split_kwargs({})
    for name, inputs in (("batch", batch_inputs), ("blocking17", blocking17_inputs)):
        H, W, K, imgs = inputs()
        out[name] = [ans.run(imgs[b], K, args, manhattan=False, warm=False)[0] for b in range(len(imgs))]
    H, W, K, frames = stream_inputs()
    res = []
    for b in range(frames[0].shape[0]):
        cl = ans.initialize(frames[0][b], K)
        chain = []
        for t in range(len(frames)):
            o, p = ans.iterate(frames[t][b], cl, args, manhattan=False)
            chain.append((o, cl.copy()))
        res.append(chain)
    out["stream"] = res
    H, W, K, imgs = alternating_inputs()
    out["alternating"] = [ans.run(img, K, args, manhattan=(t % 2 == 0), warm=False)[0] for t, img in enumerate(imgs)]
    return out
