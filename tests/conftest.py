import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

REFERENCE_DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_digests.json")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def port():
    from oracle.oracle import Port
    return Port()


def _usable_cores():
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def _digest(*items):
    """SHA-256 over arrays (dtype, shape and bytes) and plain values, in order."""
    h = hashlib.sha256()
    for x in items:
        if isinstance(x, np.ndarray):
            x = np.ascontiguousarray(x)
            h.update(repr((x.dtype.str, x.shape)).encode())
            h.update(x.tobytes())
        else:
            h.update(repr(x).encode())
        h.update(b"\0")
    return h.hexdigest()


class ReferenceAnswers:
    """What the parity tests compare against: the answers of the original fast-slic (the unmodified reference,
    compiled by oracle/Makefile into oracle/_ref, SlicAvx2 path), kept in tests/golden/reference_digests.json as
    SHA-256 digests of its outputs keyed by a digest of each call's inputs.

    Every call runs the plain-C restatement (oracle.Port), asserts that its outputs have the digest the reference
    produced for the same inputs, and returns them, so the comparison with the original holds on machines that do not
    have it.  With FSLIC_RECORD_REFERENCE=<file> set (and oracle/_ref built), calls run the compiled reference instead
    and the session writes the table, extended by their digests, to <file>; a call the reference answers differently
    from an existing entry fails.  The reference's answer does not depend on its OpenMP thread count, so that is not
    part of a key."""

    def __init__(self):
        from oracle.oracle import Port, Ref
        with open(REFERENCE_DIGESTS) as f:
            self.table = json.load(f)
        self.record_to = os.environ.get("FSLIC_RECORD_REFERENCE")
        if self.record_to:
            if not Ref.available():
                raise RuntimeError("FSLIC_RECORD_REFERENCE needs the compiled reference (oracle/_ref)")
            self.ref = Ref()
            self.threads = min(8, _usable_cores())   # not "all cores": a CPU quota may be far below the core count
        else:
            self.port = Port()

    def _pin(self, call, key_items, outputs):
        key, got = _digest(call, *key_items), _digest(*outputs)
        if self.record_to:
            assert self.table.setdefault(key, got) == got, "%s: the reference answers a recorded call differently" % call
            return
        assert key in self.table, "%s: no recorded reference answer for these inputs (record with FSLIC_RECORD_REFERENCE)" % call
        assert got == self.table[key], "%s: the restatement's outputs differ from the reference's" % call

    def write(self):
        with open(self.record_to, "w") as f:
            json.dump(self.table, f, indent=0, sort_keys=True)
            f.write("\n")

    def _threads(self, num_threads):
        return self.threads if num_threads is None else num_threads

    def initialize(self, image, K):
        cl = (self.ref if self.record_to else self.port).initialize(image, K)
        self._pin("initialize", (image, int(K)), [cl])
        return cl

    def iterate(self, image, clusters, max_iter=10, compactness=10.0, min_size_factor=0.25, stride=3,
                convert_to_lab=True, stages=False, arch="x64/avx2", num_threads=None, preemptive=False,
                preemptive_thres=0.05):
        args = (int(max_iter), float(compactness), float(min_size_factor), int(stride), bool(convert_to_lab))
        key = (image, clusters.copy()) + args + (bool(stages), arch, bool(preemptive), float(preemptive_thres))
        if self.record_to:
            res = self.ref.iterate(image, clusters, *args, stages=stages, arch=arch, num_threads=self._threads(num_threads),
                                   preemptive=preemptive, preemptive_thres=preemptive_thres)
        else:
            res = self.port.iterate(image, clusters, *args, stages=stages, preemptive=preemptive,
                                    preemptive_thres=preemptive_thres)
        if stages:  # the reference's preemptive entry point has no Lab stage output
            out, quad, pre = res
            outputs = [out, pre] + ([] if preemptive else [quad])
        else:
            outputs = [res]
        self._pin("iterate", key, outputs + [clusters])
        return res

    def iterate_real(self, variant, image, clusters, max_iter=10, compactness=10.0, min_size_factor=0.25, stride=3,
                     convert_to_lab=True, stages=False, num_threads=None):
        args = (int(max_iter), float(compactness), float(min_size_factor), int(stride), bool(convert_to_lab))
        key = (int(variant), image, clusters.copy()) + args
        if self.record_to:
            out, pre = self.ref.iterate_real(variant, image, clusters, *args, stages=True,
                                             num_threads=self._threads(num_threads))
        else:
            out, pre = self.port.iterate_real(variant, image, clusters, *args, stages=True)
        self._pin("iterate_real", key, [out, pre, clusters])
        return (out, pre) if stages else out

    def enforce_connectivity(self, labels, K, thres, num_threads=None):
        if self.record_to:
            out = self.ref.enforce_connectivity(labels, K, thres, num_threads=self._threads(num_threads))
        else:
            out = self.port.enforce_connectivity(labels, K, thres)
        self._pin("enforce_connectivity", (labels, int(K), int(thres)), [out])
        return out

    def get_connectivity(self, labels, K):
        nb = (self.ref if self.record_to else self.port).get_connectivity(labels, K)
        self._pin("get_connectivity", (labels, int(K)), [nb])
        return nb

    def get_mask_density(self, clusters, labels, mask):
        dens = (self.ref if self.record_to else self.port).get_mask_density(clusters, labels, mask)
        self._pin("get_mask_density", (clusters, labels, mask), [dens])
        return dens

    def density_to_mask(self, K, labels, densities):
        out = (self.ref if self.record_to else self.port).density_to_mask(K, labels, densities)
        self._pin("density_to_mask", (int(K), labels, densities), [out])
        return out


_answers = []


@pytest.fixture(scope="session")
def ref():
    if not _answers:
        _answers.append(ReferenceAnswers())
    return _answers[0]


@pytest.fixture(scope="session")
def checker(ref):
    return ref


def pytest_sessionfinish(session, exitstatus):
    if _answers and _answers[0].record_to:
        _answers[0].write()
