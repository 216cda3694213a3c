"""The Euclidean spatial metric (`manhattan_spatial_dist=False`) on the CPU: the restatement's hypotf, its answers against
the compiled reference's recorded digests for every call the GPU tests make, and that the option changes the answer."""
import ctypes
import ctypes.util

import numpy as np
import pytest
import torch

import spatial_metric_common as smc


@pytest.fixture(scope="module")
def answers():
    yield smc.answers()
    smc.finish()


def test_double_sqrt_equals_libm_hypotf_on_the_integer_grid():
    """float(sqrt(double(a)^2 + double(b)^2)) == libm hypotf(a, b) for 0 <= a, b <= 4096 (S never comes close)."""
    libm = ctypes.CDLL(ctypes.util.find_library("m"))
    libm.hypotf.restype = ctypes.c_float
    libm.hypotf.argtypes = [ctypes.c_float, ctypes.c_float]
    a = np.arange(4097, dtype=np.float64)
    mine = np.sqrt(a[:, None] ** 2 + a[None, :] ** 2).astype(np.float32)
    rows = np.empty_like(mine)
    for i in range(4097):
        fi = float(i)
        rows[i] = [libm.hypotf(fi, float(j)) for j in range(4097)]
    bad = np.argwhere(rows != mine)
    assert bad.size == 0, "hypotf differs at %d points, first %s" % (len(bad), bad[:4].tolist())


def test_restatement_hypotf_and_patch():
    from oracle.metric import MetricPort
    p = MetricPort()
    for a, b in [(0, 0), (3, 4), (1, 1), (4096, 4095), (-7, 24)]:
        assert p.hypotf(a, b) == np.float32(np.sqrt(float(a) ** 2 + float(b) ** 2))
    S, compactness = 12, 10.0
    coef = np.float32(1.0) / (np.float32(S) / np.float32(compactness)) * np.float32(2)
    d = np.arange(-S, S + 1)
    h = np.sqrt(d[:, None].astype(np.float64) ** 2 + d[None, :] ** 2).astype(np.float32)
    want = (coef * h).astype(np.float32).astype(np.uint16)
    assert (p.spatial_patch(S, compactness, 1) == want).all()


def test_every_gpu_reference_call_matches_the_recorded_reference(answers):
    smc.all_reference_calls(answers)


def _differs(a, b):
    return any(not np.array_equal(x, y) for x, y in zip(a, b))


# where the two metrics cannot disagree: one-pixel-wide images (|di| or |dj| is 0, so hypot(di, dj) = |di| + |dj|), a
# spatial term that rounds to nothing (compactness 0.01) and a 5 x 7 image with three clusters
SAME_BY_CONSTRUCTION = ("edge_tiny_5x7_K3", "edge_row_1x200_K7", "edge_col_200x1_K7", "edge_compact0.01")


@pytest.mark.parametrize("case", [c for c in smc.INT_CASES + smc.PREEMPT_CASES if c[0] not in SAME_BY_CONSTRUCTION],
                         ids=lambda c: c[0])
def test_euclidean_changes_the_answer(answers, case):
    """The option bites: cold-start labels (pre-CCA, final) or clusters differ from the Manhattan answer."""
    from oracle.metric import MetricPort
    img, K, args = smc.case_image(case)
    kind = "preempt" if case in smc.PREEMPT_CASES else "int"
    eu = answers.run(img, K, args, manhattan=False, kind=kind, warm=False)[0]
    port = MetricPort()
    cl = port.initialize(img, K)
    out, pre = port.iterate(img, cl, args["max_iter"], args["compactness"], args["min_size_factor"], args["subsample_stride"],
                            args["convert_to_lab"], preemptive=(kind == "preempt"), manhattan=True)
    assert _differs(eu[1:], (out, pre, cl)), case[0] + ": the Euclidean answer equals the Manhattan one"


@pytest.mark.parametrize("case", smc.REAL_CASES, ids=lambda c: c[0])
def test_euclidean_real_variants(answers, case):
    """SlicRealDist and SlicRealDistNoQ change with the metric; SlicRealDistL2 ignores it (context.cpp:435-445)."""
    from oracle.metric import MetricPort
    img, K, args = smc.case_image(case)
    port = MetricPort()
    for v in (0, 1, 2):
        eu = answers.run(img, K, args, manhattan=False, kind="real", variant=v, warm=False)[0]
        cl = port.initialize(img, K)
        out, pre = port.iterate_real(v, img, cl, args["max_iter"], args["compactness"], args["min_size_factor"],
                                     args["subsample_stride"], args["convert_to_lab"], manhattan=True)
        if v == 1:
            assert not _differs(eu[1:], (out, pre, cl)), "%s: SlicRealDistL2 depends on the metric" % case[0]
        else:
            assert _differs(eu[1:], (out, pre, cl)), "%s variant %d: the Euclidean answer equals the Manhattan one" % (case[0], v)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without a GPU")
def test_euclidean_is_accepted_without_a_gpu():
    """manhattan_spatial_dist=False is a supported option: without a GPU it fails like every other call, not with
    NotImplementedError."""
    from fast_slic_b200 import Slic, SlicRealDistNoQ
    img = np.zeros((32, 32, 3), np.uint8)
    for cls in (Slic, SlicRealDistNoQ):
        with pytest.raises(RuntimeError, match="CUDA"):
            cls(num_components=4, manhattan_spatial_dist=False).iterate(img)
