"""CPU-only tests: the oracle against the golden vectors and the compiled reference's recorded answers (conftest.ref),
the C ABI surface, the host-side logic, and the world_size-2 sharding path over gloo."""
import ctypes
import hashlib
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from cases import EDGE_CASES, PIPELINE_CASES, make_image, split_kwargs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "golden_v1.npz")


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


GOLDEN_CASES = [c for c in PIPELINE_CASES if c[2] * c[3] <= 80000]


@pytest.mark.parametrize("case", GOLDEN_CASES, ids=[c[0] for c in GOLDEN_CASES])
def test_oracle_matches_golden(port, golden, case):
    """The plain-C restatement reproduces what the unmodified reference produced (tests/golden/make_golden.py)."""
    name, kind, H, W, K, kw = case
    sigma, a = split_kwargs(kw)
    img = make_image(kind, H, W, seed=7, sigma=sigma)
    cl = port.initialize(img, K)
    assert cl.tobytes() == golden[name + "/init"].tobytes()
    lab, quad, pre = port.iterate(img, cl, a["max_iter"], a["compactness"], a["min_size_factor"],
                                  a["subsample_stride"], a["convert_to_lab"], stages=True)
    assert (lab == golden[name + "/labels"]).all()
    assert cl.tobytes() == golden[name + "/clusters"].tobytes()
    assert hashlib.sha256(quad.tobytes()).digest() == golden[name + "/quad_sha"].tobytes()
    assert hashlib.sha256(pre.tobytes()).digest() == golden[name + "/pre_sha"].tobytes()


def test_oracle_cca_golden(port, golden):
    assert (port.enforce_connectivity(golden["cca5/in"], 10, 0) == golden["cca5/out"]).all()
    for t in range(4):
        thres, K = golden["cca_rand%d/thres" % t]
        got = port.enforce_connectivity(golden["cca_rand%d/in" % t], int(K), int(thres))
        assert (got == golden["cca_rand%d/out" % t]).all()


@pytest.mark.parametrize("case", PIPELINE_CASES[:12], ids=[c[0] for c in PIPELINE_CASES[:12]])
def test_oracle_matches_compiled_reference(port, ref, case):
    """Differential test against the compiled reference's answers (conftest.ReferenceAnswers)."""
    name, kind, H, W, K, kw = case
    sigma, a = split_kwargs(kw)
    img = make_image(kind, H, W, seed=13, sigma=sigma)
    c1, c2 = port.initialize(img, K), ref.initialize(img, K)
    assert c1.tobytes() == c2.tobytes()
    args = (a["max_iter"], a["compactness"], a["min_size_factor"], a["subsample_stride"], a["convert_to_lab"])
    o1, q1, p1 = port.iterate(img, c1, *args, stages=True)
    o2, q2, p2 = ref.iterate(img, c2, *args, stages=True, num_threads=2)
    assert (q1 == q2).all() and (p1 == p2).all() and (o1 == o2).all() and c1.tobytes() == c2.tobytes()


@pytest.mark.parametrize("case", EDGE_CASES, ids=[c[0] for c in EDGE_CASES])
def test_oracle_matches_compiled_reference_edge(port, ref, case):
    name, kind, H, W, K, kw = case
    sigma, a = split_kwargs(kw)
    img = make_image(kind, H, W, seed=5, sigma=sigma)
    c1, c2 = port.initialize(img, K), ref.initialize(img, K)
    args = (a["max_iter"], a["compactness"], a["min_size_factor"], a["subsample_stride"], a["convert_to_lab"])
    o1, o2 = port.iterate(img, c1, *args), ref.iterate(img, c2, *args, num_threads=2)
    assert (o1 == o2).all() and c1.tobytes() == c2.tobytes()


def test_oracle_initialize_above_2p24_pixels(port):
    """context.cpp:88 indexes the image with a FLOAT expression (one fused multiply-add under the reference's build
    flags); above 2^24 pixels it lands on a neighbouring pixel for some centres.  Known answer = SHA-256 of the
    compiled reference's Cluster bytes for this seeded 4100x4200 image (found by the round-2 GPU run: the restatement
    used exact integer indexing until then)."""
    img = make_image("tiled", 4100, 4200, seed=11, sigma=20.0)
    cl = port.initialize(img, 3000)
    assert hashlib.sha256(cl.tobytes()).hexdigest() == "f344f4422d2aae58b78e3c8f096b7bb1969c8289666fb817d5a5e59a07c71b3b"
    exact = np.array([img[int(c["y"]), int(c["x"])] for c in cl], np.float32)
    assert (np.stack([cl["r"], cl["g"], cl["b"]], 1) != exact).any(), "the case must exercise the inexact index"


def test_oracle_initialize_above_2p24_pixels_live(port, ref):
    img = make_image("tiled", 4100, 4200, seed=11, sigma=20.0)
    assert port.initialize(img, 3000).tobytes() == ref.initialize(img, 3000).tobytes()


@pytest.mark.parametrize("H,W,K,kind,msf", [(120, 160, 48, "syn", 0.25), (97, 131, 37, "noise", 0.0), (200, 300, 150, "blocks", 0.0),
                                            (64, 64, 1500, "noise", 0.0), (180, 240, 70, "syn", 0.1)])
def test_oracle_graph_and_density_match_compiled_reference(port, ref, H, W, K, kind, msf):
    """fast-slic.cpp:16-78, 141-168 (adjacency graph with its 12-neighbour cap, mask density, density broadcast):
    restatement == compiled reference.  (knn_connectivity, :80-130, overflows its cell vector -- see slic_oracle.c.)"""
    img = make_image(kind, H, W, seed=17)
    cl = ref.initialize(img, K)
    lab = ref.iterate(img, cl, 10, 10.0, msf, 3, True, num_threads=2)
    assert port.get_connectivity(lab, K) == ref.get_connectivity(lab, K)
    # saturated nodes (more than 12 distinct neighbours).  Labels >= K are left out: the reference reads
    # num_neighbors[source] before its range check (fast-slic.cpp:34-35), out of bounds for the 0xFFFF sentinel
    raw = (make_image("noise", H, W, seed=3)[..., 0].astype(np.uint16) % min(K, 40)).astype(np.uint16)
    assert port.get_connectivity(raw, K) == ref.get_connectivity(raw, K)
    mask = make_image("syn", H, W, seed=5)[..., 1]
    d1, d2 = port.get_mask_density(cl, lab, mask), ref.get_mask_density(cl, lab, mask)
    assert (d1 == d2).all()
    assert (port.density_to_mask(K, lab, d1) == ref.density_to_mask(K, lab, d1)).all()
    big = raw.copy()
    big[::7, ::5] = 0xFFFF
    assert (port.density_to_mask(K, big, d1) == ref.density_to_mask(K, big, d1)).all()
    assert (port.get_mask_density(cl, big, mask) == ref.get_mask_density(cl, big, mask)).all()


@pytest.mark.parametrize("seed", range(10))
def test_oracle_matches_compiled_reference_random_configs(port, ref, seed):
    """Seeded random shapes / K / parameters: the restatement against the compiled reference, all stages."""
    rng = np.random.RandomState(1000 + seed)
    H, W = int(rng.randint(20, 160)), int(rng.randint(20, 200))
    K = int(rng.randint(1, max(2, H * W // 40)))
    kind = ["syn", "noise", "blocks"][seed % 3]
    args = (int(rng.randint(0, 13)), float(rng.choice([0.5, 3.0, 10.0, 40.0])), float(rng.choice([0.0, 0.1, 0.25, 1.0])),
            int(rng.randint(1, 6)), bool(rng.randint(0, 2)))
    img = make_image(kind, H, W, seed=seed, sigma=float(rng.choice([5.0, 12.0, 30.0])))
    c1, c2 = port.initialize(img, K), ref.initialize(img, K)
    assert c1.tobytes() == c2.tobytes()
    o1, q1, p1 = port.iterate(img, c1, *args, stages=True)
    o2, q2, p2 = ref.iterate(img, c2, *args, stages=True, num_threads=2)
    assert (q1 == q2).all() and (p1 == p2).all() and (o1 == o2).all() and c1.tobytes() == c2.tobytes(), (H, W, K, args)


def test_reference_thread_and_arch_invariance(ref):
    img = make_image("syn", 120, 160, seed=3)
    outs = []
    for arch, nt in (("standard", 1), ("x64/avx2", 1), ("x64/avx2", 3)):
        cl = ref.initialize(img, 40)
        outs.append((ref.iterate(img, cl, 10, 10.0, 0.1, 3, True, arch=arch, num_threads=nt).tobytes(), cl.tobytes()))
    assert outs[0] == outs[1] == outs[2]


def test_lab_known_answers(port):
    """Known answers measured from the reference (SURVEY.md section 8c); the reference's own gtest triples
    (src/cpptest/test_cielab.cpp:5-37) are for an older un-doubled scale and no longer hold for its own code."""
    px = np.array([[[139, 91, 30], [255, 255, 255], [255, 255, 0], [0, 0, 0]]], np.uint8)
    q = port.rgb_to_quad(px, True)[0]
    assert q[:, :3].tolist() == [[85, 156, 210], [200, 128, 128], [194, 84, 255], [0, 128, 128]]
    assert (q[:, 3] == 0).all()
    gamma, lab, cb = port.lab_tables()
    assert hashlib.sha256(lab.astype("<i4").tobytes()).hexdigest() == \
        "ee38090c38e046060ca5987d76d797bbf2c71e6519c88e9718dd30e8119c8c56"
    assert cb.tolist() == [28440, 24656, 12442, 13938, 46868, 4730, 1164, 7175, 57202]
    assert gamma[0] == 0 and gamma[255] == 8192 and lab.max() == 8192


@pytest.mark.parametrize("n,middle,maxarea", [(40, 7, 3), (500, 100, 4), (3000, 1600, 6), (5000, 30, 2), (64, 64, 3)])
def test_heap_select_port_vs_libstdcxx(port, n, middle, maxarea):
    """The hand-restated __heap_select against the real std::partial_sort on tie-saturated inputs."""
    for seed in range(6):
        rng = np.random.RandomState(seed * 1000 + n)
        area = rng.randint(1, maxarea + 1, n).astype(np.int32)
        assert (port.heap_select(area, middle) == port.stl_partial_sort(area, middle)).all()


def test_spatial_lut_matches_patch(port):
    lut = port.spatial_lut(24, 10.0, 1)
    coef = np.float32(1.0) / (np.float32(24) / np.float32(10.0)) * np.float32(2)
    want = (coef * np.arange(49, dtype=np.float32)).astype(np.uint16)
    assert (lut == want).all()


# ---- the C ABI ------------------------------------------------------------------------------------------
def test_abi_library_exports_every_declared_symbol():
    from fast_slic_b200 import _lib
    L = _lib.lib()  # loads without a GPU
    header = open(os.path.join(ROOT, "include", "fslic_b200.h")).read()
    declared = set(re.findall(r"\b(fslic_b200_\w+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    for sym in declared:
        assert hasattr(L, sym), sym
    assert L.fslic_b200_sizeof_cluster() == 32
    assert L.fslic_b200_version().startswith(b"fast_slic_b200")


def test_abi_is_sm100a_only():
    out = subprocess.run(["cuobjdump", "--list-elf", os.path.join(ROOT, "fast_slic_b200", "libfslic_b200.so")],
                         capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_cluster_struct_layout():
    from fast_slic_b200 import CLUSTER_DTYPE
    offs = {n: CLUSTER_DTYPE.fields[n][1] for n in CLUSTER_DTYPE.names}
    # == /root/reference/src/fast-slic-common.h:10-23
    assert offs == {"y": 0, "x": 4, "r": 8, "g": 12, "b": 16, "a": 20, "number": 24, "is_active": 26,
                    "is_updatable": 27, "num_members": 28}
    assert CLUSTER_DTYPE.itemsize == 32


# ---- host logic (mirrors cfast_slic.pyx error behaviour; no GPU needed) -----------------------------------
def test_slic_model_argument_errors():
    from fast_slic_b200 import Slic, SlicModel, get_supported_archs, is_supported_arch, supported_archs
    assert supported_archs == ("cuda/sm_100a",) and get_supported_archs() == ["cuda/sm_100a"]
    assert is_supported_arch("cuda/sm_100a") and not is_supported_arch("x64/avx2")
    with pytest.raises(ValueError):
        SlicModel(0)
    with pytest.raises(ValueError):
        SlicModel(65534)
    with pytest.raises(NotImplementedError):
        SlicModel(10, "arm/neon")
    m = SlicModel(10)
    with pytest.raises(RuntimeError, match="not initialized"):
        m.iterate(np.zeros((8, 8, 3), np.uint8), 10, 10.0, 0.25, 3)
    m.initialized = True
    with pytest.raises(ValueError, match="nchan != 3"):
        m.iterate(np.zeros((8, 8, 4), np.uint8), 10, 10.0, 0.25, 3)
    with pytest.raises(ValueError):
        m.iterate(np.zeros((8, 8, 3), np.float32), 10, 10.0, 0.25, 3)
    with pytest.raises(ValueError):
        m.iterate(np.zeros((8, 16, 3), np.uint8)[:, ::2], 10, 10.0, 0.25, 3)
    s = Slic(num_components=77, compactness=5, min_size_factor=0.1, convert_to_lab=False)
    assert s.num_components == 77 and s.convert_to_lab is False and s.last_assignment is None
    assert s.slic_model.preemptive is False and s.slic_model.manhattan_spatial_dist is True


def test_clusters_roundtrip_and_copy():
    from fast_slic_b200 import SlicModel
    m = SlicModel(5)
    with pytest.raises(OverflowError):  # Cython range-checks object -> uint8_t
        m.clusters = [dict(number=0, yx=(1, 1), color=(300.0, 2.0, 1.0), num_members=4)]
    cl = [dict(number=9, yx=(3.7, 4.2), color=(200.9, 2.0, 1.0), num_members=4) for _ in range(3)]
    m.clusters = cl
    assert m.num_components == 3 and m.initialized
    got = m.clusters
    assert [c["number"] for c in got] == [0, 1, 2]          # number = index (cfast_slic.pyx:80)
    assert got[0]["yx"] == (3.0, 4.0)                          # uint16 truncation (cfast_slic.pyx:69)
    assert got[0]["color"] == (200.0, 2.0, 1.0)                # uint8 truncation (cfast_slic.pyx:70)
    c2 = m.copy()
    assert c2.clusters == got and c2.initialized
    c2._clusters["y"][0] = 1
    assert m.clusters[0]["yx"] == (3.0, 4.0)


def test_product_never_imports_the_oracle():
    for fn in os.listdir(os.path.join(ROOT, "fast_slic_b200")):
        if fn.endswith(".py"):
            assert "oracle" not in open(os.path.join(ROOT, "fast_slic_b200", fn)).read(), fn


def test_requires_cuda_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from fast_slic_b200 import Slic
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Slic(num_components=10).iterate(np.zeros((16, 16, 3), np.uint8))


# ---- sharding over gloo, world_size 2 ---------------------------------------------------------------------
def test_shard_range_partitions():
    from fast_slic_b200.sharding import shard_range
    for n in (0, 1, 7, 8, 256, 257):
        for world in (1, 2, 3, 8):
            r = [shard_range(n, k, world) for k in range(world)]
            assert r[0][0] == 0 and r[-1][1] == n
            assert all(r[k][1] == r[k + 1][0] for k in range(world - 1))
            sizes = [e - s for s, e in r]
            assert max(sizes) - min(sizes) <= 1


_GLOO_SCRIPT = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from fast_slic_b200.sharding import shard_range, gather_labels
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
n_total, H, W = 5, 6, 7
full = (torch.arange(n_total * H * W, dtype=torch.int32).reshape(n_total, H, W) % 3000).to(torch.int16)
s, e = shard_range(n_total, rank, world)
out = gather_labels(full[s:e].clone(), n_total)
assert out.shape == full.shape and torch.equal(out, full), rank
t = torch.tensor([float(rank + 1)], dtype=torch.float64)
dist.all_reduce(t, op=dist.ReduceOp.MAX)      # the max-over-ranks timing reduction bench.py uses
assert t.item() == world
dist.barrier()
print("rank", rank, "ok")
"""


def test_gloo_world_size_2_gather(tmp_path):
    script = tmp_path / "gloo_gather.py"
    script.write_text(_GLOO_SCRIPT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29731", str(script), ROOT],
                       capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("ok") == 2


def _build_cython_stub(tmp_path):
    pytest.importorskip("Cython")
    if not os.path.exists(os.path.join(ROOT, "fast_slic_b200", "libfslic_b200.so")):
        pytest.skip("libfslic_b200.so not built")
    subprocess.check_call(["bash", os.path.join(ROOT, "integration", "build_stub.sh"), str(tmp_path)],
                          stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    sys.path.insert(0, str(tmp_path))
    try:
        import importlib
        return importlib.import_module("cfast_slic_b200")
    finally:
        sys.path.pop(0)


def test_cython_stub_builds_and_binds(tmp_path):
    """INTEGRATION.md section 2 for real: the Cython branch a maintainer of the reference would add compiles against
    include/fslic_b200.h, links libfslic_b200.so, keeps the reference's signatures / exception types, and -- on this
    GPU-less box -- fails loudly instead of falling back to anything."""
    m = _build_cython_stub(tmp_path)
    assert m.sizeof_cluster() == 32
    with pytest.raises(ValueError):
        m.SlicModelCuda(70000)
    model = m.SlicModelCuda(50)
    with pytest.raises(RuntimeError):                       # cfast_slic.pyx:151
        model.iterate(np.zeros((48, 64, 3), np.uint8), 10, 10.0, 0.25, 3)
    with pytest.raises(ValueError):                         # cfast_slic.pyx:125
        model.initialize(np.zeros((48, 64, 4), np.uint8))
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            model.initialize(np.zeros((48, 64, 3), np.uint8))


@pytest.mark.parametrize("variant", [0, 1, 2])
def test_oracle_real_dist_variants_match_compiled_reference(port, ref, variant):
    """ContextRealDist / ContextRealDistL2 / ContextRealDistNoQ (context.cpp:394-499): the restatement's float
    arithmetic (one multiply + one add; fma(dj, dj, di*di); left-to-right |.| sums and float quotients) reproduces the
    compiled reference bit for bit -- pre-CCA labels, final labels, Cluster bytes."""
    for kind, H, W, K, kw in [("syn", 120, 160, 48, {}), ("noise", 97, 131, 37, dict(min_size_factor=0.0)),
                              ("syn", 240, 320, 150, dict(compactness=30.0)), ("blocks", 200, 300, 150, {}),
                              ("syn", 150, 200, 30, dict(subsample_stride=2, max_iter=3)), ("flat", 97, 131, 37, {}),
                              ("syn", 180, 240, 70, dict(convert_to_lab=False))]:
        sigma, a = split_kwargs(kw)
        img = make_image(kind, H, W, seed=31, sigma=sigma)
        c1, c2 = port.initialize(img, K), ref.initialize(img, K)
        args = (a["max_iter"], a["compactness"], a["min_size_factor"], a["subsample_stride"], a["convert_to_lab"])
        o1, p1 = port.iterate_real(variant, img, c1, *args, stages=True)
        o2, p2 = ref.iterate_real(variant, img, c2, *args, stages=True)
        assert (p1 == p2).all() and (o1 == o2).all() and c1.tobytes() == c2.tobytes(), (variant, kind, H, W, K)


def test_oracle_preemptive_matches_compiled_reference(port, ref):
    """PreemptiveGrid (preemptive.h) + the branches of assign / update that consult it (context.cpp:218, 307-385): the
    restatement reproduces the compiled reference with preemptive = true -- pre-CCA labels, final labels, Cluster bytes
    (is_updatable countdown included), both arch contexts -- and the option changes the result."""
    for kind, H, W, K, thres, kw in [("syn", 120, 160, 48, 0.05, {}), ("syn", 200, 300, 150, 0.05, {}),
                                     ("syn", 240, 320, 200, 0.2, dict(max_iter=15)),
                                     ("syn", 181, 257, 90, 0.1, dict(subsample_stride=1, max_iter=6)),
                                     ("blocks", 240, 320, 64, 0.5, dict(subsample_stride=2)),
                                     ("syn", 300, 400, 300, 0.02, dict(sigma=4.0))]:
        sigma, a = split_kwargs(kw)
        img = make_image(kind, H, W, seed=43, sigma=sigma)
        args = (a["max_iter"], a["compactness"], a["min_size_factor"], a["subsample_stride"], a["convert_to_lab"])
        plain = ref.iterate(img, ref.initialize(img, K), *args)
        for arch in ("x64/avx2", "standard"):
            c1, c2 = port.initialize(img, K), ref.initialize(img, K)
            for round_ in range(2):  # cold start, then warm start on the records the first call left
                o1, _, p1 = port.iterate(img, c1, *args, stages=True, preemptive=True, preemptive_thres=thres)
                o2, _, p2 = ref.iterate(img, c2, *args, stages=True, arch=arch, num_threads=2, preemptive=True,
                                        preemptive_thres=thres)
                assert (p1 == p2).all() and (o1 == o2).all() and c1.tobytes() == c2.tobytes(), (kind, H, W, K, thres, arch, round_)
                if round_ == 0:
                    assert (o2 != plain).any(), "the case does not exercise the option"


def test_import_compatibility_classes():
    """`from fast_slic import LSC` / `from fast_slic.avx2 import SlicAvx2, LSCAvx2` (fast_slic/base_slic.py:87-89,
    fast_slic/avx2.py:10-14) keep importing from this package; LSC is outside the engine and says so at iterate()."""
    import fast_slic_b200 as fs
    from fast_slic_b200.avx2 import LSCAvx2, SlicAvx2
    assert issubclass(SlicAvx2, fs.Slic) and issubclass(LSCAvx2, fs.LSC) and issubclass(fs.LSC, fs.SlicRealDist)
    assert SlicAvx2(num_components=7).slic_model.num_components == 7
    for cls in (fs.LSC, LSCAvx2):
        with pytest.raises(NotImplementedError):
            cls(num_components=5).iterate(np.zeros((8, 8, 3), np.uint8))


def test_slic_model_to_yxmrgb():
    """cfast_slic.pyx:100-113: float64 [K, 6] = (y, x, num_members, r, g, b) per cluster."""
    import fast_slic_b200 as fs
    m = fs.SlicModel(3)
    m._clusters["y"], m._clusters["x"], m._clusters["num_members"] = [1, 2, 3], [4, 5, 6], [7, 8, 9]
    m._clusters["r"], m._clusters["g"], m._clusters["b"] = [10, 11, 12], [13, 14, 15], [16, 17, 18]
    out = m.to_yxmrgb()
    assert out.dtype == np.float64 and out.shape == (3, 6)
    assert out.tolist() == [[1, 4, 7, 10, 13, 16], [2, 5, 8, 11, 14, 17], [3, 6, 9, 12, 15, 18]]
