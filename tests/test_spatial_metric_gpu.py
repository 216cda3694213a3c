"""GPU parity of the Euclidean spatial metric (`manhattan_spatial_dist=False`) against the reference, bit-exact: labels
before and after connectivity enforcement and the raw Cluster records, cold and warm start, on every path."""
import numpy as np
import pytest
import torch

import spatial_metric_common as smc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def want():
    yield smc.all_reference_calls(smc.answers())
    smc.finish()


def _engine(H, W, K, B=1):
    from fast_slic_b200 import get_engine
    return get_engine(H, W, K, B, 0)


def _run_engine(img, K, args, variant=None, preempt=False):
    """Cold and warm start through the device entry points of one cached context, Euclidean for the call only."""
    H, W, _ = img.shape
    eng = _engine(H, W, K)
    with eng.lock:
        eng.set_manhattan_spatial_dist(False)
        try:
            t = torch.from_numpy(img).cuda()[None].contiguous()
            cl = eng.initialize_clusters(t)
            init = cl[0].cpu().numpy().copy()
            p = eng.params(args["compactness"], args["min_size_factor"], args["subsample_stride"], args["convert_to_lab"],
                           args["max_iter"])
            res = []
            for _ in range(2):
                if variant is not None:
                    lab = eng.iterate_real(("standard", "l2", "noq")[variant], t, cl, p)
                elif preempt:
                    lab = eng.iterate_preemptive(t, cl, p, 0.05)
                else:
                    lab = eng.iterate(t, cl, p)
                _, pre = eng.debug_stages(1)
                torch.cuda.synchronize()
                res.append((init, lab[0].cpu().numpy().view(np.uint16), pre[0].cpu().numpy().view(np.uint16),
                            cl[0].cpu().numpy().copy()))
        finally:
            eng.set_manhattan_spatial_dist(True)
    return eng, res


def _compare(name, got, want):
    for n, (g, w) in enumerate(zip(got, want)):
        tag = "%s (%s start)" % (name, "warm" if n else "cold")
        ginit, glab, gpre, gcl = g
        winit, wlab, wpre, wcl = w
        assert ginit.tobytes() == winit.tobytes(), tag + ": initialize_clusters differs"
        assert (gpre == wpre).all(), tag + ": pre-CCA labels differ (%d px)" % (gpre != wpre).sum()
        assert gcl.tobytes() == wcl.tobytes(), tag + ": Cluster records differ"
        assert (glab == wlab).all(), tag + ": final labels differ (%d px)" % (glab != wlab).sum()


@pytest.mark.parametrize("case", smc.INT_CASES, ids=lambda c: c[0])
def test_integer_path(want, monkeypatch, case):
    from fast_slic_b200 import clear_engine_cache
    img, K, args = smc.case_image(case)
    path = case[6]
    if path == "ldg_forced":
        monkeypatch.setenv("FSLIC_ASSIGN", "4")
        clear_engine_cache()
    try:
        eng, got = _run_engine(img, K, args)
        _compare(case[0], got, want[case[0]])
        if path == "tma":
            assert eng.assign_impl() == 5, "the TMA-staged kernel did not run (impl %d)" % eng.assign_impl()
        elif path in ("ldg", "ldg_forced"):
            assert eng.assign_impl() == 4, "the LDG kernel did not run (impl %d)" % eng.assign_impl()
        elif path == "generic":
            assert eng.S > 110 and eng.assign_impl() == 0
    finally:
        if path == "ldg_forced":
            clear_engine_cache()


@pytest.mark.parametrize("variant", [0, 1, 2], ids=["SlicRealDist", "SlicRealDistL2", "SlicRealDistNoQ"])
@pytest.mark.parametrize("case", smc.REAL_CASES, ids=lambda c: c[0])
def test_real_dist_variants(want, case, variant):
    img, K, args = smc.case_image(case)
    _compare("%s/%d" % (case[0], variant), _run_engine(img, K, args, variant=variant)[1], want[(case[0], variant)])


@pytest.mark.parametrize("case", smc.PREEMPT_CASES, ids=lambda c: c[0])
def test_preemptive(want, case):
    img, K, args = smc.case_image(case)
    _compare(case[0], _run_engine(img, K, args, preempt=True)[1], want[case[0]])


def test_python_classes(want):
    """Slic / SlicRealDistNoQ(manhattan_spatial_dist=False).iterate, twice (warm start), through the public surface."""
    from fast_slic_b200 import Slic, SlicRealDistNoQ
    for case, cls, key in ((smc.INT_CASES[4], Slic, smc.INT_CASES[4][0]),
                           (smc.REAL_CASES[0], SlicRealDistNoQ, (smc.REAL_CASES[0][0], 2))):
        img, K, args = smc.case_image(case)
        s = cls(num_components=K, compactness=args["compactness"], min_size_factor=args["min_size_factor"],
                subsample_stride=args["subsample_stride"], convert_to_lab=args["convert_to_lab"], manhattan_spatial_dist=False)
        for n in range(2):
            lab = s.iterate(img, max_iter=args["max_iter"])
            assert (lab.view(np.uint16) == want[key][n][1]).all(), (key, n)
            assert s.slic_model.cluster_array.tobytes() == want[key][n][3].tobytes(), (key, n)


def test_iterate_batch_host_and_device(want):
    from fast_slic_b200 import Slic
    H, W, K, imgs = smc.batch_inputs()
    s = Slic(num_components=K, manhattan_spatial_dist=False)
    lab_d, cl_d = s.iterate_batch(torch.from_numpy(imgs).cuda(), return_clusters=True)
    lab_h, cl_h = s.iterate_batch(imgs, return_clusters=True)
    lab_d = lab_d.cpu().numpy().view(np.uint16)
    for b, (_, wlab, _, wcl) in enumerate(want["batch"]):
        assert (lab_d[b] == wlab).all() and (lab_h[b].view(np.uint16) == wlab).all(), b
        assert cl_d[b].cpu().numpy().tobytes() == wcl.tobytes() == cl_h[b].tobytes(), b


def test_blocking_host_call_of_17_images(want):
    """>= 16 images in one blocking host call: the two halves run as two overlapping pipelines."""
    from fast_slic_b200 import Slic
    H, W, K, imgs = smc.blocking17_inputs()
    lab, cl = Slic(num_components=K, manhattan_spatial_dist=False).iterate_batch(imgs, return_clusters=True)
    for b, (_, wlab, _, wcl) in enumerate(want["blocking17"]):
        assert (lab[b].view(np.uint16) == wlab).all(), b
        assert cl[b].tobytes() == wcl.tobytes(), b


def test_stream_warm_start(want):
    from fast_slic_b200 import SlicStream
    H, W, K, frames = smc.stream_inputs()
    st = SlicStream(H, W, K, batch=2, depth=2, warm_start=True, manhattan_spatial_dist=False)
    try:
        for t, frame in enumerate(frames):
            st.submit(frame)
            labs, cls = st.collect()
            for b in range(2):
                wlab, wcl = want["stream"][b][t]
                assert (labs[b].view(np.uint16) == wlab).all(), (t, b)
                assert cls[b].tobytes() == wcl.tobytes(), (t, b)
    finally:
        st.close()


def test_graph_replay_alternating_metrics_on_one_context(want):
    """One cached context, Manhattan and Euclidean calls in turn with the same coef: single-image host calls replay a
    captured CUDA graph, and the spatial patch is cached, yet every call gets its own metric's answer."""
    from fast_slic_b200 import Slic
    H, W, K, imgs = smc.alternating_inputs()
    man, euc = Slic(num_components=K), Slic(num_components=K, manhattan_spatial_dist=False)
    for rnd in range(2):  # the second round replays graphs that exist by then
        for t, img in enumerate(imgs):
            s = man if t % 2 == 0 else euc
            s.slic_model.initialized = False  # a cold start every call, like the reference's answers
            lab = s.iterate(img)
            _, wlab, _, wcl = want["alternating"][t]
            assert (lab.view(np.uint16) == wlab).all(), (rnd, t)
            assert s.slic_model.cluster_array.tobytes() == wcl.tobytes(), (rnd, t)
