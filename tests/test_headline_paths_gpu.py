"""GPU parity for the exact call patterns bench.py times (VERDICT r1 "what's weak" 1-2): the blocking and the
streamed HOST entry points at batch 32 (two half uploads, sliced front half, early label download keyed on the
per-image need_sim flag) and at an odd batch, and several contexts on several streams at once -- every image
of every step compared with the compiled reference's recorded answers (conftest.ReferenceAnswers).  Tolerance 0:
labels and raw Cluster bytes.
"""
import numpy as np
import pytest
import torch

from cases import make_image

pytestmark = pytest.mark.gpu

H, W, K = 720, 1280, 1600          # BASELINE configs[1]
ARGS = (10, 10.0, 0.0, 3, True)    # max_iter, compactness, min_size_factor, stride, convert_to_lab


def _images(n, seed0, sigmas=(12.0,)):
    return np.stack([make_image("syn", H, W, seed=seed0 + b, sigma=sigmas[b % len(sigmas)]) for b in range(n)])


def _want(checker, img, msf=0.0):
    cl = checker.initialize(img, K)
    lab = checker.iterate(img, cl, ARGS[0], ARGS[1], msf, ARGS[3], ARGS[4])
    return lab, cl


def _pinned(shape, dtype):
    return torch.empty(shape, dtype=dtype).pin_memory()


@pytest.fixture(scope="module")
def batch32(checker):
    imgs = _images(32, 5000, sigmas=(12.0, 12.0, 12.0, 40.0))
    want = [_want(checker, imgs[b]) for b in range(32)]
    return imgs, want


@pytest.mark.parametrize("nb", [32, 17, 9])
def test_blocking_host_call_batch(checker, batch32, nb):
    """fslic_b200_iterate_host at batch 32 and 17 (two overlapping half pipelines with their own streams and scratch
    windows, early D2H per half; 17 = odd halves) and 9 (one pipeline: split uploads + early D2H)."""
    from fast_slic_b200 import Engine
    imgs, want = batch32
    eng = Engine(H, W, K, 32)
    p = eng.params(ARGS[1], ARGS[2], ARGS[3], ARGS[4], ARGS[0])
    pin = _pinned((nb, H, W, 3), torch.uint8)
    pin.numpy()[...] = imgs[:nb]
    cl = eng.initialize_clusters_host(pin.numpy())
    lab = eng.iterate_host(pin.numpy(), cl, p)
    need_sim = [eng.cca_counters(b)["need_sim"] for b in range(nb)]
    for b in range(nb):
        assert (lab[b].view(np.uint16) == want[b][0]).all(), "image %d (need_sim=%d): %d px differ" % (
            b, need_sim[b], int((lab[b].view(np.uint16) != want[b][0]).sum()))
        assert cl[b].tobytes() == want[b][1].tobytes(), "clusters of image %d" % b
    # a second call on the same context (buffers reused) with pageable inputs
    cl2 = eng.initialize_clusters_host(imgs[:nb])
    lab2 = eng.iterate_host(np.ascontiguousarray(imgs[:nb]), cl2, p)
    for b in range(nb):
        assert (lab2[b].view(np.uint16) == want[b][0]).all() and cl2[b].tobytes() == want[b][1].tobytes()
    eng.close()


def test_streamed_host_calls_four_contexts(checker, batch32):
    """bench.py's e2e arm: fslic_b200_iterate_host_async / fslic_b200_wait round-robin over 4 contexts, batch 32,
    pinned buffers; every step's outputs are checked (steps use rotated images so a stale buffer would show)."""
    from fast_slic_b200 import CLUSTER_DTYPE, Engine
    imgs, want = batch32
    NCTX, STEPS, B = 4, 6, 32
    engs = [Engine(H, W, K, B) for _ in range(NCTX)]
    p = engs[0].params(ARGS[1], ARGS[2], ARGS[3], ARGS[4], ARGS[0])
    pristine = engs[0].initialize_clusters_host(imgs[:1]).view(np.uint8).reshape(K, 32).copy()
    host_in = _pinned((STEPS, B, H, W, 3), torch.uint8).numpy()
    for s in range(STEPS):
        host_in[s] = np.roll(imgs, s, axis=0)
    slots = [(_pinned((B, K, 32), torch.uint8).numpy(), _pinned((B, H, W), torch.int16).numpy()) for _ in range(NCTX)]
    results = {}

    def harvest(step):
        cl, lab = slots[step % NCTX]
        results[step] = (lab.copy(), cl.copy())

    for s in range(STEPS):
        e = engs[s % NCTX]
        e.wait()
        if s >= NCTX:
            harvest(s - NCTX)
        cl, lab = slots[s % NCTX]
        cl[...] = pristine
        e.iterate_host_async(host_in[s], cl.view(CLUSTER_DTYPE).reshape(B, K), p, lab)
    for s in range(max(0, STEPS - NCTX), STEPS):
        engs[s % NCTX].wait()
        harvest(s)
    for s in range(STEPS):
        lab, cl = results[s]
        for b in range(B):
            w = want[(b - s) % 32]   # np.roll(imgs, s)[b] == imgs[(b - s) % 32]
            assert (lab[b].view(np.uint16) == w[0]).all(), "step %d image %d" % (s, b)
            assert cl[b].tobytes() == w[1].tobytes(), "step %d clusters %d" % (s, b)
    for e in engs:
        e.close()


def test_device_calls_four_contexts_four_streams(checker, batch32):
    """bench.py's `value` arm: fslic_b200_iterate on device buffers, steps issued round-robin over 4 contexts with one
    stream each (fork / join on events), batch 32; all steps' outputs compared."""
    from fast_slic_b200 import Engine
    imgs, want = batch32
    dev = torch.device("cuda", 0)
    NCTX, STEPS, B = 4, 8, 32
    engs = [Engine(H, W, K, B) for _ in range(NCTX)]
    streams = [torch.cuda.Stream(dev) for _ in range(NCTX)]
    p = engs[0].params(ARGS[1], ARGS[2], ARGS[3], ARGS[4], ARGS[0])
    d_imgs = torch.from_numpy(imgs).to(dev)
    pool = [torch.roll(d_imgs, s, 0).contiguous() for s in range(STEPS)]
    pristine = engs[0].initialize_clusters(d_imgs)
    torch.cuda.synchronize()
    outs = []
    main = torch.cuda.current_stream(dev)
    fork = torch.cuda.Event()
    fork.record(main)
    for st in streams:
        st.wait_event(fork)
    for s in range(STEPS):
        with torch.cuda.stream(streams[s % NCTX]):
            cl = pristine.clone()
            lab = engs[s % NCTX].iterate(pool[s], cl, p)
            outs.append((lab, cl))
    for st in streams:
        j = torch.cuda.Event()
        j.record(st)
        main.wait_event(j)
    torch.cuda.synchronize()
    for s, (lab, cl) in enumerate(outs):
        lab = lab.cpu().numpy().view(np.uint16)
        cl = cl.cpu().numpy()
        for b in range(B):
            w = want[(b - s) % 32]
            assert (lab[b] == w[0]).all(), "step %d image %d: %d px differ" % (s, b, int((lab[b] != w[0]).sum()))
            assert cl[b].tobytes() == w[1].tobytes(), "step %d clusters %d" % (s, b)
    for e in engs:
        e.close()


def test_two_python_threads_same_shape(checker):
    """ADVICE r1: two threads segmenting same-sized images through the cached engine must not corrupt each other
    (ctypes drops the GIL during the call; the cached context is guarded by a lock)."""
    import threading
    from fast_slic_b200 import Slic
    h, w, k = 240, 320, 120
    imgs = [make_image("syn" if t % 2 else "noise", h, w, seed=900 + t) for t in range(2)]
    wants = []
    for im in imgs:
        cl = checker.initialize(im, k)
        wants.append((checker.iterate(im, cl, 10, 10.0, 0.1, 3, True), cl))
    errs = []

    def work(t):
        try:
            for _ in range(12):
                s = Slic(num_components=k, min_size_factor=0.1)
                got = s.iterate(imgs[t]).view(np.uint16)
                if not (got == wants[t][0]).all() or s.slic_model.cluster_array.tobytes() != wants[t][1].tobytes():
                    errs.append("thread %d: result differs" % t)
                    return
        except Exception as e:  # noqa: BLE001
            errs.append("thread %d: %r" % (t, e))

    th = [threading.Thread(target=work, args=(t,)) for t in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
