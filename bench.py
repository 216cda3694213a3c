#!/usr/bin/env python
"""bench.py -- megapixels/s of the SLIC iterate() hot path (Lab LUT -> 10 x (assign+update) -> full
assign -> connectivity enforcement) on B200, with the reference's own CPU build timed beside it.

Workload (BASELINE.json configs[1]): 1280x720 RGB, K=1600, compactness=10, 10 iterations,
subsample_stride=3, convert_to_lab, min_size_factor=0 (BASELINE.md section 2).  One step = one batch of
`--batch` independent images of that shape per GPU (default 32: the north star's "synthetic image
batches"; the single-image latency of configs[1] is reported beside it under "single_image").  Each rank
owns its own images (weak scaling, no collective on the data path).

  python bench.py --gpus 1 --steps 20 --warmup 5            # this framework
  python bench.py --impl reference --steps 5 --warmup 1     # the reference's CPU path on the host cores
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

def usable_cores():
    """CPUs this process may really use: min(affinity, cgroup cpu quota).  The GPU boxes show 128 logical
    CPUs but run the container under a 16-CPU cgroup quota; OpenMP with 128 threads then thrashes."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def bind_to_gpu_numa_node(local_rank):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, so pinned host buffers (first touch) and the
    copy threads are local to it: on the 2-socket GPU boxes a far-node pinned buffer uploads at ~22 GB/s instead of
    ~53 GB/s.  Best effort; returns a short description for the JSON line."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id if hasattr(
            torch.cuda.get_device_properties(local_rank), "pci_bus_id") else None
        dom = getattr(torch.cuda.get_device_properties(local_rank), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local_rank), "pci_device_id", 0)
        if bus is None:
            return "pci id unavailable"
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return "numa node unknown"
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return "numa node %d has no allowed cpu" % node
        os.sched_setaffinity(0, allowed)
        return "bound to numa node %d (%d cpus)" % (node, len(allowed))
    except Exception as e:  # noqa: BLE001
        return "not bound (%s)" % type(e).__name__


WORKLOADS = {
    # name: H, W, K, min_size_factor
    "B": (720, 1280, 1600, 0.0),     # configs[1]
    "B_msf0.1": (720, 1280, 1600, 0.1),  # configs[4]
    "C": (1080, 1920, 2000, 0.0),    # configs[2]
    "D": (2160, 3840, 4000, 0.0),    # configs[3]
    "A": (480, 640, 200, 0.25),      # configs[0]
}
COMPACTNESS, MAX_ITER, STRIDE = 10.0, 10, 3
CONFIG_INDEX = {"A": 0, "B": 1, "C": 2, "D": 3, "B_msf0.1": 4}   # BASELINE.json configs[i] each workload's shape comes from


def workload_string(name, B):
    """One string for both arms (the driver compares them): the BASELINE.json config the shape and parameters come
    from, and how many independent images of it make one step on each GPU."""
    H, W, K, msf = WORKLOADS[name]
    return ("%dx%d RGB, K=%d, compactness=10, 10 iters, stride 3, Lab, min_size_factor=%g (BASELINE configs[%d]), "
            "%d independent image(s)/step/GPU" % (W, H, K, msf, CONFIG_INDEX[name], B))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="B", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=32, help="images per step per GPU")
    ap.add_argument("--sigma", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--contexts", type=int, default=4,
                    help="independent batches in flight per GPU (contexts used round-robin, one stream each); "
                         "1 = strictly one step after the other")
    ap.add_argument("--extra-batched", type=int, default=1,
                    help="also report throughput at this batch size (0 = skip); default 1 = single-image latency")
    ap.add_argument("--no-gather", action="store_true",
                    help="N > 1 only: skip the extra timed loop that all-gathers every step's labels over NCCL")
    ap.add_argument("--no-parity-check", action="store_true",
                    help="skip the post-run comparison of one image per arm with the CPU oracle")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the labels and clusters of the last timed step of the headline arm (rank 0) to "
                         "DIR/<name>.npy, so that two builds can be compared output for output")
    return ap.parse_args()


# ---------------------------------------------------------------------------------------------------
def synth_images_torch(n, H, W, seed, sigma, device):
    """SURVEY.md section 8(d) synthetic inputs, generated on the device (seeded)."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    y = torch.arange(H, device=device, dtype=torch.float32)[:, None]
    x = torch.arange(W, device=device, dtype=torch.float32)[None, :]
    base = torch.stack([torch.sin(x / 37 + y / 91), torch.cos(y / 53 - x / 113), torch.sin((x + y) / 71)], -1)
    out = torch.empty((n, H, W, 3), dtype=torch.uint8, device=device)
    for i in range(n):
        phase = 0.37 * i
        img = 127 + 100 * torch.roll(base, shifts=(7 * i) % W, dims=1) * (1.0 - 0.1 * np.sin(phase))
        img = img + torch.randn((H, W, 3), generator=g, device=device) * sigma
        out[i] = img.clamp(0, 255).to(torch.uint8)
    return out


def pool_images_host(n, H, W, seed, sigma):
    """The first `n` images of the GPU arm's input pool as a host array -- the SAME bytes the GPU arm segments
    (generated by the same seeded generator on the same kind of device, then copied back).  Without a GPU (this
    happens only off the bench box) the same formula runs on the CPU generator."""
    import torch
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))) if torch.cuda.is_available() else torch.device("cpu")
    return synth_images_torch(n, H, W, seed, sigma, dev).cpu().numpy()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the GPU is under this benchmark's load (B200_PROFILING.md
    recipe).  Started before the warm-up (nvidia-smi needs ~0.5 s to produce its first line); `mark()` brackets
    the timed region; samples inside the bracket are preferred, else all samples taken under load are used."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc, self.t0, self.t1 = [], None, None, None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def wait_first(self, timeout=3.0):
        t = time.time()
        while self.proc and not self.lines and time.time() - t < timeout:
            time.sleep(0.02)

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()

        def parse(lines):
            sm, mx, reasons = [], [], set()
            for _, ln in lines:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0])); mx.append(float(f[1]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons
        inside = [x for x in self.lines if self.t0 and self.t1 and self.t0 <= x[0] <= self.t1 + 0.05]
        scope = "timed region"
        if len(inside) < 2:
            inside, scope = self.lines[1:] or self.lines, "warm-up + timed region (timed region shorter than the sampling period)"
        sm, mx, reasons = parse(inside)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "scope": scope}


DUMP_BYTES = 63_000_000   # array data of --dump-outputs: under 64 MB in all with the .npy headers


def dump_outputs(out_dir, labels, clusters):
    """What the last timed step returned to its caller: labels [B, H, W] (u16 superpixel ids, as float32) and the
    Cluster records [B, K] (one float64 column per field, in CLUSTER_DTYPE order).  An array larger than its share of
    DUMP_BYTES is written as a sorted sample of its flat elements (labels) or records (clusters), drawn with a fixed
    seed, beside the flat indices of the sample as <name>_index.npy."""
    from fast_slic_b200 import CLUSTER_DTYPE
    os.makedirs(out_dir, exist_ok=True)
    B, K = clusters.shape[:2]
    lab = labels.view(np.uint16).astype(np.float32)
    cl = np.ascontiguousarray(clusters).reshape(B * K, 32).view(CLUSTER_DTYPE).reshape(-1)
    rec = np.stack([cl[f].astype(np.float64) for f in CLUSTER_DTYPE.names], -1)
    for name, a, rows, share in (("labels", lab, lab.reshape(-1), 0.75),
                                 ("clusters", rec.reshape(B, K, -1), rec, 0.25)):
        if a.nbytes > share * DUMP_BYTES:
            n = int(share * DUMP_BYTES // (rows[0].nbytes + 8))
            idx = np.sort(np.random.RandomState(0).choice(len(rows), n, replace=False))
            np.save(os.path.join(out_dir, name + "_index.npy"), idx.astype(np.float64))
            a = rows[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------
def _ref_impl():
    from oracle.oracle import Port, Ref
    use_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libfslic_ref.so")) or os.path.isdir("/root/reference/src")
    return (Ref() if use_ref else Port()), use_ref


def _ref_one(impl, use_ref, img, K, msf, threads):
    """Seconds of ONE iterate() of the reference on one image.  initialize() -- Context construction + grid seeding,
    cfast_slic.pyx:124-147 -- is outside the clock, like on the GPU arm (BASELINE.md section 3)."""
    cl = impl.initialize(img, K)
    t0 = time.perf_counter()
    if use_ref:
        impl.iterate(img, cl, MAX_ITER, COMPACTNESS, msf, STRIDE, True, arch="x64/avx2", num_threads=threads)
    else:
        impl.iterate(img, cl, MAX_ITER, COMPACTNESS, msf, STRIDE, True)
    return time.perf_counter() - t0


def pick_ref_threads(impl, use_ref, imgs, K, msf, reps=5):
    """Thread count that makes the reference fastest on this box (it does not scale past a few cores on small
    images, and oversubscribing a cgroup quota is catastrophic): best of `reps` runs per count, up to the usable cores."""
    if not use_ref:
        return 1, {}
    cores = usable_cores()
    cands = sorted({c for c in (1, 2, 4, 8, 16, 32, 64, cores) if c <= cores})
    best, sweep = (1e9, 1), {}
    for c in cands:
        _ref_one(impl, use_ref, imgs[0], K, msf, c)  # warm the OpenMP pool at this size
        t = min(_ref_one(impl, use_ref, imgs[r % len(imgs)], K, msf, c) for r in range(reps))
        sweep[c] = t
        if t < best[0]:
            best = (t, c)
    return best[1], sweep


def cpu_reference_run(imgs, K, msf, seconds_budget):
    """Times the reference's CPU implementation (oracle/_ref = unmodified reference compiled from source;
    falls back to the plain-C port) on this box's host cores, on images copied back from the GPU arm's own input
    pool.  Bounded sample, one image at a time (the reference has no batch API), iterate() only."""
    impl, use_ref = _ref_impl()
    H, W = imgs[0].shape[:2]
    threads, sweep = pick_ref_threads(impl, use_ref, imgs, K, msf)
    _ref_one(impl, use_ref, imgs[0], K, msf, threads)
    times, t_start = [], time.perf_counter()
    while len(times) < 3 or (time.perf_counter() - t_start < seconds_budget and len(times) < 400):
        times.append(_ref_one(impl, use_ref, imgs[len(times) % len(imgs)], K, msf, threads))
    mp = H * W / 1e6
    return {
        "value": mp / float(np.mean(times)), "best": mp / float(np.min(times)), "median": mp / float(np.median(times)),
        "unit": "megapixels/s", "cores": threads, "kind": "reference" if use_ref else "port",
        "sample": "%d x iterate() (initialize outside the clock) over %d images of the GPU arm's own pool, %dx%d K=%d "
                  "(mean; SlicAvx2 path, %d OpenMP threads = fastest of the sweep %s [best of 5 each] on %d usable "
                  "cores), after warm-up"
                  % (len(times), len(imgs), W, H, K, threads, {k: round(1e3 * v, 1) for k, v in sweep.items()},
                     usable_cores()),
        "single_thread_value": (mp / sweep[1]) if 1 in sweep else None,
        "ms_per_image": 1e3 * float(np.mean(times)),
    }


def run_reference_arm(args):
    H, W, K, msf = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    impl, use_ref = _ref_impl()
    imgs = list(pool_images_host(8, H, W, 1000, args.sigma))     # == rank 0's first 8 pool images on the GPU arm
    cores, sweep = pick_ref_threads(impl, use_ref, imgs, K, msf)
    per_step = max(1, args.batch)

    def step(i):  # seconds spent inside iterate() for one step's images
        return sum(_ref_one(impl, use_ref, imgs[(i * per_step + b) % len(imgs)], K, msf, cores) for b in range(per_step))

    for i in range(args.warmup):
        step(i)
    per = [step(i) for i in range(args.steps)]
    dt = float(np.sum(per))
    value = per_step * args.steps * H * W / 1e6 / dt
    out = {
        "impl": "reference", "metric": "megapixels/sec (10 iters, K=%d)" % K, "value": value, "unit": "megapixels/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "ms_per_step_median": 1e3 * float(np.median(per)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u16 integer",
        "data": "synthetic",
        "config": {"workload": workload_string(args.workload, per_step),
                   "how": "one image at a time (the reference has no batch API); clock around iterate() only, like the "
                          "GPU arm; images = the first 8 of the GPU arm's pool (same seeded bytes)"},
        "cpu_baseline": {"value": value, "unit": "megapixels/s", "cores": cores,
                         "kind": "reference" if use_ref else "port",
                         "sample": "%d timed steps of %d image(s), SlicAvx2 path of the unmodified reference, %d OpenMP "
                                   "threads (fastest of sweep %s, best of 5 each; %d usable cores)"
                                   % (args.steps, per_step, cores, {k: round(1e3 * v, 1) for k, v in sweep.items()},
                                      usable_cores())},
        "e2e": {"value": value, "unit": "megapixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


# ---------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    import torch
    import torch.distributed as dist
    from fast_slic_b200 import Slic, get_engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        # NCCL may print its version banner to stdout when the communicator is created; the contract is ONE JSON
        # line on stdout, so stdout points at stderr until the first collective is through
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            warm = torch.zeros(1, device=device)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    H, W, K, msf = WORKLOADS[args.workload]
    B = max(1, args.batch)
    MP = H * W / 1e6

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- inputs: a pool of distinct images larger than L2 (126 MB) so no step finds its input cached ----
    img_bytes = H * W * 3
    pool_steps = max(2, int(np.ceil(300e6 / (img_bytes * B))))
    pool_steps = min(pool_steps, 128)
    pool = synth_images_torch(pool_steps * B, H, W, 1000 * (rank + 1), args.sigma, device).view(pool_steps, B, H, W, 3)
    eng = get_engine(H, W, K, max(B, args.extra_batched if args.extra_batched > 0 else 1), local_rank)
    pristine = eng.initialize_clusters(pool[0])           # centres are image independent; colours get re-seeded
    clusters = pristine.clone()
    labels = torch.empty((B, H, W), dtype=torch.int16, device=device)
    p_fast = eng.params(COMPACTNESS, msf, STRIDE, True, MAX_ITER, collect_timing=0)
    p_prof = eng.params(COMPACTNESS, msf, STRIDE, True, MAX_ITER, collect_timing=2)

    def step(i, params):
        clusters.copy_(pristine)                           # every step is a cold start, like a fresh Slic()
        eng.iterate(pool[i % pool_steps], clusters, params, labels)

    # ---- kernel-resident throughput: inputs already in HBM ----
    # (1) one step after the other on one stream
    for i in range(args.warmup):
        step(i, p_fast)
    barrier()
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    marks[0].record()
    for i in range(args.steps):
        step(args.warmup + i, p_fast)
        marks[i + 1].record()
    barrier()
    ms_seq = max_over_ranks(marks[0].elapsed_time(marks[-1]))
    seq_steps = [marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps)]
    launches = eng.launches_last_iterate() * args.steps
    seq_last = (args.warmup + args.steps - 1) % pool_steps     # pool slot of the last sequential step (parity check)
    seq_out = (labels.clone(), clusters.clone())

    # (2) the same K steps issued round-robin over NCTX contexts, one stream each: successive batches are
    # independent, so the latency-bound stretch of one (the std::partial_sort replay) runs under the
    # bandwidth-hungry kernels of the next.  Timed with events on the launching stream: fork before, join after.
    from fast_slic_b200 import Engine
    NCTX = max(1, args.contexts)
    lanes = [(eng, clusters, labels, torch.cuda.Stream(device))]
    for _ in range(NCTX - 1):
        lanes.append((Engine(H, W, K, B, local_rank), pristine.clone(), torch.empty_like(labels), torch.cuda.Stream(device)))

    lane_last = {}

    def lane_step(i):
        e, cl, lab, st = lanes[i % NCTX]
        lane_last[i % NCTX] = i % pool_steps
        with torch.cuda.stream(st):
            cl.copy_(pristine, non_blocking=True)
            e.iterate(pool[i % pool_steps], cl, p_fast, lab)

    def fork_join(n, first):
        main = torch.cuda.current_stream(device)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(main)
        for _, _, _, st in lanes:
            st.wait_event(a)
        for i in range(n):
            lane_step(first + i)
        for _, _, _, st in lanes:
            j = torch.cuda.Event()
            j.record(st)
            main.wait_event(j)
        b.record(main)
        return a, b

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.wait_first()
    fork_join(max(args.warmup, NCTX), 0)
    barrier()
    barrier()
    if sampler:
        sampler.mark_begin()
    e0, e1 = fork_join(args.steps, args.warmup)
    barrier()
    if sampler:
        sampler.mark_end()
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler else None
    value = world * B * args.steps * MP / (ms / 1e3)
    last_lane = (args.warmup + args.steps - 1) % NCTX
    value_out = (lane_last[last_lane], lanes[last_lane][2].clone(), lanes[last_lane][1].clone())

    # ---- N > 1: the same loop with the one collective the path has -- the final label gather (SURVEY 8e) ----
    # Every step's u16 label maps are all-gathered over NCCL (int16 on the wire) on a side stream, so the gather of
    # step i overlaps the kernels of step i+1; a lane's label buffer is not reused before its gather has drained.
    gather = None
    if world > 1 and not args.no_gather:
        comm = torch.cuda.Stream(device)
        gbuf = [torch.empty((world, B, H, W), dtype=torch.int16, device=device) for _ in range(NCTX)]
        drained = [None] * NCTX

        def gather_step(i):
            e, cl, lab, st = lanes[i % NCTX]
            if drained[i % NCTX] is not None:
                st.wait_event(drained[i % NCTX])            # labels of this lane's previous step have left
            with torch.cuda.stream(st):
                cl.copy_(pristine, non_blocking=True)
                e.iterate(pool[i % pool_steps], cl, p_fast, lab)
                done = torch.cuda.Event()
                done.record(st)
            with torch.cuda.stream(comm):
                comm.wait_event(done)
                # raw bytes on the wire: NCCL's process group has no int16, and the labels are opaque u16 anyway
                dist.all_gather_into_tensor(gbuf[i % NCTX].view(torch.uint8).view(-1), lab.view(torch.uint8).view(-1))
                ev = torch.cuda.Event()
                ev.record(comm)
                drained[i % NCTX] = ev

        def gather_run(n, first):
            main = torch.cuda.current_stream(device)
            a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(main)
            for _, _, _, st in lanes:
                st.wait_event(a)
            comm.wait_event(a)
            for i in range(n):
                gather_step(first + i)
            for _, _, _, st in lanes:
                j = torch.cuda.Event(); j.record(st); main.wait_event(j)
            j = torch.cuda.Event(); j.record(comm); main.wait_event(j)
            b2.record(main)
            return a, b2

        gather_run(max(args.warmup, NCTX), 0)
        barrier()
        g0, g1 = gather_run(args.steps, args.warmup)
        barrier()
        gms = max_over_ranks(g0.elapsed_time(g1))
        # every rank must now hold every rank's labels of the last step: check one word per rank against the source
        chk = gbuf[(args.warmup + args.steps - 1) % NCTX]
        mine = lanes[(args.warmup + args.steps - 1) % NCTX][2]
        ok = bool((chk[rank] == mine).all().item())
        gather = {"value": world * B * args.steps * MP / (gms / 1e3), "unit": "megapixels/s",
                  "ms_per_step": gms / args.steps, "collective": "ncclAllGather of int16 labels [B,H,W] per rank per step "
                  "(torch.distributed all_gather_into_tensor) on a side stream, overlapped with the next step's kernels",
                  "bytes_received_per_rank_per_step": (world - 1) * B * H * W * 2, "own_shard_intact": ok,
                  "without_gather_value": value}

    # ---- roofline of the dominant kernel: per-launch CUDA events on the launch stream, same workload ----
    k_ms, k_n = 0.0, 0
    for i in range(max(3, min(args.steps, 10))):
        step(i, p_prof)
        a, n = eng.assign_kernel_time()
        k_ms += a
        k_n += n
    stage = eng.stage_ms()
    cca_stage = eng.cca_stage_ms()
    kernel_name = ("k_assign5<TS,3,true,TPS> (TMA-staged fused assign+update, subsampled pass)" if eng.assign_impl() == 5
                   else "k_assign_warp<TS,3,true> (fused assign+update, subsampled pass)")
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    if os.path.exists(peaks_path):
        try:
            peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "MEASURED_PEAKS.json hbm_gbs"
        except Exception:
            pass
    sub_px = B * W * ((H + STRIDE - 1) // STRIDE)          # pixels one subsampled launch touches (rem = 0 rows)
    alg_bytes = 6.0 * sub_px                               # 4 B quad read + 2 B label written per pixel
    avg_ms = k_ms / max(k_n, 1)
    achieved = alg_bytes / (avg_ms * 1e-3) / 1e9 if k_n else 0.0
    traffic = None  # dram__bytes_read + dram__bytes_write per launch, from the committed ncu --set full capture
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "assign_traffic.json")))
        traffic = tj.get("%s_batch%d" % (args.workload, B), {}).get("traffic")
    except Exception:
        pass
    roofline = {"kernel": kernel_name, "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "bytes_per_launch": alg_bytes, "avg_launch_us": avg_ms * 1e3,
                "launches_timed": k_n, "stage_ms_last_step": stage}
    if any(v > 0 for v in cca_stage.values()):  # the connectivity sub-stages are only timed for batches below 4 (one stream)
        roofline["cca_stage_ms_last_step"] = cca_stage

    # ---- end to end through the public API with HOST buffers (H2D + compute + D2H inside the timed region) ----
    slic = Slic(num_components=K, compactness=COMPACTNESS, min_size_factor=msf, subsample_stride=STRIDE)
    slic.slic_model.device = local_rank
    n_host = min(pool_steps, 8)
    host_imgs = torch.empty((n_host, B, H, W, 3), dtype=torch.uint8).pin_memory()
    host_imgs.copy_(pool[:n_host])
    host_np = host_imgs.numpy()
    host_pristine = torch.empty(pristine.shape, dtype=torch.uint8).pin_memory()
    host_pristine.copy_(pristine)
    from fast_slic_b200 import CLUSTER_DTYPE
    cl_u8 = host_pristine.numpy()                      # raw bytes: a structured-dtype assignment copies field by field
    work_u8 = torch.empty(pristine.shape, dtype=torch.uint8).pin_memory().numpy()
    work_cl = work_u8.view(CLUSTER_DTYPE).reshape(B, K)
    lab_np = torch.empty((B, H, W), dtype=torch.int16).pin_memory().numpy()

    def e2e_step(i):
        work_u8[...] = cl_u8
        slic.iterate_batch(host_np[i % n_host], max_iter=MAX_ITER, clusters=work_cl)

    # iterate_batch allocates its own label array; for a tight loop use the engine's host entry directly
    def e2e_step_tight(i):
        work_u8[...] = cl_u8                                   # every step is a cold start, like a fresh Slic()
        eng.iterate_host(host_np[i % n_host], work_cl, p_fast, lab_np)

    e2e_step(0)
    for i in range(args.warmup):
        e2e_step_tight(i)
    barrier()
    per_step = []
    t0 = time.perf_counter()
    for i in range(args.steps):
        ts = time.perf_counter()
        e2e_step_tight(i)
        per_step.append(time.perf_counter() - ts)
    blocking_last = (args.steps - 1) % n_host
    blocking_out = (lab_np[0].copy(), work_u8[0].copy())       # slot 0 is reused by the streamed arm below
    torch.cuda.synchronize()
    dt_block = max_over_ranks(time.perf_counter() - t0)
    barrier()
    h2d = B * (H * W * 3 + K * 32)
    d2h = B * (H * W * 2 + K * 32)

    # streaming form of the same call: two contexts, fslic_b200_iterate_host_async / fslic_b200_wait alternating, so
    # one batch's PCIe copies overlap the other's kernels.  Every step still uploads its own images + clusters and
    # downloads its own labels + clusters inside the timed region.
    from fast_slic_b200 import Engine
    slots = [(eng, work_u8, work_cl, lab_np)]
    for lane in lanes[1:]:
        wu_b = torch.empty(pristine.shape, dtype=torch.uint8).pin_memory().numpy()
        slots.append((lane[0], wu_b, wu_b.view(CLUSTER_DTYPE).reshape(B, K),
                      torch.empty((B, H, W), dtype=torch.int16).pin_memory().numpy()))

    def e2e_submit(i):
        e, wu, wcl, lab = slots[i % NCTX]
        e.wait()                                               # results of step i-2 are in host memory
        wu[...] = cl_u8
        e.iterate_host_async(host_np[i % n_host], wcl, p_fast, lab)

    for i in range(max(args.warmup, NCTX)):
        e2e_submit(i)
    for e, _, _, _ in slots:
        e.wait()
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_submit(i)
    for e, _, _, _ in slots:
        e.wait()
    dt = max_over_ranks(time.perf_counter() - t0)
    stream_last = ((args.steps - 1) % n_host, (args.steps - 1) % NCTX)
    barrier()
    e2e_value = world * B * args.steps * MP / dt

    # ---- informational: batched throughput on the same image shape ----
    batched = None
    if args.extra_batched > 0 and args.extra_batched != B:
        EB = args.extra_batched
        nsteps_b = args.steps
        flat = pool.view(-1, H, W, 3)
        nb = flat.shape[0] // EB
        if nb >= 1:
            pr = eng.initialize_clusters(flat[:EB])
            cb = pr.clone()
            lb = torch.empty((EB, H, W), dtype=torch.int16, device=device)
            # on a stream of its own: from the second call with the same cluster / label buffers fslic_b200_iterate replays a
            # CUDA graph for fewer than 4 images (the legacy default stream cannot be captured)
            side = torch.cuda.Stream(device)
            side.wait_stream(torch.cuda.current_stream(device))
            with torch.cuda.stream(side):
                for i in range(4):
                    cb.copy_(pr); eng.iterate(flat[(i % nb) * EB:(i % nb + 1) * EB], cb, p_fast, lb)
                side.synchronize()
                barrier()
                b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                b0.record(side)
                for i in range(nsteps_b):
                    cb.copy_(pr); eng.iterate(flat[(i % nb) * EB:(i % nb + 1) * EB], cb, p_fast, lb)
                b1.record(side)
                side.synchronize()
            barrier()
            bms = max_over_ranks(b0.elapsed_time(b1))
            kb_ms, kb_n = 0.0, 0
            for i in range(3):
                cb.copy_(pr); eng.iterate(flat[(i % nb) * EB:(i % nb + 1) * EB], cb, p_prof, lb)
                a, n = eng.assign_kernel_time(); kb_ms += a; kb_n += n
            ach = 6.0 * EB * W * ((H + STRIDE - 1) // STRIDE) / (kb_ms / max(kb_n, 1) * 1e-3) / 1e9
            # end to end (host buffers) at this batch size
            hcl0 = torch.empty(pr.shape, dtype=torch.uint8).pin_memory()
            hcl0.copy_(pr)
            hcl = torch.empty(pr.shape, dtype=torch.uint8).pin_memory()
            hl = torch.empty((EB, H, W), dtype=torch.int16).pin_memory()
            hl_np = hl.numpy()
            hcl0_u8, hcl_u8 = hcl0.numpy(), hcl.numpy()
            hcl_np = hcl_u8.view(CLUSTER_DTYPE).reshape(EB, K)
            n_rot = max(1, min(16, flat.shape[0] // EB))         # rotate through several inputs like the device loop
            hbr = torch.empty((n_rot, EB, H, W, 3), dtype=torch.uint8).pin_memory()
            hbr.copy_(flat[:n_rot * EB].view(n_rot, EB, H, W, 3))
            hbr_np = hbr.numpy()
            for i in range(3):
                hcl_u8[...] = hcl0_u8
                eng.iterate_host(hbr_np[i % n_rot], hcl_np, p_fast, hl_np)
            t0b = time.perf_counter()
            per_call = []
            for i in range(nsteps_b):
                hcl_u8[...] = hcl0_u8
                tc = time.perf_counter()
                eng.iterate_host(hbr_np[i % n_rot], hcl_np, p_fast, hl_np)
                per_call.append(time.perf_counter() - tc)
            dtb = max_over_ranks(time.perf_counter() - t0b)
            # the same host calls, streamed: several independent requests of this size in flight (one context each)
            n_req = 8
            req = []
            for _ in range(n_req):
                e_r = Engine(H, W, K, EB, local_rank)
                cl_r = torch.empty(pr.shape, dtype=torch.uint8).pin_memory().numpy()
                req.append((e_r, cl_r, cl_r.view(CLUSTER_DTYPE).reshape(EB, K),
                            torch.empty((EB, H, W), dtype=torch.int16).pin_memory().numpy()))

            def req_submit(i):
                e_r, cu, ccl, lab_r = req[i % n_req]
                e_r.wait()
                cu[...] = hcl0_u8
                e_r.iterate_host_async(hbr_np[i % n_rot], ccl, p_fast, lab_r)

            for i in range(2 * n_req):
                req_submit(i)
            for r_ in req:
                r_[0].wait()
            nsteps_s = args.steps
            t0s = time.perf_counter()
            for i in range(nsteps_s):
                req_submit(i)
            for r_ in req:
                r_[0].wait()
            dts = max_over_ranks(time.perf_counter() - t0s)
            for r_ in req:
                r_[0].close()
            batched = {"batch": EB, "what": "same workload at this batch size (informational)",
                       "e2e_streamed": {"value": world * EB * nsteps_s * MP / dts, "unit": "megapixels/s",
                                        "ms_per_step": 1e3 * dts / nsteps_s, "requests_in_flight": n_req,
                                        "api": "fslic_b200_iterate_host_async / fslic_b200_wait, one context per request"},
                       "value": world * EB * nsteps_b * MP / (bms / 1e3), "unit": "megapixels/s",
                       "ms_per_step": bms / nsteps_b, "e2e_value": world * EB * nsteps_b * MP / dtb,
                       "e2e_ms_per_step": 1e3 * dtb / nsteps_b,
                       "e2e_ms_per_call_median": 1e3 * float(np.median(per_call)),
                       "e2e_ms_per_call_p90": 1e3 * float(np.percentile(per_call, 90)),
                       "e2e_note": "images whose K-th largest component area is tied ambiguously replay std::partial_sort on "
                                   "one warp (+ ~1 ms); the median is the common case, the mean includes them",
                       "assign_kernel_GBps": ach,
                       "assign_kernel_frac": ach / peak, "stage_ms": eng.stage_ms()}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_run(list(pool.view(-1, H, W, 3)[:8].cpu().numpy()), K, msf, seconds_budget=12.0)

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, value_out[1].cpu().numpy(), value_out[2].cpu().numpy())

    # ---- parity self-check, outside every timed region: image 0 of the LAST timed step of each arm against the CPU
    # oracle (the compiled reference when oracle/_ref is there).  A fast wrong answer must not print a number.
    parity = None
    if not args.no_parity_check:
        impl, use_ref = _ref_impl()

        def oracle_of(img_u8):
            cl0 = impl.initialize(img_u8, K)
            if use_ref:
                lab0 = impl.iterate(img_u8, cl0, MAX_ITER, COMPACTNESS, msf, STRIDE, True, arch="x64/avx2",
                                    num_threads=min(8, usable_cores()))
            else:
                lab0 = impl.iterate(img_u8, cl0, MAX_ITER, COMPACTNESS, msf, STRIDE, True)
            return lab0, cl0

        checks = {}
        cases = {
            "sequential": (pool[seq_last][0], seq_out[0][0], seq_out[1][0]),
            "value": (pool[value_out[0]][0], value_out[1][0], value_out[2][0]),
            "e2e_blocking": (host_imgs[blocking_last][0], torch.from_numpy(blocking_out[0]), torch.from_numpy(blocking_out[1])),
            "e2e": (host_imgs[stream_last[0]][0], torch.from_numpy(slots[stream_last[1]][3][0]),
                    torch.from_numpy(slots[stream_last[1]][1][0])),
        }
        for name, (img_t, lab_t, cl_t) in cases.items():
            want_lab, want_cl = oracle_of(np.ascontiguousarray(img_t.cpu().numpy()))
            got = lab_t.cpu().numpy().view(np.uint16)
            checks[name] = bool((got == want_lab).all()) and cl_t.cpu().numpy().tobytes() == want_cl.tobytes()
        parity = {"checked": True, "oracle": "reference" if use_ref else "port", "arms": checks,
                  "what": "image 0 of the last timed step of each arm: labels and raw Cluster bytes, tolerance 0"}
        if not all(checks.values()):
            raise SystemExit("bench.py: PARITY FAILURE on rank %d: %s -- no number is reported" % (rank, checks))

    numa_all = [numa]
    if world > 1:
        numa_all = [None] * world
        dist.all_gather_object(numa_all, numa)

    if rank == 0:
        out = {
            "metric": "megapixels/sec (10 iters, K=%d)" % K, "value": value, "unit": "megapixels/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u16 integer",
            "data": "synthetic",
            "config": {"workload": workload_string(args.workload, B),
                       "l2": "inputs rotate through a %d MB pool of distinct images (> 126 MB L2)"
                             % (pool_steps * B * img_bytes // 1000000),
                       "parallelism": "independent images per rank, no data-path collective",
                       "concurrency": "%d independent batches in flight per GPU (contexts used round-robin, one stream "
                                      "each); 'sequential' = one step after the other on one stream" % NCTX},
            "sequential": {"value": world * B * args.steps * MP / (ms_seq / 1e3), "unit": "megapixels/s",
                           "ms_per_step": ms_seq / args.steps, "ms_per_step_median": float(np.median(seq_steps)),
                           "ms_per_step_min": float(np.min(seq_steps)), "ms_per_step_max": float(np.max(seq_steps))},
            "parity_checked": bool(parity and parity["checked"]), "parity": parity,
            "gather": gather,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "megapixels/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * dt / args.steps,
                    "api": "fslic_b200_iterate_host_async + fslic_b200_wait (fast_slic_b200.Engine), %d contexts "
                           "round-robin, pinned host buffers; every step uploads its images+clusters and downloads "
                           "its labels+clusters inside the timed region" % NCTX,
                    "blocking": {"value": world * B * args.steps * MP / dt_block, "unit": "megapixels/s",
                                 "ms_per_step": 1e3 * dt_block / args.steps,
                                 "ms_per_step_median": 1e3 * float(np.median(per_step)),
                                 "ms_per_step_min": 1e3 * float(np.min(per_step)),
                                 "api": "fslic_b200_iterate_host (one blocking call per step, like the reference's "
                                        "iterate())"},
                    "numa": numa_all},
            "gpu_launches": launches,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "single_image" if (batched and batched["batch"] == 1) else "batched": batched,
        }
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
