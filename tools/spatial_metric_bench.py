"""Manhattan vs Euclidean spatial term (`manhattan_spatial_dist`) on the flagship workload.

Workload: BASELINE.json configs[1] (1280x720 RGB, K=1600, compactness 10, 10 iterations, stride 3, Lab,
min_size_factor 0), a batch of 32 images resident in device memory, one context.  Both metrics run in the same process,
alternating step by step, so clock and thermal drift hit them alike.  Per metric: the median wall time of one
iterate() of the batch (CUDA events on the launch stream) and the summed time of the fused assign+update kernel
launches of that call (collect_timing=2, events around each launch).  Prints one JSON line with the card name and its
power limit beside the numbers.

    python tools/spatial_metric_bench.py [--steps 20] [--warmup 3] [--batch 32]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def power_limit_w(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        return float(out)
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32)
    a = ap.parse_args()
    from fast_slic_b200 import Engine
    from oracle.oracle import synthetic_image

    H, W, K = 720, 1280, 1600
    B = a.batch
    dev = torch.device("cuda", 0)
    imgs = torch.from_numpy(np.stack([synthetic_image(H, W, seed=1000 + b) for b in range(B)])).to(dev)
    eng = Engine(H, W, K, B, 0)
    seed = eng.initialize_clusters(imgs)
    clusters = seed.clone()
    labels = torch.empty((B, H, W), dtype=torch.int16, device=dev)
    p_plain = eng.params(10.0, 0.0, 3, True, 10)
    p_timed = eng.params(10.0, 0.0, 3, True, 10, collect_timing=2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {True: {"ms": [], "assign_ms": [], "assign_launches": None}, False: {"ms": [], "assign_ms": [], "assign_launches": None}}
    for step in range(a.warmup + a.steps):
        for manhattan in (True, False):
            eng.set_manhattan_spatial_dist(manhattan)
            clusters.copy_(seed)
            torch.cuda.synchronize()
            e0.record()
            eng.iterate(imgs, clusters, p_plain, labels)
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            clusters.copy_(seed)
            eng.iterate(imgs, clusters, p_timed, labels)  # synchronous: it reads its events back
            kms, n = eng.assign_kernel_time()
            if step >= a.warmup:
                r = res[manhattan]
                r["ms"].append(ms)
                r["assign_ms"].append(kms)
                r["assign_launches"] = n
    eng.set_manhattan_spatial_dist(True)
    out = {"workload": "BASELINE configs[1] %dx%d K=%d, batch %d resident on the device" % (W, H, K, B),
           "card": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(0),
           "steps": a.steps, "warmup": a.warmup}
    for manhattan, name in ((True, "manhattan"), (False, "euclidean")):
        r = res[manhattan]
        med = statistics.median(r["ms"])
        out[name] = {"iterate_ms_median": round(med, 4), "iterate_ms_min": round(min(r["ms"]), 4),
                     "images_per_s": round(B * 1000.0 / med, 1),
                     "assign_kernel_ms_median": round(statistics.median(r["assign_ms"]), 4),
                     "assign_kernel_launches": r["assign_launches"]}
    out["euclidean_over_manhattan"] = round(out["euclidean"]["iterate_ms_median"] / out["manhattan"]["iterate_ms_median"], 4)
    print(json.dumps(out))
    eng.close()


if __name__ == "__main__":
    main()
