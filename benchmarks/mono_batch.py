"""The training batch of MonoDataset on one GPU (MonoBatch) against the reference's host chain, measured.

    python benchmarks/mono_batch.py [--out profiles/mono_batch_b200.json] [--reps 50]

Prints the card name, power limit and max SM clock, then one JSON line (also written to --out).  Batch 12 of KITTI's
1242x375 native frames, half the samples flipped and half augmented, for mono [0,-1,1] and mono+stereo [0,-1,1,"s"] at
640x192 and mono at 1024x320:

  gpu_ms:        MonoBatch.build per batch: CUDA events over replays of one CUDA graph per native batch, 4 native batches
                 in rotation (their frames and outputs together exceed the 126 MB L2);
  launches:      kernels and memsets of one call (torch.profiler, eager call);
  kernels_us:    per-kernel time of an eager call (torch.profiler, mean over calls);
  bytes / gbps:  algorithmic bytes (native frames read + color and color_aug written) over gpu_ms, and that rate over
                 7.7 TB/s;
  h2d_ms:        the one host-to-device copy of a packed native batch from pinned memory (CUDA events);
  host:          the reference's chain (oracle/mono_batch.py: PIL flip, LANCZOS pyramid, jitter, ToTensor, collation's
                 stack excluded) per sample, on one core and on a process pool over every host core, in samples/s.

It needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import re
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from benchmarks.amp_step import card, events_ms  # noqa: E402
from oracle import mono_batch as OM  # noqa: E402

B, NATIVE = 12, (375, 1242)
HBM_BPS = 7.7e12
N_BATCHES = 4
CONFIGS = [("mono_640x192", 192, 640, [0, -1, 1]), ("mono+stereo_640x192", 192, 640, [0, -1, 1, "s"]),
           ("mono_1024x320", 320, 1024, [0, -1, 1])]


def make_items(fids, seed):
    rng = np.random.default_rng(seed)
    items = []
    for b in range(B):
        torch.manual_seed(seed * 100 + b)
        aug = b % 2 == 1
        params = OM.jitter_params() if aug else None
        frames = {f: rng.integers(0, 256, NATIVE + (3,), dtype=np.uint8) for f in fids}
        items.append({"frames": frames, "do_color_aug": aug, "do_flip": (b // 2) % 2 == 1, "color_aug": params,
                      "side": "l" if b < B // 2 else "r"})
    return items


def _host_sample(args):
    torch.set_num_threads(1)
    item, H, W = args
    t = time.perf_counter()
    OM.get_item(item["frames"], item["do_flip"], item["color_aug"], item["side"], H, W, 4)
    return time.perf_counter() - t


def host_arm(items, H, W):
    torch.set_num_threads(1)
    n1 = 6
    t = time.perf_counter()
    for i in range(n1):
        _host_sample((items[i % len(items)], H, W))
    one = n1 / (time.perf_counter() - t)
    cores = os.cpu_count() or 1
    work = [(items[i % len(items)], H, W) for i in range(max(2 * cores, 24))]
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_host_sample, work[:cores])                 # start-up
        t = time.perf_counter()
        pool.map(_host_sample, work)
        pooled = len(work) / (time.perf_counter() - t)
    return {"one_core_samples_per_s": one, "pool_samples_per_s": pooled, "pool_processes": cores}


def gpu_arm(name, H, W, fids, reps):
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    natives = [collate_native(make_items(fids, 10 + k), pin_memory=True) for k in range(N_BATCHES)]
    mb = MonoBatch(H, W, fids, 4)
    flats = [mb.upload(nb) for nb in natives]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for nb, fl in zip(natives, flats):
            mb.build(nb, fl)
    torch.cuda.current_stream().wait_stream(side)
    graphs, outs = [], []
    for nb, fl in zip(natives, flats):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            outs.append(mb.build(nb, fl))
        graphs.append(g)
    for g in graphs:
        g.replay()
    gpu_ms = min(events_ms(lambda i: graphs[i % N_BATCHES].replay(), reps * N_BATCHES) for _ in range(3))
    h2d_ms = min(events_ms(lambda i: flats[i % N_BATCHES].copy_(natives[i % N_BATCHES].buffer, non_blocking=True), reps)
                 for _ in range(3))

    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(N_BATCHES):
            mb.build(natives[k], flats[k])
        torch.cuda.synchronize()
    kernels, launches = {}, 0
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            m = re.search(r"(md2_\w+)(<\d+>)?", e.name)
            key = m.group(1) + (m.group(2) or "") if m else e.name.split("(")[0].strip()
            if "Memcpy" in e.name:
                continue
            kernels.setdefault(key, []).append(e.device_time)
            launches += 1
    n_img = B * len(fids)
    native_bytes = n_img * NATIVE[0] * NATIVE[1] * 3
    elems = n_img * 3 * sum((H >> s) * (W >> s) for s in range(4))
    bytes_ = native_bytes + elems * (1 + 4)
    return {"config": name, "batch": B, "native": "%dx%d" % (NATIVE[1], NATIVE[0]), "frame_ids": [str(f) for f in fids],
            "gpu_ms": gpu_ms, "launches": launches / N_BATCHES,
            "kernels_us": {k: sum(v) / N_BATCHES for k, v in sorted(kernels.items())},
            "algorithmic_bytes": bytes_, "gbps": bytes_ / (gpu_ms * 1e-3) / 1e9,
            "hbm_share": bytes_ / (gpu_ms * 1e-3) / HBM_BPS, "h2d_ms": h2d_ms,
            "h2d_bytes": natives[0].buffer.numel()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mono_batch_b200.json"))
    ap.add_argument("--reps", type=int, default=50)
    a = ap.parse_args()
    host = {name: host_arm(make_items(fids, 1), H, W) for name, H, W, fids in CONFIGS}    # before CUDA starts: fork
    c = card()
    print("card: %s, power limit %s, max SM clock %s" % (c["name"], c.get("power_limit"), c.get("max_sm_clock")),
          flush=True)
    res = {"card": c, "configs": []}
    for name, H, W, fids in CONFIGS:
        r = gpu_arm(name, H, W, fids, a.reps)
        r["host"] = host[name]
        res["configs"].append(r)
        print(name, "gpu %.4f ms, %d launches, %.0f GB/s, h2d %.3f ms, host %.1f samples/s (1 core) %.1f (%d procs)" % (
            r["gpu_ms"], r["launches"], r["gbps"], r["h2d_ms"], r["host"]["one_core_samples_per_s"],
            r["host"]["pool_samples_per_s"], r["host"]["pool_processes"]), flush=True)
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
