"""KITTI raw depth_gt on one GPU (md2_velo_depth) against the reference's host chain, measured.

    python benchmarks/velo_depth.py [--out profiles/velo_depth_b200.json] [--reps 50]

Prints the card name, power limit and max SM clock, then one JSON line (also written to --out).  A batch of 12
KITTI-like velodyne sweeps (monodepth2_b200.synthetic.velodyne_scan: 121 600 points each, KITTI's 2011_09_26
calibration, cameras 2 and 3, the five KITTI native sizes, half the samples flipped) -> (12, 1, 375, 1242):

  gpu_ms:        one md2_velo_depth call per batch: CUDA events over replays of one CUDA graph per batch, 8 batches in
                 rotation (their scans, scratch and outputs together exceed the 126 MB L2);
  launches:      kernels of one call, and kernels_us their time in an eager call (torch.profiler, mean over calls);
  h2d_bytes:     the scans and job table copied per batch, against host_depth_gt_bytes, the float32 maps the host chain
                 would copy instead;
  host:          the reference's chain (oracle/kitti_depth.py get_depth: read the scan, project, Counter loop, order-0
                 resize, flip, float32) per sample, on one core and on a process pool over every host core, in
                 samples/s;
  mono_batch_ms: MonoBatch.build for mono [0, -1, 1] at 640x192 from native frames, with and without the velodyne
                 scans in the batch (CUDA graph replays, 4 batches in rotation).

It needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import re
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from benchmarks.amp_step import card, events_ms  # noqa: E402
from monodepth2_b200 import synthetic as S  # noqa: E402
from oracle import kitti_depth as OK  # noqa: E402

B, OUT = 12, (375, 1242)
N_BATCHES = 8


def make_drive(root):
    """One calibration directory per native size, and the samples of N_BATCHES batches: (date, cam, scan file, flip)."""
    samples = []
    for k, shape in enumerate(S.KITTI_NATIVE_SIZES):
        S.write_kitti_calibration(os.path.join(root, "date%d" % k), shape)
    os.makedirs(os.path.join(root, "scans"), exist_ok=True)
    for n in range(N_BATCHES * B):
        path = os.path.join(root, "scans", "%010d.bin" % n)
        S.velodyne_scan(n).tofile(path)
        samples.append(("date%d" % (n % 5), 2 + (n // 5) % 2, path, (n // 2) % 2 == 1))
    return samples


def _host_sample(args):
    """KITTIRAWDataset.get_depth + the float32 conversion of __getitem__, from the files."""
    root, (date, cam, path, flip) = args
    t = time.perf_counter()
    d = OK.generate_depth_map(os.path.join(root, date), path, cam)
    d = OK.resize_nearest(d, OUT)
    if flip:
        d = np.fliplr(d)
    np.expand_dims(d, 0).astype(np.float32)
    return time.perf_counter() - t


def host_arm(root, samples):
    n1 = 24
    t = time.perf_counter()
    for i in range(n1):
        _host_sample((root, samples[i]))
    one = n1 / (time.perf_counter() - t)
    cores = os.cpu_count() or 1
    work = [(root, samples[i % len(samples)]) for i in range(max(4 * cores, 48))]
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_host_sample, work[:cores])                 # start-up
        t = time.perf_counter()
        pool.map(_host_sample, work)
        pooled = len(work) / (time.perf_counter() - t)
    return {"one_core_samples_per_s": one, "pool_samples_per_s": pooled, "pool_processes": cores}


def velo_items(root, samples):
    from monodepth2_b200.kitti_depth import VeloScan, velo_to_image
    out = []
    for date, cam, path, flip in samples:
        P, im_shape = velo_to_image(os.path.join(root, date), cam)
        out.append((VeloScan(np.fromfile(path, np.float32).reshape(-1, 4), P, im_shape), flip))
    return out


def graphed(fn, args_list):
    """One CUDA graph per argument set of ``fn`` (warmed up on a side stream first)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for a in args_list:
            fn(*a)
    torch.cuda.current_stream().wait_stream(side)
    graphs, outs = [], []
    for a in args_list:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            outs.append(fn(*a))
        graphs.append(g)
    for g in graphs:
        g.replay()
    torch.cuda.synchronize()
    return graphs, outs


def gpu_arm(root, samples, reps):
    from monodepth2_b200 import _capi, kitti_depth as KD
    lib = _capi.load_library()
    items = velo_items(root, samples)
    batches = []
    for k in range(N_BATCHES):
        chunk = items[k * B:(k + 1) * B]
        scans = [v for v, _ in chunk]
        scans_off = KD._align(B * KD.VELO_JOB_DTYPE.itemsize)
        buf = torch.empty(scans_off + KD.packed_bytes(scans), dtype=torch.uint8, pin_memory=True)
        KD.pack_jobs(buf.numpy(), 0, scans_off, scans, [f for _, f in chunk], False)
        batches.append((buf, buf.to("cuda")))
    run = lambda buf, flat: KD.run(lib, flat, buf.data_ptr(), 0, B, OUT)
    graphs, outs = graphed(run, batches)
    gpu_ms = min(events_ms(lambda i: graphs[i % N_BATCHES].replay(), reps * N_BATCHES) for _ in range(3))
    h2d_ms = min(events_ms(lambda i: batches[i % N_BATCHES][1].copy_(batches[i % N_BATCHES][0], non_blocking=True),
                           reps) for _ in range(3))
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for buf, flat in batches:
            run(buf, flat)
        torch.cuda.synchronize()
    kernels, launches = {}, 0
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "Memcpy" not in e.name:
            m = re.search(r"(md2_\w+)", e.name)
            kernels.setdefault(m.group(1) if m else e.name.split("(")[0].strip(), []).append(e.device_time)
            launches += 1
    n_points = [int(v.scan.shape[0]) for v, _ in items[:B]]
    return {"batch": B, "points_per_scan": n_points[0], "gpu_ms": gpu_ms, "launches": launches / N_BATCHES,
            "kernels_us": {k: sum(v) / N_BATCHES for k, v in sorted(kernels.items())},
            "h2d_ms": h2d_ms, "h2d_bytes": batches[0][0].numel(), "host_depth_gt_bytes": B * OUT[0] * OUT[1] * 4,
            "scratch_bytes": _scratch_bytes(lib)}


def _scratch_bytes(lib):
    import ctypes as C
    n = C.c_size_t(0)
    lib.md2_velo_depth_scratch_bytes(B, OUT[0], OUT[1], C.byref(n))
    return n.value


def mono_batch_arm(root, samples, reps):
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    fids = [0, -1, 1]
    items = velo_items(root, samples)
    res = {}
    for with_depth in (False, True):
        natives = []
        for k in range(4):
            rng = np.random.default_rng(k)
            its = []
            for b in range(B):
                v, flip = items[k * B + b]
                it = {"frames": {f: rng.integers(0, 256, (375, 1242, 3), dtype=np.uint8) for f in fids},
                      "do_color_aug": False, "do_flip": flip, "color_aug": None, "side": "l"}
                if with_depth:
                    it["velodyne"] = v
                its.append(it)
            natives.append(collate_native(its, pin_memory=True))
        mb = MonoBatch(192, 640, fids, 4)
        flats = [mb.upload(nb) for nb in natives]
        graphs, _ = graphed(mb.build, list(zip(natives, flats)))
        ms = min(events_ms(lambda i: graphs[i % 4].replay(), reps * 4) for _ in range(3))
        res["with_depth" if with_depth else "without_depth"] = {"gpu_ms": ms, "h2d_bytes": natives[0].buffer.numel()}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "velo_depth_b200.json"))
    ap.add_argument("--reps", type=int, default=50)
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as root:
        samples = make_drive(root)
        host = host_arm(root, samples)                       # before CUDA starts: fork
        c = card()
        print("card: %s, power limit %s, max SM clock %s" % (c["name"], c.get("power_limit"), c.get("max_sm_clock")),
              flush=True)
        r = gpu_arm(root, samples, a.reps)
        r["host"] = host
        r["mono_batch_ms"] = mono_batch_arm(root, samples, a.reps)
    res = {"card": c, "velo_depth": r}
    print("gpu %.4f ms / batch of %d, %d launches, h2d %d B (maps: %d B), host %.1f samples/s (1 core) %.1f (%d procs); "
          "MonoBatch %.4f ms without depth, %.4f ms with" % (
              r["gpu_ms"], B, r["launches"], r["h2d_bytes"], r["host_depth_gt_bytes"],
              host["one_core_samples_per_s"], host["pool_samples_per_s"], host["pool_processes"],
              r["mono_batch_ms"]["without_depth"]["gpu_ms"], r["mono_batch_ms"]["with_depth"]["gpu_ms"]), flush=True)
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
