"""The training frames' PNG decode on one GPU (md2_png_decode) against Pillow on the host, measured.

    python benchmarks/png_decode.py [--out profiles/png_decode_b200.json] [--reps 30]

Prints the card name, power limit and max SM clock, then one JSON line (also written to --out).  A batch is 36
KITTI-size frames (mono [0, -1, 1] x 12 samples; the five native sizes; synthetic camera-like content with noise,
saved by Pillow at its default compress_level 6, as KITTI's own PNGs are zlib streams of that kind):

  gpu_ms:         one md2_png_decode call per batch: CUDA events over replays of one CUDA graph per batch, 8 batches in
                  rotation (their streams, scratch and frames together exceed the 126 MB L2);
  kernels_us:     each kernel's time in eager calls (torch.profiler, mean per batch);
  h2d:            bytes and time of the packed batch's host-to-device copy, compressed against native frames;
  mono_batch_ms:  MonoBatch.build for mono 640x192 from PNG items against native-frame items (graph replays);
  host:           Pillow's decode (pil_loader) in frames/s on one core and on a process pool over every host core.

It needs a CUDA device.
"""
from __future__ import annotations

import argparse
import io
import json
import multiprocessing as mp
import os
import re
import sys
import time

import numpy as np
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from benchmarks.amp_step import card, events_ms  # noqa: E402
from benchmarks.velo_depth import graphed  # noqa: E402
from monodepth2_b200 import synthetic as S  # noqa: E402

B, FIDS = 12, [0, -1, 1]
N = B * len(FIDS)
N_BATCHES = 8


def _frame(seed, h, w):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.stack([120 + 90 * np.sin(x / (17.0 + seed % 7) + c) * np.cos(y / 11.0 - c) for c in (0.0, 1.3, 2.6)], -1)
    return np.clip(base + rng.normal(0, 14, (h, w, 3)) + 15, 0, 255).astype(np.uint8)


def make_files():
    """N_BATCHES * N PNG files' bytes."""
    from PIL import Image
    out = []
    for n in range(N_BATCHES * N):
        h, w = S.KITTI_NATIVE_SIZES[n % 5]
        b = io.BytesIO()
        Image.fromarray(_frame(n, h, w)).save(b, "PNG")
        out.append(b.getvalue())
    return out


def _pil(data):
    from PIL import Image
    t = time.perf_counter()
    np.array(Image.open(io.BytesIO(data)).convert("RGB"))
    return time.perf_counter() - t


def host_arm(files):
    n1 = 36
    t = time.perf_counter()
    for d in files[:n1]:
        _pil(d)
    one = n1 / (time.perf_counter() - t)
    cores = os.cpu_count() or 1
    work = [files[i % len(files)] for i in range(max(8 * cores, 72))]
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_pil, work[:cores])
        t = time.perf_counter()
        pool.map(_pil, work)
        pooled = len(work) / (time.perf_counter() - t)
    return {"one_core_frames_per_s": one, "pool_frames_per_s": pooled, "pool_processes": cores}


def gpu_arm(files, reps):
    from monodepth2_b200 import _capi, png as PN
    lib = _capi.load_library()
    batches, caps = [], []
    for k in range(N_BATCHES):
        streams = [PN.parse_png(d) for d in files[k * N:(k + 1) * N]]
        outs, total = [], 0
        for s in streams:
            outs.append(total)
            total = PN._align(total + s.nbytes)
        body = PN._align(N * PN.JOB_DTYPE.itemsize, 64)
        buf = torch.empty(body + PN.body_bytes(streams), dtype=torch.uint8, pin_memory=True)
        sb, rb = PN.pack(buf.numpy(), 0, body, streams, outs)
        caps.append((sb, rb, total))
        batches.append((buf, buf.to("cuda")))
    max_stream, max_raw, native = (max(c[i] for c in caps) for i in range(3))
    frames = [torch.empty(native, dtype=torch.uint8, device="cuda") for _ in range(N_BATCHES)]
    status = torch.empty(N, dtype=torch.int32, device="cuda")

    def run(i):
        buf, flat = batches[i]
        PN.run(lib, flat, buf.data_ptr(), 0, N, frames[i], status, max_stream, max_raw)
        return frames[i]
    graphs, _ = graphed(run, [(i,) for i in range(N_BATCHES)])
    assert not status.any().item()
    want = [np.array(Image.open(io.BytesIO(d)).convert("RGB")) for d in files[:N]]
    got = run(0)
    torch.cuda.synchronize()
    exact = all(np.array_equal(got[o:o + w.size].view(*w.shape).cpu().numpy(), w)
                for o, w in zip([int(j) for j in batches[0][0][:N * PN.JOB_DTYPE.itemsize].numpy()
                                 .view(PN.JOB_DTYPE)["out_offset"]], want))
    gpu_ms = min(events_ms(lambda i: graphs[i % N_BATCHES].replay(), reps * N_BATCHES) for _ in range(3))
    h2d_ms = min(events_ms(lambda i: batches[i % N_BATCHES][1].copy_(batches[i % N_BATCHES][0], non_blocking=True),
                           reps) for _ in range(3))
    native_host = torch.empty(native, dtype=torch.uint8, pin_memory=True)
    native_dev = torch.empty(native, dtype=torch.uint8, device="cuda")
    h2d_native_ms = min(events_ms(lambda i: native_dev.copy_(native_host, non_blocking=True), reps) for _ in range(3))
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(N_BATCHES):
            run(i)
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            m = re.search(r"(md2_\w+)", e.name)
            kernels.setdefault(m.group(1) if m else e.name.split("(")[0].strip(), []).append(e.device_time)
    comp = [len(d) for d in files]
    return {"frames": N, "compress_level": 6, "compressed_bytes_per_frame_mean": float(np.mean(comp)),
            "compressed_bytes_per_frame_min": min(comp), "compressed_bytes_per_frame_max": max(comp),
            "byte_exact_with_pillow": exact, "gpu_ms": gpu_ms,
            "kernels_us": {k: sum(v) / N_BATCHES for k, v in sorted(kernels.items())},
            "h2d_bytes": batches[0][0].numel(), "h2d_ms": h2d_ms, "h2d_native_bytes": native,
            "h2d_native_ms": h2d_native_ms, "capacity_stream_bytes": max_stream, "capacity_raw_bytes": max_raw}


def mono_batch_arm(files, reps):
    from monodepth2_b200 import png as PN
    from monodepth2_b200.mono_batch import MonoBatch, collate_native
    res = {}
    for kind in ("native", "png"):
        natives = []
        for k in range(4):
            its = []
            for b in range(B):
                fr = {}
                for fi, f in enumerate(FIDS):
                    d = files[k * N + fi * B + b]
                    s = PN.parse_png(d)
                    fr[f] = s if kind == "png" else np.array(Image.open(io.BytesIO(d)).convert("RGB"))
                its.append({"frames": fr, "do_color_aug": b % 2 == 0, "do_flip": b % 3 == 0,
                            "color_aug": None, "side": "l"})
            natives.append(collate_native(its, pin_memory=True))
        cap = None
        if kind == "png":
            cap = tuple(max(v) for v in zip(*[(n.native_bytes, n.png_stream_bytes, n.png_raw_bytes) for n in natives]))
        mb = MonoBatch(192, 640, FIDS, 4, png_capacity=cap)
        flats = [mb.upload(nb) for nb in natives]
        graphs, _ = graphed(mb.build, list(zip(natives, flats)))
        ms = min(events_ms(lambda i: graphs[i % 4].replay(), reps * 4) for _ in range(3))
        h2d = min(events_ms(lambda i: flats[i % 4].copy_(natives[i % 4].buffer, non_blocking=True), reps)
                  for _ in range(3))
        res[kind] = {"gpu_ms": ms, "h2d_bytes": natives[0].buffer.numel(), "h2d_ms": h2d}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "png_decode_b200.json"))
    ap.add_argument("--reps", type=int, default=30)
    a = ap.parse_args()
    files = make_files()
    host = host_arm(files)                                   # before CUDA starts: fork
    c = card()
    print("card: %s, power limit %s, max SM clock %s" % (c["name"], c.get("power_limit"), c.get("max_sm_clock")),
          flush=True)
    r = gpu_arm(files, a.reps)
    r["host"] = host
    r["mono_batch"] = mono_batch_arm(files, a.reps)
    line = json.dumps({"card": c, "png_decode": r})
    print("decode %.4f ms / %d frames (%s); h2d %d B %.4f ms vs native %d B %.4f ms; Pillow %.1f frames/s (1 core), "
          "%.1f (%d procs); MonoBatch %.4f ms (native) %.4f ms (png)" % (
              r["gpu_ms"], N, r["kernels_us"], r["h2d_bytes"], r["h2d_ms"], r["h2d_native_bytes"], r["h2d_native_ms"],
              host["one_core_frames_per_s"], host["pool_frames_per_s"], host["pool_processes"],
              r["mono_batch"]["native"]["gpu_ms"], r["mono_batch"]["png"]["gpu_ms"]), flush=True)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
