#!/usr/bin/env python
"""Benchmark of the fused view-synthesis loss (BASELINE.json metric: reproj-loss fwd+bwd frames/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

Own arm: a "step" is one md2_view_synthesis_loss call (generate_images_pred + compute_losses +
the adjoint to the 4 disparities and the poses) over one synthetic batch of 12 frames per GPU,
inputs resident in HBM; N GPUs = N independent shards of the batch dimension (no data-path
collective, SURVEY.md 8e), time = max over ranks of the CUDA-event duration of K steps.
Reference arm (--impl reference): the CPU restatement of the reference's own PyTorch path
(oracle/view_synthesis.py = the reference's --no_cuda path) on the box's host cores.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

# stdout carries exactly ONE line, the JSON result: everything else that libraries print on fd 1 (e.g. the
# "NCCL version ..." banner) is sent to stderr while the benchmark runs
_RESULT_FD = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


WORKLOADS = {
    # name: (H, W, frame_ids, avg_reprojection, disable_automasking)
    "mono_640x192_b12": (192, 640, [0, -1, 1], False, False),
    "mono+stereo_640x192_b12": (192, 640, [0, -1, 1, "s"], False, False),
    "mono_1024x320_b12": (320, 1024, [0, -1, 1], False, False),
    "mono_640x192_b12_avg_reprojection": (192, 640, [0, -1, 1], True, False),
    "mono_640x192_b12_disable_automasking": (192, 640, [0, -1, 1], False, True),
}
BATCH = 12
L2_NOTE = "GPU arm: 4 rotating batches of ~110 MB each, together larger than the 126 MB L2 (no flush); the reference arm runs on the CPU"
METRIC = "reproj-loss fwd+bwd frames/s"
UNIT = "frames/s"


def algorithmic_bytes(B, H, W, n_src, n_id, S=4):
    """A_alg of SURVEY.md 8(d): compulsory reads/writes of one batch, loss fwd+bwd."""
    tot = 0
    for s in range(S):
        hw, hsws = H * W, (H >> s) * (W >> s)
        fwd = 3 * hw + 3 * n_src * hw + hsws + (3 * hsws if s > 0 else 0) + n_id * hw
        bwd = 3 * hw + 3 * n_src * hw + hsws + (3 * hsws if s > 0 else 0) + hsws
        tot += fwd + bwd
    return 4 * B * tot


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.001)      # (the default timed region is ~25 ms)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------- reference arm
def oracle_step(B, H, W, frame_ids, avg, noauto, batch, threads, device=None):
    """One fwd+bwd of the reference path (oracle port).  device=None: CPU, wall clock;
    device=cuda: the same code on torch's CUDA kernels (the reference's PyTorch-CUDA path), the
    batch must already be resident on the device."""
    from oracle import view_synthesis as O
    inputs, outputs, pose, noise = batch
    cfg = O.OracleConfig(height=H, width=W, frame_ids=tuple(frame_ids), avg_reprojection=avg,
                         disable_automasking=noauto)
    outs = {}
    leaves = []
    for s in range(4):
        d = outputs[("disp", s)][:B].clone().requires_grad_(True)
        outs[("disp", s)] = d
        leaves.append(d)
    for f, (aa, tr) in pose.items():
        a = aa[:B].reshape(B, 1, 3).clone().requires_grad_(True)
        t = tr[:B].reshape(B, 1, 3).clone().requires_grad_(True)
        leaves += [a, t]
        outs[("cam_T_cam", 0, f)] = O.transformation_from_parameters(a, t, invert=(f < 0))
    ins = {k: v[:B] for k, v in inputs.items()}
    nz = [n[:B] for n in noise] if noise is not None else None
    if device is not None:
        torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    losses = O.view_synthesis_loss(ins, outs, cfg, nz)
    losses["loss"].backward()
    if device is not None:
        torch.cuda.synchronize(device)
    return time.perf_counter() - t0, float(losses["loss"].detach())


def batch_to(batch, dev):
    inputs, outputs, pose, noise = batch
    return ({k: v.to(dev) for k, v in inputs.items()}, {k: v.to(dev) for k, v in outputs.items()},
            {f: (a.to(dev), t.to(dev)) for f, (a, t) in pose.items()},
            [n.to(dev) for n in noise] if noise is not None else None)


def torch_cuda_baseline(H, W, frame_ids, avg, noauto, batch, dev, reps=10):
    """The reference's PyTorch-CUDA path (BASELINE.json configs[1]: "vs the reference's PyTorch CUDA
    path"): the oracle port on torch's stock CUDA kernels, full batch, inputs resident in HBM."""
    db = batch_to(batch, dev)
    for _ in range(3):
        oracle_step(BATCH, H, W, frame_ids, avg, noauto, db, 0, dev)
    ts = [oracle_step(BATCH, H, W, frame_ids, avg, noauto, db, 0, dev)[0] for _ in range(reps)]
    ts.sort()
    med = ts[len(ts) // 2]
    return {"value": BATCH / med, "unit": UNIT, "ms_per_step": 1e3 * med, "best_ms": 1e3 * ts[0],
            "kind": "port on torch CUDA kernels (oracle/view_synthesis.py, ~2.1k ATen launches per step)",
            "sample": "%d full batches of %d frames, fwd+bwd, median" % (reps, BATCH)}


def run_reference(args, wl):
    """The reference's CPU implementation of the path (oracle port), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from monodepth2_b200.synthetic import make_batch
    H, W, frame_ids, avg, noauto = WORKLOADS[wl]
    n_src = len(frame_ids) - 1
    n_id = 0 if noauto else (1 if avg else n_src)
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    batch = make_batch(BATCH, H, W, frame_ids, 4, 0, "iid", n_id=max(n_id, 1))
    if n_id == 0:
        batch = (batch[0], batch[1], batch[2], None)
    # size the per-step sample so that (K+W) steps finish in a few minutes
    # (probe after one untimed call: the first call pays torch's one-off initialisation and would make the
    # sample - and with it the reference's frames/s - smaller than the host can sustain)
    oracle_step(1, H, W, frame_ids, avg, noauto, batch, threads)
    t_probe = min(oracle_step(1, H, W, frame_ids, avg, noauto, batch, threads)[0] for _ in range(2))
    budget = 150.0 / max(1, args.steps + args.warmup)
    Bs = int(max(1, min(BATCH, budget / max(t_probe, 1e-3))))
    for _ in range(args.warmup):
        oracle_step(Bs, H, W, frame_ids, avg, noauto, batch, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_step(Bs, H, W, frame_ids, avg, noauto, batch, threads)
    dt = time.perf_counter() - t0
    fps = Bs * args.steps / dt
    sample = "%d of %d frames of the batch per step, %d steps" % (Bs, BATCH, args.steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": wl, "batch_per_gpu": BATCH, "frame_ids": [str(f) for f in frame_ids], "scales": 4,
                   "l2": L2_NOTE},
        "notes": {"device": "cpu (reference --no_cuda path, oracle port: oracle/view_synthesis.py)"},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------- own arm
class DeviceBatch:
    """One synthetic batch resident in HBM plus the prebuilt C-ABI argument block."""

    def __init__(self, plan, batch, dev):
        from monodepth2_b200._capi import Md2Tensors, MAX_SCALES
        inputs, outputs, pose, noise = batch
        self.keep = []
        self.noise = []
        t = Md2Tensors()

        def put(x):
            x = x.to(dev).contiguous()
            self.keep.append(x)
            return x.data_ptr()

        B, H, W = plan.batch_size, plan.height, plan.width
        t.target = put(inputs[("color", 0, 0)])
        for i, f in enumerate(plan.src_ids):
            t.source[i] = put(inputs[("color", f, 0)])
            if f == "s":
                t.T[i] = put(inputs["stereo_T"])
                t.pose_requires_grad[i] = 0
            else:
                t.T[i] = put(outputs[("cam_T_cam", 0, f)])
                t.pose_requires_grad[i] = 1
            g = torch.empty((B, 4, 4), device=dev)
            self.keep.append(g)
            t.grad_T[i] = g.data_ptr()
        t.K = put(inputs[("K", 0)])
        t.inv_K = put(inputs[("inv_K", 0)])
        self.grad_disp = []
        for s in range(4):
            t.disp[s] = put(outputs[("disp", s)])
            t.color[s] = put(inputs[("color", 0, s)])
            if plan.n_id > 0:
                t.noise[s] = put(noise[s])
                self.noise.append(self.keep[-1])
            g = torch.empty((B, 1, H >> s, W >> s), device=dev)
            self.grad_disp.append(g)
            t.grad_disp[s] = g.data_ptr()
        self.losses = torch.zeros(MAX_SCALES + 1, device=dev)
        t.losses = self.losses.data_ptr()
        self.t = t


class PublicStep:
    """One rotating batch driven through the PUBLIC call: view_synthesis_loss(plan, inputs, outputs) with the
    tie-break noise drawn inside (torch.randn, trainer.py:468-469) + losses["loss"].backward() through the
    autograd wrapper, captured once in a CUDA graph and replayed (tests/test_gpu_parity.py shows capture
    replays identically)."""

    def __init__(self, plan, batch, dev):
        from monodepth2_b200.fused_loss import view_synthesis_loss
        inputs, outputs, pose, noise = batch
        self.plan, self.fn = plan, view_synthesis_loss
        self.ins = {k: v.to(dev) for k, v in inputs.items()}
        self.leaves = {k: v.to(dev).requires_grad_(True) for k, v in outputs.items()}
        self.graph, self.loss = None, None

    def run(self):
        for v in self.leaves.values():
            v.grad = None
        losses = self.fn(self.plan, self.ins, dict(self.leaves))
        losses["loss"].backward()
        self.losses = {k: v.detach() for k, v in losses.items()}
        return self.losses["loss"]

    def results(self):
        """What a caller of the public call receives from the last step: the losses dict and the gradients of the
        disparity and pose leaves, by file-name-safe names."""
        out = {k.replace("/", "_"): v for k, v in self.losses.items()}
        for k, v in self.leaves.items():
            out["grad_" + "_".join(str(x) for x in k)] = v.grad
        return out

    def capture(self):
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(2):
                self.run()
        cur.wait_stream(side)
        torch.cuda.synchronize()
        for v in self.leaves.values():
            v.grad = None
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = self.run()

    def step(self):
        if self.graph is not None:
            self.graph.replay()
        else:
            self.loss = self.run()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(arrays, out_dir):
    """Writes every array as <out_dir>/<name>.npy in float32, so that two builds can be compared output for output."""
    import numpy as np
    host = {name: t.detach().float().cpu().numpy() for name, t in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def quantise_u8(x):
    """float frame in [0,1] -> the uint8 frame a dataloader holds before ToTensor, interleaved (B,H,W,3)"""
    return (x * 255.0).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()


def run_own(args, wl):
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    from monodepth2_b200.synthetic import make_batch
    from monodepth2_b200 import _capi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the fused loss has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one process per GPU: stay on the CPUs next to this GPU, so that the pinned staging buffers of the e2e leg sit on
    # its NUMA node (at 8 GPUs the copies otherwise share the socket interconnect: e2e efficiency 0.53)
    from monodepth2_b200.fused_loss import bind_to_gpu_cpus
    numa_cpus = bind_to_gpu_cpus(dev) if os.environ.get("MD2_BENCH_BIND", "1") != "0" else None
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    H, W, frame_ids, avg, noauto = WORKLOADS[wl]
    plan = LossPlan(BATCH, H, W, frame_ids, avg_reprojection=avg, disable_automasking=noauto,
                    rows_per_segment=args.rows)
    lib = plan.lib
    n_src, n_id = plan.n_src, plan.n_id
    nrot = 4        # rotating batches: ~110 MB each, together larger than the 126 MB L2
    host = [make_batch(BATCH, H, W, frame_ids, 4, seed=1000 * rank + i, kind="iid", n_id=max(n_id, 1))
            for i in range(nrot)]
    stream = torch.cuda.current_stream()
    sptr = C.c_void_p(stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps, warmup, sample_clocks=False):
        """warm-up, barrier, K steps between CUDA events on the launching stream, max over ranks"""
        for i in range(warmup):
            step_fn(i)
        barrier()
        sampler = None
        if sample_clocks:
            sampler = ClockSampler(local)
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            step_fn(i)
        e1.record(stream)
        barrier()
        clocks = sampler.stop() if sampler else None
        tt = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item()), clocks

    # ---- value: the public call (noise drawn inside, autograd wrapper and backward() included), inputs resident
    # in HBM, one CUDA graph per rotating batch
    # the public call draws its tie-break noise from the default generator: seeded, every run with the same arguments
    # computes on the same inputs
    torch.manual_seed(0)
    pub = [PublicStep(plan, b, dev) for b in host]
    if not args.no_graph:
        for p in pub:
            p.capture()
    ms_total, clocks = timed(lambda i: pub[i % nrot].step(), args.steps, max(args.warmup, 3), sample_clocks=True)
    value = world * BATCH * args.steps / (ms_total * 1e-3)
    loss_val = float(pub[(args.steps - 1) % nrot].loss.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(pub[(args.steps - 1) % nrot].results(), args.dump_outputs)

    # ---- the raw C-ABI call with pre-drawn noise tensors (round 1's headline; kept as an extra key): what the
    # library itself costs without the 4 torch.randn draws and the autograd wrapper
    devb = [DeviceBatch(plan, b, dev) for b in host]
    ws = plan.workspace(dev)
    prob = plan.problem(True)

    def launch(i, stream_ptr):
        st = lib.md2_view_synthesis_loss(C.byref(prob), C.byref(devb[i % nrot].t), ws.data_ptr(), ws.numel(), stream_ptr)
        if st != 0:
            _capi.check(lib, st, "md2_view_synthesis_loss")

    graphs = None
    if not args.no_graph:
        launch(0, sptr)
        torch.cuda.synchronize()
        graphs = []
        for i in range(nrot):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                launch(i, C.c_void_p(torch.cuda.current_stream().cuda_stream))
            graphs.append(g)
    ms_cabi, _ = timed((lambda i: graphs[i % nrot].replay()) if graphs else (lambda i: launch(i, sptr)),
                       args.steps, 3)

    # ---- roofline of the dominant kernel (md2_march_roles): per-launch CUDA events, live
    lib.md2_profile_enable(1)
    march = []
    for i in range(min(args.steps, 20)):
        launch(i, sptr)                       # plain calls: the event pair is recorded by the library
        ms = C.c_float(0)
        lib.md2_profile_march_ms(C.byref(ms))
        march.append(ms.value)
    lib.md2_profile_enable(0)
    march_ms = sum(march) / len(march)
    a_alg = algorithmic_bytes(BATCH, H, W, n_src, n_id)
    peak, peak_src = measured_peak_gbs()
    achieved = a_alg / (march_ms * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "march_traffic.json"))).get(wl)
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "md2_march_roles", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": a_alg, "kernel_ms": march_ms,
                "frac_of_8TBs_nominal": achieved / 8000.0,
                "whole_step_achieved": a_alg / (ms_total / args.steps * 1e-3) / 1e9}

    # ---- e2e: public API through the uint8 entry; every step's inputs are copied from pinned host memory
    # (frames as the uint8 the dataloader holds before ToTensor, mono_dataset.py:106-109; disparities / poses /
    # intrinsics as fp32) and every step's loss is read back
    pinned = []
    for b in host[:2]:
        inputs, outputs, pose, noise = b
        pin_in = {}
        for f in frame_ids:
            pin_in[("color", f, 0)] = quantise_u8(inputs[("color", f, 0)]).pin_memory()
        for s_ in range(1, 4):
            pin_in[("color", 0, s_)] = quantise_u8(inputs[("color", 0, s_)]).pin_memory()
        for k in [("K", 0), ("inv_K", 0)] + (["stereo_T"] if "s" in frame_ids else []):
            pin_in[k] = inputs[k].pin_memory()
        pin_out = {k: v.pin_memory() for k, v in outputs.items()}
        pinned.append((pin_in, pin_out))
    h2d = sum(v.numel() * v.element_size() for v in pinned[0][0].values()) + \
        sum(v.numel() * v.element_size() for v in pinned[0][1].values())

    # Public API: monodepth2_b200.fused_loss.GraphedLoss (the fused call + backward captured in a CUDA graph over
    # static buffers).  Two instances alternate: the H2D copy of step i+1 (copy stream, pinned host -> static buffers)
    # overlaps the compute of step i (what a training input pipeline does); every step's inputs are copied inside the
    # timed region and every step's loss is read back to the host.
    from monodepth2_b200.fused_loss import GraphedLoss
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream()
    graphed = []
    for pin_in, pin_out in pinned:
        graphed.append(GraphedLoss(plan, {k: v.to(dev) for k, v in pin_in.items()}, {k: v.to(dev) for k, v in pin_out.items()}))
    ev_loaded = [torch.cuda.Event() for _ in graphed]
    ev_done = [torch.cuda.Event() for _ in graphed]
    for e in ev_done:
        e.record(main_stream)

    # pinned staging buffers laid out like the static device buffers (GraphedLoss.staging): filled once here (what a
    # dataloader's collate step does per batch), copied to the device EVERY step, one copy per step
    staged = []
    for j, (pin_in, pin_out) in enumerate(pinned):
        flat, s_in, s_out = graphed[j].staging()
        for k, v in pin_in.items():
            s_in[k].copy_(v)
        for k, v in pin_out.items():
            s_out[k].copy_(v)
        staged.append(flat)
    h2d = int(staged[0].numel())          # bytes copied per step (the tensors above + padding to 256-byte boundaries)

    def stage(i):
        j = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_done[j])          # the buffers of instance j are free once its last replay is done
            graphed[j].load_staged(staged[j])
            ev_loaded[j].record(copy_stream)

    def e2e_run(n):
        """Every step: H2D copy of its inputs (copy stream), graph replay, D2H read of its loss.  The read of step i is
        put in flight with the step (pinned slot + event, GraphedLoss.run_async) and collected after step i+1 has been
        enqueued, so the host never drains the GPU between steps; every step's loss reaches the host inside the region."""
        stage(0)
        last = 0.0
        for i in range(n):
            j = i % 2
            stage(i + 1)
            main_stream.wait_event(ev_loaded[j])
            graphed[j].run_async()
            ev_done[j].record(main_stream)
            if i >= 1:
                last = graphed[1 - j].read()              # D2H read of step i-1's result
        last = graphed[(n - 1) % 2].read()
        return last

    # (freshly pinned host buffers copy at a fraction of the PCIe rate for their first few dozen transfers - measured
    # 0.73 ms falling to 0.41 ms per 22.5 MB, scripts/e2e_probe.py - so the warm-up is longer than for the kernels)
    e2e_run(40)
    barrier()
    n_e2e = max(5, min(args.steps, 50))
    t0 = time.perf_counter()
    e2e_run(n_e2e)
    barrier()
    dt = time.perf_counter() - t0
    te = torch.tensor([dt], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e = {"value": world * BATCH * n_e2e / float(te.item()), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": 4, "steps": n_e2e, "pipeline": "GraphedLoss (public API): one H2D copy per step from a pinned staging buffer (GraphedLoss.staging / load_staged) into the static buffers, step i+1's copy overlapping the graph replay of step i; the loss of step i is copied to a pinned host slot with the step and read by the host after step i+1 has been enqueued (GraphedLoss.run_async / read)",
           "entry": "uint8 frames (B,H,W,3) + uint8 target pyramid, converted in-kernel (x/255 = ToTensor); fp32 "
                    "disparities, cam_T_cam, K, inv_K"}

    # ---- CPU baseline (oracle port) on rank 0 at N=1, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        torch.set_num_threads(threads)
        cb = host[0] if n_id > 0 else (host[0][0], host[0][1], host[0][2], None)
        oracle_step(2, H, W, frame_ids, avg, noauto, cb, threads)          # warm-up
        t_used, n_fr, reps = 0.0, 0, 0
        while t_used < 10.0 and reps < 5:
            dt1, _ = oracle_step(BATCH, H, W, frame_ids, avg, noauto, cb, threads)
            t_used += dt1
            n_fr += BATCH
            reps += 1
        cpu = {"value": n_fr / t_used, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "%d full batches of %d frames (oracle/view_synthesis.py, fwd+bwd)" % (reps, BATCH)}

    tcb = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cb = host[0] if n_id > 0 else (host[0][0], host[0][1], host[0][2], None)
        try:
            tcb = torch_cuda_baseline(H, W, frame_ids, avg, noauto, cb, dev)
        except Exception as e:      # a baseline leg must not take the bench line down
            tcb = {"error": repr(e)[:200]}

    # ---- the caller of the path: full training step (nets + loss + backward + Adam, DDP all-reduce at N > 1),
    # so that the per-N records carry a training curve (BASELINE.json: "train steps/s at 1-8 GPUs")
    train = None
    if not args.no_train:
        del pub, devb, graphs
        torch.cuda.empty_cache()
        try:
            train = train_record(args, wl, dev, dist, rank, world, steps=min(args.steps, 10), warmup=3)
        except Exception as e:
            train = {"error": repr(e)[:300]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # `config` names the workload and is identical in both arms; everything about how this arm ran is in `notes`
            "config": {"workload": wl, "batch_per_gpu": BATCH, "frame_ids": [str(f) for f in frame_ids], "scales": 4,
                       "l2": L2_NOTE},
            "notes": {"device": "cuda (B200)", "cpu_affinity": numa_cpus,
                       "rows_per_segment": plan.problem(True).rows_per_segment or "library default (wave-quantisation model)", "loss": loss_val,
                       "launch": ("eager public calls" if args.no_graph else "CUDA-graph replay of the public call") +
                                 ": view_synthesis_loss(plan, inputs, outputs) + losses['loss'].backward(); the 4 "
                                 "torch.randn tie-break draws of trainer.py:468-469 and the autograd wrapper are inside "
                                 "the timed region"},
            "value_cabi_predrawn_noise": world * BATCH * args.steps / (ms_cabi * 1e-3),
            "ms_per_step_cabi_predrawn_noise": ms_cabi / args.steps,
            "roofline": roofline, "cpu_baseline": cpu, "torch_cuda_baseline": tcb, "e2e": e2e,
            "gpu_launches": 9 * args.steps,      # prologue, disp_mean, smooth, smooth_scalars, depth_up, identity, march_roles, final, scale_tensors
            "clocks": clocks,
            "train": train,
        }
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------- full training step
def train_record(args, wl, dev, dist, rank, world, steps, warmup, impl="own", num_layers=18):
    """nets + loss + backward + Adam (+ DDP all-reduce), batch 12 per GPU, synthetic batches resident in HBM
    (SURVEY.md 8d(3), 8e; the caller is Trainer.run_epoch / process_batch, trainer.py:193-260).  Returns the
    record; the max over ranks of the CUDA-event time is taken like for the loss path."""
    import contextlib
    from benchmarks.train_step import Nets, TrainStep, parameter_count
    from monodepth2_b200.synthetic import make_batch

    H, W, frame_ids, avg, noauto = WORKLOADS[wl]
    torch.manual_seed(1234)                         # identical initial weights on every rank
    nets = Nets(frame_ids, num_layers).to(dev)
    n_params = parameter_count(nets)
    model = nets
    if world > 1:
        from torch.nn.parallel import DistributedDataParallel as DDP
        model = DDP(nets, device_ids=[dev.index], gradient_as_bucket_view=True, bucket_cap_mb=args.bucket_mb,
                    static_graph=True)

    if impl == "reference":
        from oracle import view_synthesis as O
        cfg = O.OracleConfig(height=H, width=W, frame_ids=tuple(frame_ids), avg_reprojection=avg,
                             disable_automasking=noauto)

        def loss_fn(inputs, outputs):
            return O.view_synthesis_loss(inputs, outputs, cfg, None)
        pose_fn = O.transformation_from_parameters
        loss_name = "reference PyTorch-CUDA loss path (oracle port)"
    else:
        from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
        pose_fn = None          # the fused call takes the pose leaves and builds cam_T_cam itself
        plan = LossPlan(BATCH, H, W, frame_ids, avg_reprojection=avg, disable_automasking=noauto)

        def loss_fn(inputs, outputs):
            return view_synthesis_loss(plan, inputs, outputs)
        loss_name = "fused md2_view_synthesis_loss"

    nrot = 2
    batches = []
    for i in range(nrot):
        inputs, _, _, _ = make_batch(BATCH, H, W, frame_ids, 4, seed=1000 * rank + i, kind="structured")
        batches.append({k: v.to(dev) for k, v in inputs.items()})
    step = TrainStep(model, frame_ids, loss_fn, pose_fn)
    torch.backends.cudnn.benchmark = True

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run(n, w, ctx):
        with ctx():
            for i in range(w):
                step(batches[i % nrot])
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            loss = None
            for i in range(n):
                loss = step(batches[i % nrot])
            e1.record()
            barrier()
        tt = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item()) / n, loss

    sampler = ClockSampler(dev.index)
    sampler.start()
    ms, loss = run(steps, max(warmup, 3), contextlib.nullcontext)
    clocks = sampler.stop()
    rec = {
        "impl": impl, "metric": "train steps/s (nets + view-synthesis loss + backward + Adam)",
        "value": 1e3 / ms, "unit": "steps/s", "n_gpus": world, "steps": steps, "ms_per_step": ms,
        "frames_per_s": world * BATCH * 1e3 / ms, "gradient_bytes": n_params * 4,
        "config": {"workload": wl, "mode": "train", "batch_per_gpu": BATCH, "global_batch": world * BATCH,
                   "frame_ids": [str(f) for f in frame_ids], "scales": 4,
                   "nets": "stand-in ResNet-%d encoder + depth decoder + pose encoder/decoder, %.2f M params, "
                           "random init, fp32 (TF32 off)" % (num_layers, n_params / 1e6),
                   "loss": loss_name, "parallelism": ("ddp%d (NCCL all-reduce of %.1f MB of gradients, bucket_cap_mb=%d, "
                                                      "static_graph, gradient_as_bucket_view)" %
                                                      (world, n_params * 4 / 1e6, args.bucket_mb)) if world > 1 else "single GPU",
                   "last_loss": float(loss.item())},
        "clocks": clocks,
    }
    if world > 1:
        # the same step without the gradient all-reduce (DDP no_sync): what the collective leaves exposed
        ms_local, _ = run(steps, 2, model.no_sync)
        rec["ms_per_step_no_allreduce"] = ms_local
        rec["exposed_allreduce_ms"] = ms - ms_local
    return rec


def run_train(args, wl):
    """--mode train: the training-step record alone (--impl own: fused loss; --impl reference: the reference's
    PyTorch-CUDA loss path in the same harness)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --mode train needs a CUDA device")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    rec = train_record(args, wl, dev, dist, rank, world, args.steps, args.warmup, args.impl, args.num_layers)
    if rank == 0:
        rec.update({"warmup": max(args.warmup, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                    "dtype": "f32", "data": "synthetic"})
        emit(rec)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--workload", default="mono_640x192_b12", choices=sorted(WORKLOADS))
    ap.add_argument("--rows", type=int, default=0, help="rows per marching segment (0 = library default)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-graph", action="store_true", help="plain C-ABI calls instead of CUDA-graph replay")
    ap.add_argument("--mode", default="loss", choices=["loss", "train"],
                    help="loss: the hot path alone (the contract metric); train: the full training step around it")
    ap.add_argument("--num-layers", type=int, default=18, choices=[18, 50], help="--mode train: ResNet depth")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step sub-record of the default mode")
    ap.add_argument("--bucket-mb", type=int, default=25, help="DDP bucket_cap_mb of the training-step record")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="fused loss path only (--impl own --mode loss): write the losses and gradients of the last "
                         "timed step of the public call as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.mode == "train" or args.impl == "reference"):
        ap.error("--dump-outputs applies to the fused loss path (--impl own --mode loss)")
    if args.mode == "train":
        run_train(args, args.workload)
    elif args.impl == "reference":
        run_reference(args, args.workload)
    else:
        run_own(args, args.workload)


if __name__ == "__main__":
    main()
