"""Mixed precision on one GPU: what bf16 leaves cost and gain, measured.

    python benchmarks/amp_step.py [--out FILE] [--rounds 5] [--steps 20]

Prints the card name and power limit, then one JSON line (also written to --out).  Three legs:

  (a) "loss": the public call view_synthesis_loss(plan, inputs, outputs) + backward() at 640x192, batch 12,
      frame_ids 0 -1 1, 4 scales - float32 leaves against bfloat16 leaves (the disparities and cam_T_cam rounded to
      bf16, the same values in both arms), one CUDA graph per rotating batch, 4 rotating batches of ~110 MB together
      larger than the 126 MB L2, the two arms alternated round by round.  The difference is the cost of the
      conversion pass (md2_widen) plus the typed gradient scaling.
  (b) "head": DispConvSigmoid forward + backward (grad_x, grad_weight, grad_bias) at the four decoder scales of batch
      12, float32 against bfloat16 feature maps, CUDA-graph replayed over 3 rotating inputs; GB/s on the algorithmic
      bytes (x read three times, grad_x written once, disp / grad_disp planes).
  (c) "train": the stand-in training step (benchmarks/train_step.Nets, pose leaves straight into the fused loss,
      Adam) at 640x192, batch 12, float32 against torch.autocast(dtype=torch.bfloat16); ms per step.

Times are CUDA-event times; each arm's figure is the median over rounds.  It needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B, H, W, FIDS = 12, 192, 640, [0, -1, 1]


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                       "-i", str(torch.cuda.current_device())], text=True).strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:         # the name from torch at least
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % e}


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def graph_of(fn):
    """Warm ``fn`` up on a side stream, then capture it once."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


# ------------------------------------------------------------------------------ (a) the public call
def leg_loss(rounds, steps):
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    from monodepth2_b200.synthetic import make_batch
    dev = torch.device("cuda")
    plan = LossPlan(B, H, W, FIDS)
    nrot = 4
    torch.manual_seed(0)
    arms = {torch.float32: [], torch.bfloat16: []}
    keep = []          # a graph reads the tensors it was captured on: they must outlive it
    for i in range(nrot):
        inputs, outputs, _, _ = make_batch(B, H, W, FIDS, 4, seed=i, kind="iid")
        ins = {k: v.to(dev) for k, v in inputs.items()}
        narrow = {k: v.to(dev, torch.bfloat16) for k, v in outputs.items()}      # the same values in both arms
        for dt in arms:
            leaves = {k: v.to(dt).requires_grad_(True) for k, v in narrow.items()}

            def run(leaves=leaves, ins=ins):
                for v in leaves.values():
                    v.grad = None
                view_synthesis_loss(plan, ins, dict(leaves))["loss"].backward()
            arms[dt].append(graph_of(run))
            keep.append((ins, leaves))
    ms = {dt: [] for dt in arms}
    for r in range(rounds):
        for dt in arms:
            for i in range(3):
                arms[dt][i % nrot].replay()
            ms[dt].append(events_ms(lambda i: arms[dt][i % nrot].replay(), steps))
    f32, bf16 = statistics.median(ms[torch.float32]), statistics.median(ms[torch.bfloat16])
    return {"what": "view_synthesis_loss + backward, %dx%d batch %d, frame_ids 0 -1 1, CUDA-graph replay, %d rotating "
                    "batches" % (W, H, B, nrot),
            "ms_f32": f32, "ms_bf16": bf16, "bf16_minus_f32_us": (bf16 - f32) * 1e3,
            "rounds_f32": ms[torch.float32], "rounds_bf16": ms[torch.bfloat16]}


# ------------------------------------------------------------------------------ (b) the disparity head
HEAD_SHAPES = [(12, 16, 192, 640), (12, 32, 96, 320), (12, 64, 48, 160), (12, 128, 24, 80)]


def leg_head(rounds, steps):
    from monodepth2_b200.layers import DispConvSigmoid
    out = []
    for (b, c, h, w) in HEAD_SHAPES:
        torch.manual_seed(c)
        head = DispConvSigmoid(c).cuda()
        rec = {"shape": [b, c, h, w]}
        graphs, keep = {}, []
        for dt in (torch.float32, torch.bfloat16):
            gs = []
            for i in range(3):
                x = torch.randn(b, c, h, w, device="cuda").to(dt).requires_grad_(True)
                up = torch.randn(b, 1, h, w, device="cuda").to(dt)

                def run(x=x, up=up):
                    y = head(x)
                    torch.autograd.grad(y, (x, head.conv.weight, head.conv.bias), up)
                gs.append(graph_of(run))
                keep.append((x, up))
            graphs[dt] = gs
        ms = {dt: [] for dt in graphs}
        for r in range(rounds):
            for dt, gs in graphs.items():
                ms[dt].append(events_ms(lambda i: gs[i % 3].replay(), steps))
        for dt, name in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
            e = 4 if dt == torch.float32 else 2
            # forward reads x, writes disp; grad_x pass reads grad_disp + disp, writes grad_x; weight pass reads x,
            # grad_disp, disp (the 9 C + 1 fp32 gradients are negligible)
            nbytes = e * (3 * b * c * h * w + 5 * b * h * w)
            t = statistics.median(ms[dt])
            rec["ms_" + name] = t
            rec["gbps_" + name] = nbytes / (t * 1e-3) / 1e9
            rec["algorithmic_mb_" + name] = nbytes / 1e6
        rec["speedup_bf16"] = rec["ms_f32"] / rec["ms_bf16"]
        out.append(rec)
        del graphs, keep
        torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------ (c) the stand-in training step
def leg_train(rounds, steps):
    from benchmarks.train_step import Nets
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    from monodepth2_b200.synthetic import make_batch
    dev = torch.device("cuda")
    torch.manual_seed(1234)
    nets = Nets(FIDS, 18).to(dev)
    opt = torch.optim.Adam(nets.parameters(), 1e-4)
    plan = LossPlan(B, H, W, FIDS)
    batches = []
    for i in range(2):
        inputs, _, _, _ = make_batch(B, H, W, FIDS, 4, seed=i, kind="structured")
        batches.append({k: v.to(dev) for k, v in inputs.items()})
    torch.backends.cudnn.benchmark = True

    def step(i, amp):
        inputs = batches[i % 2]
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            outputs = nets({f: inputs[("color", f, 0)] for f in FIDS})
            losses = view_synthesis_loss(plan, inputs, outputs)
        opt.zero_grad(set_to_none=True)
        losses["loss"].backward()
        opt.step()
    ms = {False: [], True: []}
    for amp in ms:
        for i in range(3):
            step(i, amp)
    for r in range(rounds):
        for amp in ms:
            step(0, amp)
            ms[amp].append(events_ms(lambda i: step(i, amp), steps))
    f32, bf16 = statistics.median(ms[False]), statistics.median(ms[True])
    return {"what": "stand-in ResNet-18 nets + fused loss (pose leaves) + backward + Adam, %dx%d batch %d, eager"
                    % (W, H, B),
            "ms_f32": f32, "ms_autocast_bf16": bf16, "speedup": f32 / bf16,
            "rounds_f32": ms[False], "rounds_autocast_bf16": ms[True]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("amp_step.py needs a CUDA device")
    c = card()
    print("card: %s, power limit %s" % (c["name"], c.get("power_limit")), flush=True)
    line = {"benchmark": "amp_step", "card": c, "torch": torch.__version__, "tf32": torch.backends.cuda.matmul.allow_tf32}
    line["loss"] = leg_loss(args.rounds, args.steps)
    torch.cuda.empty_cache()
    line["head"] = leg_head(args.rounds, args.steps)
    torch.cuda.empty_cache()
    line["train"] = leg_train(args.rounds, max(5, args.steps // 2))
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
