"""The fused decoder stages on one GPU: upcat_pad against torch's upsample + cat + ReflectionPad2d chain, measured.

    python benchmarks/decoder_stages.py [--out profiles/decoder_stages_b200.json] [--rounds 5] [--steps 20]

Prints the card name, power limit and max SM clock, then one JSON line (also written to --out).  Two legs:

  (a) "producers": each of the 10 ConvBlock inputs of the reference DepthDecoder (networks/depth_decoder.py:48-65) at
      640x192, batch 12, ResNet-18 and ResNet-50 encoder channels, fp32 and bf16 - forward upcat_pad(x, skip, up)
      against F.pad(torch.cat([F.interpolate(x, scale_factor=2), skip], 1), reflect), and the backward of each
      (torch.autograd.grad of the retained graph, so torch's arm is exactly what autograd runs: reflection_pad2d_backward
      with its zero fill and atomics, the cat slice, upsample_nearest2d_backward).  Each arm is one CUDA graph of n calls
      on n rotating input sets of together more than 256 MB (twice the 126 MB L2), replayed; time per call = replay
      time / n.  GB/s on algorithmic bytes: forward reads x and skip and writes out, backward reads grad_out and writes
      grad_x and grad_skip; "hbm_share" is that rate over 7.7 TB/s.
  (b) "decoder": the whole reference DepthDecoder forward + backward (parameter and feature gradients) from fixed
      encoder features at 640x192, batch 12, fused stages (fuse_decoder_stages) against unfused, disparity heads fused
      (fuse_disp_heads) in both arms; fp32 and torch.autocast(dtype=torch.bfloat16); eager, cudnn.benchmark on.  The
      two arms alternate round by round; each figure is the median over rounds of CUDA-event times.

It needs a CUDA device.
"""
from __future__ import annotations

import argparse
import copy
import json
import math
import os
import statistics
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from benchmarks.amp_step import card, events_ms  # noqa: E402

B, H, W = 12, 192, 640
ENC = {18: [64, 64, 128, 256, 512], 50: [64, 256, 512, 1024, 2048]}
DEC = [16, 32, 64, 128, 256]
HBM_BPS = 7.7e12
ROTATE_BYTES = 256e6


def block_inputs(layers):
    enc, out = ENC[layers], []
    for i in range(4, -1, -1):
        h, w = H >> (i + 1), W >> (i + 1)
        out.append(("upconv_%d_0" % i, enc[-1] if i == 4 else DEC[i + 1], 0, h, w, 1))
        out.append(("upconv_%d_1" % i, DEC[i], enc[i - 1] if i > 0 else 0, h, w, 2))
    return out


def torch_chain(x, skip, up):
    y = F.interpolate(x, scale_factor=2, mode="nearest") if up == 2 else x
    if skip is not None:
        y = torch.cat([y, skip], 1)
    return F.pad(y, (1, 1, 1, 1), mode="reflect")


_side = []


def side_stream():
    """The stream that runs every captured forward and backward: autograd runs a backward node on the stream of its
    forward, so the retained forwards of leg (a) must come from the capturing stream."""
    if not _side:
        _side.append(torch.cuda.Stream())
    return _side[0]


def captured(fn, n):
    """One CUDA graph running fn(0) .. fn(n-1) (warmed up first on the capturing stream)."""
    s = side_stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(min(n, 2)):
            fn(i)
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        for i in range(n):
            fn(i)
    torch.cuda.current_stream().wait_stream(s)
    return g


# ------------------------------------------------------------------------------------------------ (a) producers
def leg_producers(rounds, steps):
    from monodepth2_b200.layers import upcat_pad
    arms = {"fused": upcat_pad, "torch": torch_chain}
    recs = []
    for layers in (18, 50):
        for dt, dname in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
            e = torch.finfo(dt).bits // 8
            for name, cx, cs, h, w, up in block_inputs(layers):
                n_x, n_s = B * cx * h * w, B * cs * up * h * up * w
                n_o = B * (cx + cs) * (up * h + 2) * (up * w + 2)
                fwd_bytes = e * (n_x + n_s + n_o)
                bwd_bytes = e * (n_o + n_x + n_s)
                nrot = max(2, min(128, math.ceil(ROTATE_BYTES / fwd_bytes)))
                torch.manual_seed(0)
                sets = []
                for i in range(nrot):
                    x = torch.randn(B, cx, h, w, device="cuda").to(dt).requires_grad_(True)
                    skip = torch.randn(B, cs, up * h, up * w, device="cuda").to(dt).requires_grad_(True) if cs else None
                    sets.append((x, skip, torch.randn(n_o, device="cuda").to(dt).view(B, cx + cs, up * h + 2, up * w + 2)))
                graphs, keep = {}, []
                for arm, f in arms.items():
                    graphs[(arm, "fwd")] = captured(lambda i, f=f: f(sets[i][0], sets[i][1], up), nrot)
                    with torch.cuda.stream(side_stream()):
                        outs = [f(x, s, up) for x, s, _ in sets]
                    side_stream().synchronize()
                    keep.append(outs)

                    def bwd(i, outs=outs):
                        x, s, g = sets[i]
                        torch.autograd.grad(outs[i], (x, s) if s is not None else (x,), g, retain_graph=True)
                    graphs[(arm, "bwd")] = captured(bwd, nrot)
                ms = {k: [] for k in graphs}
                for r in range(rounds):
                    for k, gr in graphs.items():
                        gr.replay()
                        ms[k].append(events_ms(lambda i, gr=gr: gr.replay(), steps) / nrot)
                rec = {"encoder": "resnet%d" % layers, "dtype": dname, "block": name, "x": [B, cx, h, w],
                       "skip_channels": cs, "up": up, "rotating_sets": nrot,
                       "fwd_mb": fwd_bytes / 1e6, "bwd_mb": bwd_bytes / 1e6}
                for (arm, d), v in ms.items():
                    t = statistics.median(v)
                    nbytes = fwd_bytes if d == "fwd" else bwd_bytes
                    rec["%s_%s_us" % (arm, d)] = t * 1e3
                    rec["%s_%s_gbps" % (arm, d)] = nbytes / (t * 1e-3) / 1e9
                    rec["%s_%s_hbm_share" % (arm, d)] = nbytes / (t * 1e-3) / HBM_BPS
                rec["fwd_speedup"] = rec["torch_fwd_us"] / rec["fused_fwd_us"]
                rec["bwd_speedup"] = rec["torch_bwd_us"] / rec["fused_bwd_us"]
                recs.append(rec)
                print("%s %s %-12s fwd %7.1f us (torch %7.1f)  bwd %7.1f us (torch %7.1f)" % (
                    rec["encoder"], dname, name, rec["fused_fwd_us"], rec["torch_fwd_us"], rec["fused_bwd_us"],
                    rec["torch_bwd_us"]), flush=True)
                del graphs, keep, sets
                torch.cuda.empty_cache()
    return recs


# ------------------------------------------------------------------------------------------------ (b) the decoder
def leg_decoder(rounds, steps):
    from monodepth2_b200.layers import fuse_decoder_stages, fuse_disp_heads
    from oracle.depth_decoder import DepthDecoder
    torch.backends.cudnn.benchmark = True
    out = []
    for layers in (18, 50):
        torch.manual_seed(0)
        unfused = fuse_disp_heads(DepthDecoder(ENC[layers]).cuda())
        fused = fuse_decoder_stages(copy.deepcopy(unfused))
        feats = [torch.randn(B, c, H >> (i + 1), W >> (i + 1), device="cuda").requires_grad_(True)
                 for i, c in enumerate(ENC[layers])]
        for amp in (False, True):
            def step(i, dec, amp=amp):
                dec.zero_grad(set_to_none=True)
                for f in feats:
                    f.grad = None
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
                    outs = dec(feats)
                sum(d.float().mean() for d in outs.values()).backward()
            arms = {"unfused": unfused, "fused": fused}
            for dec in arms.values():
                for i in range(3):
                    step(i, dec)
            ms = {k: [] for k in arms}
            for r in range(rounds):
                for k, dec in arms.items():
                    step(0, dec)
                    ms[k].append(events_ms(lambda i, dec=dec: step(i, dec), steps))
            u, f = statistics.median(ms["unfused"]), statistics.median(ms["fused"])
            out.append({"encoder": "resnet%d" % layers, "precision": "autocast_bf16" if amp else "f32",
                        "ms_unfused": u, "ms_fused": f, "speedup": u / f,
                        "rounds_unfused": ms["unfused"], "rounds_fused": ms["fused"]})
            print("decoder resnet%d %s: unfused %.3f ms, fused %.3f ms" % (layers, out[-1]["precision"], u, f),
                  flush=True)
        del unfused, fused, feats
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("decoder_stages.py needs a CUDA device")
    c = card()
    print("card: %s, power limit %s, max SM clock %s" % (c["name"], c.get("power_limit"), c.get("max_sm_clock")),
          flush=True)
    line = {"benchmark": "decoder_stages", "card": c, "torch": torch.__version__,
            "batch": B, "height": H, "width": W}
    line["producers"] = leg_producers(args.rounds, args.steps)
    torch.cuda.empty_cache()
    line["decoder"] = leg_decoder(args.rounds, args.steps)
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
