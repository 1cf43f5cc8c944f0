"""bench.py --dump-outputs: the losses and gradients of the last timed step, written as .npy, are the same from run to
run with the same arguments (seeded inputs and tie-break noise) and are what the public call returns on the rotating
batch of that step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEPS = 6


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                        "--no-cpu", "--no-train", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout)


def _public_call_on_rotating_batch(step):
    """The public call on the batch bench.py's default workload (mono_640x192_b12) times at `step`: four rotating
    synthetic batches, seeds 0..3 on rank 0.  Its tie-break noise is drawn afresh, so near-tie pixels may differ."""
    import torch
    from monodepth2_b200.fused_loss import LossPlan, view_synthesis_loss
    from monodepth2_b200.synthetic import make_batch
    fids = [0, -1, 1]
    inputs, outputs, _, _ = make_batch(12, 192, 640, fids, 4, seed=step % 4, kind="iid", n_id=2)
    ins = {k: v.cuda() for k, v in inputs.items()}
    leaves = {k: v.cuda().requires_grad_(True) for k, v in outputs.items()}
    losses = view_synthesis_loss(LossPlan(12, 192, 640, fids), ins, dict(leaves))
    losses["loss"].backward()
    return float(losses["loss"]), {s: leaves[("disp", s)].grad.cpu().numpy() for s in range(4)}


@pytest.mark.gpu
def test_dump_outputs_repeat_and_are_the_last_timed_step(tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    line = _bench(a, STEPS)
    _bench(b, STEPS)
    assert line["steps"] == STEPS
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b))
    assert set(names) == ({"loss.npy", "grad_cam_T_cam_0_-1.npy", "grad_cam_T_cam_0_1.npy"} |
                          {"loss_%d.npy" % s for s in range(4)} | {"grad_disp_%d.npy" % s for s in range(4)})
    total = 0
    for n in names:
        x, y = np.load(a / n), np.load(b / n)
        assert x.dtype == np.float32 and np.isfinite(x).all(), n
        total += x.nbytes
        np.testing.assert_allclose(x, y, rtol=1e-5, atol=1e-6 * float(np.abs(x).max()), err_msg=n)
    assert total <= 64 << 20
    assert float(np.load(a / "loss.npy")) == pytest.approx(line["notes"]["loss"], rel=1e-6)

    loss, grads = _public_call_on_rotating_batch(STEPS - 1)
    assert float(np.load(a / "loss.npy")) == pytest.approx(loss, rel=1e-5)
    for s in range(4):
        got = np.load(a / ("grad_disp_%d.npy" % s))
        assert got.shape == grads[s].shape == (12, 1, 192 >> s, 640 >> s)
        # near-tie pixels that the two noise draws select differently change a small part of the gradient; the
        # gradient of another rotating batch is uncorrelated with this one (relative difference ~1.4)
        rel = float(np.linalg.norm(got - grads[s]) / np.linalg.norm(grads[s]))
        assert rel < 0.25, (s, rel)
