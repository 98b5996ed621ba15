"""bench.py --dump-outputs: the files hold what the timed path returned in its LAST timed step, so --steps decides which
seeded batch they come from, and two builds run with the same arguments can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"


def _step_outputs(seed, N, W):
    """One bench step (forward + CTC loss/grad + total loss) on bench.py's model and seeded batch, computed here."""
    import torch
    from lstm_ctc_ocr_b200 import engine, synthetic
    m = engine.CrnnModel(weight_decay=1e-5, device=DEV)
    m.load_params(synthetic.init_params(3))
    data, lab, ll, tsl = synthetic.synth_batch(N, W, seed=seed)
    t_ = lambda a: torch.tensor(a, device=DEV)
    logits = m.forward(t_(data), t_(tsl))
    costs, grad = engine.ctc_loss(logits, t_(lab), t_(ll), t_(tsl), want_grad=True, grad_scale=1.0 / N, max_label_len=int(ll.max()))
    loss = m.total_loss(costs)
    return {"logits": logits.cpu().numpy(), "ctc_costs": costs.cpu().numpy(), "ctc_grad": grad.cpu().numpy(), "loss": loss.cpu().numpy()}


def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    steps, N, W = 3, 32, 100                                  # workload c1shape; bench batch i has seed 3 + i (rank 0)
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1shape", "--steps", str(steps), "--warmup", "3",
                        "--no-cpu-baseline", "--no-decode-eq", "--no-train", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps
    got = {n: np.load(str(out / (n + ".npy"))) for n in ("logits", "ctc_costs", "ctc_grad", "loss")}
    assert sorted(os.listdir(str(out))) == sorted(n + ".npy" for n in got)
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["logits"].shape == got["ctc_grad"].shape == (W // 4 - 1, N, 64) and got["ctc_costs"].shape == (N,)
    rel = lambda a, b: float(np.abs(a - b).max() / np.abs(b).max())
    want = _step_outputs(3 + steps - 1, N, W)
    for n, a in got.items():
        assert rel(a, want[n]) <= 1e-3, (n, rel(a, want[n]))      # same kernels, same inputs: reordered sums at most
    before = _step_outputs(3 + steps - 2, N, W)
    assert rel(got["logits"], before["logits"]) > 0.05, "the dump is not the last timed step's"
