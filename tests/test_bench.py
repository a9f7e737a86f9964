"""bench.py --dump-outputs: the files hold what the last timed step returned (checked against the CPU oracle)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import helpers as H
from helpers import orc
from discontinuum_b200 import synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(cuda_device, tmp_path):
    n, steps, warmup = 1024, 2, 3
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--n", str(n), "--steps", str(steps), "--warmup",
           str(warmup), "--no-extra", "--no-cpu", "--dump-outputs", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    nlml, grad = np.load(tmp_path / "nlml.npy"), np.load(tmp_path / "grad.npy")
    assert nlml.dtype == grad.dtype == np.float64 and nlml.shape == (1,) and grad.shape == (10,)
    assert nlml[0] == line["nlml"]
    # bench.py evaluates theta_k = theta1 * (1 + 1e-3 k), k = 0 .. warmup + steps - 1; the last one is timed last
    theta = H.loadest_theta1() * (1.0 + 1e-3 * (warmup + steps - 1))
    X, y, noise = synthetic.loadest_site(n, 1000)
    v, g, _, _ = orc.nlml_grad_closed_form(orc.loadest_cov, orc.loadest_mean, H.loadest_nat_from_theta(theta), torch.tensor(X),
                                           torch.tensor(y), torch.tensor(noise))
    go = H.loadest_theta_from_nat({k: t.numpy() for k, t in g.items()})
    assert abs(nlml[0] - float(v)) <= 1e-6 * abs(float(v))
    assert np.max(np.abs(grad - go)) <= 1e-6 * np.max(np.abs(go))
