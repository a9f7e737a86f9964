"""Spec-driven float64 reference of libdgp's covariance language (TEST INFRASTRUCTURE ONLY).

`spec_features`, `spec_cov` and `spec_mean` interpret a `discontinuum_b200.spec.CovSpec` in torch float64 on the CPU, term
by term, from the oracle's own stationary factors (`k_rbf`, `k_matern`, `k_periodic`).  The periodic factor is evaluated
directly with `sin` of the scaled difference, not through the per-point sin / cos columns libdgp appends, so this reference
does not share that rewrite with the engine.  Every function is differentiable in `theta` (a 1-D tensor of natural
parameters), so gradients, posterior means and draws come from the oracle's model-independent routines
(`nlml_grad_autograd`, `predict`, `sample`) with the callables below.

tests/test_spec_generic.py pins this interpreter to the oracle's hand-written loadest / rating / PyMC covariances and mean
functions, then holds the CUDA engine to it on specs that reach every path of the language.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np
import torch

from . import gp_oracle as orc

DT = orc.DT
# kind codes of include/dgp.h (the same values as discontinuum_b200.capi; repeated so the oracle imports no product code)
RBF, MATERN32, MATERN52, PERIODIC = 0, 1, 2, 3
GATE_NONE, GATE_SIGMOID, GATE_INV_SIGMOID = 0, 1, 2
COL_COPY, COL_LOG, COL_GATE = 0, 1, 2
MEAN_ZERO, MEAN_CONST, MEAN_POWERLAW = 0, 1, 2


def spec_features(spec, X, theta):
    """Feature table W[n, ncols]: copy, log(x + eps) or gate 1 / (1 + exp(a (x - theta[b]))) of an X column."""
    cols = []
    for kind, src, tix, aux in spec.cols:
        x = X[:, src]
        if kind == COL_COPY:
            cols.append(x)
        elif kind == COL_LOG:
            cols.append(torch.log(x + aux))
        elif kind == COL_GATE:
            cols.append(1.0 / (1.0 + torch.exp(aux * (x - theta[tix]))))
        else:
            raise ValueError(f"unknown column kind {kind}")
    return torch.stack(cols, 1)


def spec_cov(spec, X1, X2, theta):
    """K(X1, X2) = sum over terms of scale x gate(x1) gate(x2) x product of factors on feature columns (no noise)."""
    W1, W2 = spec_features(spec, X1, theta), spec_features(spec, X2, theta)
    K = torch.zeros(X1.shape[0], X2.shape[0], dtype=DT, device=X1.device)
    for t in spec.terms:
        v = theta[t.scale] * torch.ones_like(K) if t.scale >= 0 else torch.ones_like(K)
        if t.gate != GATE_NONE:
            g1, g2 = W1[:, t.gate_col], W2[:, t.gate_col]
            if t.gate == GATE_INV_SIGMOID:
                g1, g2 = 1.0 - g1, 1.0 - g2
            v = v * g1[:, None] * g2[None, :]
        for f in t.factors:
            ls = [theta[i] for i in f.ls]
            if f.kind == PERIODIC:
                v = v * orc.k_periodic(W1, W2, f.cols[0], theta[f.period], ls[0])
            elif f.kind == RBF:
                v = v * orc.k_rbf(W1, W2, f.cols, ls)
            elif f.kind in (MATERN32, MATERN52):
                v = v * orc.k_matern(W1, W2, f.cols, ls, 1.5 if f.kind == MATERN32 else 2.5)
            else:
                raise ValueError(f"unknown factor kind {f.kind}")
        K = K + v
    return K


def spec_mean(spec, X, theta):
    """m(x): zero, theta[c], or the power law a + b log(x[mean_col] - c)."""
    if spec.mean_kind == MEAN_ZERO:
        return torch.zeros(X.shape[0], dtype=DT, device=X.device)
    if spec.mean_kind == MEAN_CONST:
        return theta[spec.mean_theta[0]].expand(X.shape[0])
    if spec.mean_kind == MEAN_POWERLAW:
        a, b, c = (theta[i] for i in spec.mean_theta[:3])
        return a + b * torch.log(X[:, spec.mean_col] - c)
    raise ValueError(f"unknown mean kind {spec.mean_kind}")


class SpecModel:
    """The oracle's (cov, mean, nat, extra_noise) calling convention for one spec: nat = {"theta": theta}, and the learned
    noise theta[noise_theta] (if any) as extra_noise, so that orc.predict / orc.sample add it to the diagonal of Ky."""

    def __init__(self, spec, X, y, noise):
        self.spec = spec
        self.X, self.y, self.noise = (torch.as_tensor(np.asarray(a, dtype=np.float64)) for a in (X, y, noise))

    def cov(self, X1, X2, nat):
        return spec_cov(self.spec, X1, X2, nat["theta"])

    def mean(self, X, nat):
        return spec_mean(self.spec, X, nat["theta"])

    def nat(self, theta):
        return {"theta": torch.as_tensor(np.asarray(theta, dtype=np.float64))}

    def extra(self, nat):
        return nat["theta"][self.spec.noise_theta] if self.spec.noise_theta >= 0 else None

    def K(self, theta, Xs=None):
        t = self.nat(theta)["theta"]
        return spec_cov(self.spec, self.X if Xs is None else torch.as_tensor(Xs), self.X, t).numpy()

    def nlml_grad(self, theta) -> Tuple[float, np.ndarray, np.ndarray]:
        """(NLML, dNLML/dtheta, alpha) by autograd straight through the Cholesky (orc.nlml_grad_autograd).  The learned
        noise enters as its own leaf; its gradient is added to theta[noise_theta] (chain rule through the tie)."""
        th = self.nat(theta)["theta"]
        leaves = {"theta": th}
        key = None
        if self.spec.noise_theta >= 0:
            key = "extra"
            leaves[key] = th[self.spec.noise_theta].clone()
        val, g = orc.nlml_grad_autograd(self.cov, self.mean, leaves, self.X, self.y, self.noise, extra_key=key)
        grad = g["theta"].clone()
        if key is not None:
            grad[self.spec.noise_theta] += g[key]
        with torch.no_grad():
            d = self.noise if key is None else self.noise + leaves[key]
            Ky = self.cov(self.X, self.X, leaves) + torch.diag(d)
            alpha = orc.nlml_from_K(Ky, self.y - self.mean(self.X, leaves))[2]
        return float(val), grad.numpy(), alpha.numpy()

    def predict(self, theta, Xs):
        """(mu, latent var) at Xs."""
        nat = self.nat(theta)
        mu, _, var = orc.predict(self.cov, self.mean, nat, self.X, self.y, self.noise, torch.as_tensor(Xs),
                                 extra_noise=self.extra(nat))
        return mu.numpy(), var.numpy()

    def mean_functional_grad(self, theta, Xs, c):
        """F = c' mu(Xs) and dF/dtheta by autograd through orc.predict."""
        th = self.nat(theta)["theta"].clone().requires_grad_(True)
        nat = {"theta": th}
        mu = orc.predict(self.cov, self.mean, nat, self.X, self.y, self.noise, torch.as_tensor(Xs),
                         extra_noise=self.extra(nat))[0]
        F = (torch.as_tensor(c) * mu).sum()
        (g,) = torch.autograd.grad(F, [th])
        return float(F.detach()), g.numpy()

    def sample(self, theta, Xs, Z, jitter=0.0):
        nat = self.nat(theta)
        draws, _ = orc.sample(self.cov, self.mean, nat, self.X, self.y, self.noise, torch.as_tensor(Xs),
                              torch.as_tensor(Z), extra_noise=self.extra(nat), jitter=jitter)
        return draws.numpy()
