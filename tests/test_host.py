"""CPU: host logic -- the C-ABI library loads and exports every declared symbol, the spec builders match the
reference's model definitions, the host-side objective assembly (constraints, priors, chain rule) agrees with
the oracle's objective, and the array-level data pipelines reproduce the reference's golden values."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import helpers as H
from helpers import orc
from discontinuum_b200 import capi, data, engine, models, spec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge

    ge.build()
    lib = capi.load_library()
    header = open(os.path.join(ROOT, "include", "dgp.h")).read()
    declared = set(re.findall(r"\b(dgp_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/dgp.h but not exported"
    assert set(capi.EXPORTED_SYMBOLS) == declared
    assert lib.dgp_abi_version() == capi.ABI_VERSION
    assert ctypes.sizeof(capi.DgpSpec) == 1520
    assert lib.dgp_workspace_bytes(16384, 2048) > 3 * 16384 * 16384 * 8


def test_engine_fails_loudly_without_gpu():
    """Run in a fresh process with every device hidden, so that this also holds on a machine that has a GPU."""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import pytest\n"
            "from discontinuum_b200 import capi\n"
            "with pytest.raises(capi.DgpError, match='no CUDA device'):\n"
            "    capi.Engine(max_n=128)\n") % ROOT
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]


def test_loadest_spec_structure():
    s = models.loadest_spec(2)
    assert s.ntheta == 10 and len(s.terms) == 3 and s.noise_theta == -1
    c = s.to_c()
    assert (c.nterms, c.ntheta, c.ncols, c.mean_kind) == (3, 10, 2, capi.MEAN_CONST)
    assert c.term[0].nfactors == 2 and c.term[0].factor[0].kind == capi.PERIODIC and c.term[0].factor[1].kind == capi.MATERN52
    assert c.term[1].factor[0].kind == capi.RBF and c.term[2].factor[0].kind == capi.MATERN32 and c.term[2].factor[0].ndims == 2
    s3 = models.loadest_spec(3)
    assert s3.ntheta == 12 and s3.to_c().term[1].factor[0].ndims == 2


def test_rating_spec_structure():
    s = models.rating_spec(1.1, 1.7)
    assert s.ntheta == 20 and len(s.terms) == 5
    c = s.to_c()
    assert c.noise_theta == s.index("likelihood.second_noise") and c.mean_kind == capi.MEAN_POWERLAW
    gates = [c.term[i].gate for i in range(5)]
    assert gates == [capi.GATE_SIGMOID, capi.GATE_SIGMOID, capi.GATE_INV_SIGMOID, capi.GATE_NONE, capi.GATE_NONE]
    assert c.col[1].kind == capi.COL_LOG and abs(c.col[1].aux - 1e-6) < 1e-20 and c.col[2].kind == capi.COL_GATE and c.col[2].aux == 20.0


def test_constraints_roundtrip_and_init():
    m = spec.GPModule(models.loadest_spec(2))
    nat = m.natural_dict()
    assert abs(nat["seasonal.outputscale"] - np.log(2.0)) < 1e-15 and nat["mean.constant"] == 0.0
    m.set_natural("seasonal.periodic.period_length", 1.0)
    assert abs(m.natural_dict()["seasonal.periodic.period_length"] - 1.0) < 1e-14
    r = spec.GPModule(models.rating_spec(1.1, 1.7, gate_b_init=1.3))
    d = r.natural_dict()
    assert abs(d["sigmoid.b"] - 1.3) < 1e-12 and abs(d["likelihood.second_noise"] - (np.log(2.0) + 1e-4)) < 1e-15


class _FakeEngine:
    """Stands in for libdgp on the CPU: serves NLML and its natural-parameter gradient from the oracle."""

    def __init__(self, model, X, y, noise):
        self.model, self.X, self.y, self.noise = model, torch.tensor(X), torch.tensor(y), torch.tensor(noise)

    def nlml_grad(self, theta, jitter=0.0):
        with torch.enable_grad():  # called from inside an autograd.Function.forward, where grad mode is off
            return self._eval(theta)

    def _eval(self, theta):
        if self.model == "loadest":
            nat = H.loadest_nat_from_theta(theta)
            v, g, _, _ = orc.nlml_grad_closed_form(orc.loadest_cov, orc.loadest_mean, nat, self.X, self.y, self.noise)
            return float(v), H.loadest_theta_from_nat({k: t.numpy() for k, t in g.items()}), 0
        nat = H.rating_nat_from_theta(theta)
        v, g, _, _ = orc.nlml_grad_closed_form(orc.rating_cov, orc.rating_mean, nat, self.X, self.y, self.noise, extra_key="noise")
        return float(v), H.rating_theta_from_nat({k: t.numpy() for k, t in g.items()}), 0


def test_host_objective_and_chain_rule_loadest():
    from discontinuum_b200 import synthetic

    X, y, noise = synthetic.loadest_site(60, 5)
    m = models.LoadestGP()
    m.X, m.y = X, y
    m.model = m.build_model(X, y)
    m._engine = _FakeEngine("loadest", X, y, noise)
    obj, _ = m._objective()
    obj.backward()
    raw = {k: v.clone().requires_grad_(True) for k, v in orc.loadest_init_raw().items()}
    want = orc.objective("loadest", raw, torch.tensor(X), torch.tensor(y), torch.tensor(noise))
    want.backward()
    assert abs(float(obj) - float(want)) <= 1e-12 * abs(float(want))
    got = np.concatenate([p.grad.numpy() for p in m.model.raw_list()])
    ref = np.concatenate([raw[k].grad.numpy().ravel() for k in ("mean_c", "s1", "lam", "period", "l1", "s2", "l2", "s3", "l3")])
    assert np.max(np.abs(got - ref)) <= 1e-9 * np.max(np.abs(ref))


def test_host_objective_and_chain_rule_rating():
    from discontinuum_b200 import synthetic

    X, y, noise = synthetic.rating_gauge(50, 3)
    b_lo, b_hi = models.stage_quantile_bounds(X[:, 1])
    m = models.RatingGP()
    m.X, m.y = X, y
    m.fixed_noise = noise
    m.model = spec.GPModule(models.rating_spec(b_lo, b_hi))
    m._engine = _FakeEngine("rating", X, y, noise)
    obj, _ = m._objective()
    obj.backward()
    raw = {k: v.clone().requires_grad_(True) for k, v in orc.rating_init_raw(b_lo, b_hi).items()}
    want = orc.objective("rating", raw, torch.tensor(X), torch.tensor(y), torch.tensor(noise), b_lo, b_hi)
    want.backward()
    assert abs(float(obj) - float(want)) <= 1e-12 * abs(float(want))
    got = np.concatenate([p.grad.numpy() for p in m.model.raw_list()])
    ref = np.array([float(raw[k].grad) for k in H.RATING_KEYS])
    assert np.max(np.abs(got - ref)) <= 1e-9 * np.max(np.abs(ref))


@pytest.mark.parametrize("model", ["loadest", "rating"])
def test_closed_form_host_path_matches_autograd(model):
    """GPModule.host_chain / MarginalB200._objective_closed_form against the autograd path: same objective, same
    gradient w.r.t. every raw parameter, at the initial values and after moving the raw parameters around."""
    from discontinuum_b200 import synthetic

    if model == "loadest":
        X, y, noise = synthetic.loadest_site(50, 9)
        m = models.LoadestGP()
        m.X, m.y = X, y
        m.model = m.build_model(X, y)
    else:
        X, y, noise = synthetic.rating_gauge(40, 4)
        b_lo, b_hi = models.stage_quantile_bounds(X[:, 1])
        m = models.RatingGP()
        m.X, m.y = X, y
        m.fixed_noise = noise
        m.model = spec.GPModule(models.rating_spec(b_lo, b_hi))
    m._engine = _FakeEngine(model, X, y, noise)
    rng = np.random.default_rng(1)
    for rep in range(3):
        if rep:
            with torch.no_grad():
                for p in m.model.raw_list():
                    p.add_(float(rng.normal(0.0, 0.4)))
        for p in m.model.raw_list():
            p.grad = None
        obj, _ = m._objective()
        obj.backward()
        want = np.concatenate([p.grad.numpy() for p in m.model.raw_list()])
        val, graw = m._objective_closed_form()
        assert abs(val - float(obj)) <= 1e-13 * abs(float(obj))
        assert np.max(np.abs(graw - want)) <= 1e-12 * np.max(np.abs(want))
    # softplus threshold and interval constraint at the extremes
    with torch.no_grad():
        m.model.raw_list()[1].fill_(25.0)
        m.model.raw_list()[2].fill_(-30.0)
    nat, dnat, lp, dlp = m.model.host_chain()
    ref = m.model.natural().detach().numpy()
    assert np.allclose(nat, ref, rtol=1e-15, atol=1e-300) and dnat[1] == 1.0 and np.isfinite(lp)


def test_rating_projection():
    m = models.RatingGP()
    X = np.stack([np.linspace(-1, 1, 30), np.linspace(1.0, 2.0, 30)], 1)
    m.model = spec.GPModule(models.rating_spec(1.1, 1.9, pl_b=3.0, pl_c=1.5))
    m.project_parameters(X)
    d = m.model.natural_dict()
    assert d["powerlaw.b"] == 2.5 and abs(d["powerlaw.c"] - (1.0 - 1e-6)) < 1e-15


def test_time_pipeline_reference_golden_values():
    """src/discontinuum/tests/test_pipeline.py:7-29 holds the only golden numbers of the reference's test-suite."""
    t = np.array(["2022-01-01", "2022-02-01", "2022-03-01"], dtype="datetime64[ns]")
    dy = data.datetime_to_decimal_year(t)
    assert np.allclose(dy, [2022.0, 2022.08493151, 2022.16164384], atol=1e-8)
    back = data.decimal_year_to_datetime(dy)
    assert np.all(np.abs((back - t).astype("timedelta64[s]").astype(int)) <= 1)


def test_data_manager_model_space():
    rng = np.random.default_rng(0)
    n = 50
    time = (np.datetime64("2000-01-01") + (np.sort(rng.uniform(0, 3650, n)) * 86400e9).astype("timedelta64[ns]"))
    flow = rng.lognormal(3, 1, n)
    conc = rng.lognormal(0, 0.5, n)
    m = models.LoadestGP()
    m.dm.fit(target=conc, covariates={"time": time, "flow": flow})
    X, y = m.dm.X, m.dm.y
    assert X.shape == (n, 2) and abs(X[:, 0].mean()) < 1e-9 and abs(X[:, 1].mean()) < 1e-12 and abs(X[:, 1].std() - 1) < 1e-12
    assert abs(y.mean()) < 1e-12 and abs(y.std() - 1) < 1e-12
    assert np.allclose(m.dm.y_t(y), conc)
    se = m.dm.se_t(np.full(3, 0.04))
    assert np.allclose(se, np.exp(0.2 * np.log(conc).std()))
    assert m.dm.get_dim("flow") == 1
    with pytest.raises(ValueError):
        models.LoadestGP(engine.ModelConfig(transform="bogus"))
    with pytest.raises(RuntimeError, match="hasn't been fitted"):
        models.LoadestGP().predict({"time": time, "flow": flow})


def test_xarray_adapter_branches_with_stand_in(monkeypatch):
    """The optional xarray adapter (data.py) against tests/fake_xarray.py: same model-space arrays as the numpy / dict
    route, DataArray out with the training target's attributes and name, coordinates first in the column order."""
    import fake_xarray as fx

    monkeypatch.setattr(data, "_xr", fx)
    rng = np.random.default_rng(2)
    n = 40
    time = (np.datetime64("2001-01-01") + (np.sort(rng.uniform(0, 2000, n)) * 86400e9).astype("timedelta64[ns]"))
    flow = rng.lognormal(3, 1, n)
    conc = rng.lognormal(0, 0.5, n)
    ds = fx.Dataset({"flow": ("time", flow)}, coords={"time": time})
    tgt = fx.DataArray(conc, coords={"time": time}, dims=("time",), attrs={"units": "mg/L"}, name="concentration")
    a, b = models.LoadestGP(), models.LoadestGP()
    a.dm.fit(target=tgt, covariates=ds)
    b.dm.fit(target=conc, covariates={"time": time, "flow": flow})
    assert np.array_equal(a.dm.X, b.dm.X) and np.array_equal(a.dm.y, b.dm.y)
    assert a.dm.get_dim("time") == 0 and a.dm.get_dim("flow") == 1
    back = a.dm.y_t(a.dm.y)
    assert isinstance(back, fx.DataArray) and back.attrs == {"units": "mg/L"} and back.name == "concentration"
    assert back.dims == ("time",) and np.allclose(back.values, conc)
    se = a.dm.se_t(np.full(n, 0.04))
    assert isinstance(se, fx.DataArray) and np.allclose(se.values, np.asarray(b.dm.se_t(np.full(n, 0.04))))
    placed = engine._assign_coords(back, ds)
    assert list(placed.coords) == ["time"] and np.array_equal(placed.coords["time"].values, time)
    assert isinstance(b.dm.y_t(b.dm.y), np.ndarray)  # numpy in, numpy out



def test_checkpoint_keys_follow_the_reference_module_tree():
    """engine.save writes the gpytorch key names / shapes of the reference's modules (loadest_gp/models/gpytorch.py:61-128,
    rating_gp/models/gpytorch.py:205-372; engines/gpytorch.py:147-160) and load reads a reference-format state dict."""
    from discontinuum_b200 import checkpoint

    m = spec.GPModule(models.loadest_spec(3))
    with torch.no_grad():
        for k, p in enumerate(m.raw_list()):
            p.fill_(0.1 * (k + 1))
    sd, lik = checkpoint.to_reference_state(m)
    assert lik == {}
    assert set(sd) == {"mean_module.raw_constant", "covar_module.kernels.0.raw_outputscale",
                       "covar_module.kernels.0.base_kernel.kernels.0.raw_lengthscale",
                       "covar_module.kernels.0.base_kernel.kernels.0.raw_period_length",
                       "covar_module.kernels.0.base_kernel.kernels.1.raw_lengthscale", "covar_module.kernels.1.raw_outputscale",
                       "covar_module.kernels.1.base_kernel.raw_lengthscale", "covar_module.kernels.2.raw_outputscale",
                       "covar_module.kernels.2.base_kernel.raw_lengthscale"}
    assert sd["covar_module.kernels.1.base_kernel.raw_lengthscale"].shape == (1, 2)   # ARD over the two covariates
    assert sd["covar_module.kernels.2.base_kernel.raw_lengthscale"].shape == (1, 3)
    assert sd["covar_module.kernels.0.raw_outputscale"].shape == () and sd["mean_module.raw_constant"].shape == ()
    # a reference-written checkpoint also holds constraint / prior buffers and may use the nested (A + B) + C layout
    ref = dict(sd)
    ref["covar_module.kernels.0.raw_outputscale_constraint.lower_bound"] = torch.tensor(0.0)
    ref["covar_module.kernels.0.outputscale_prior.scale"] = torch.tensor(1.0)
    m2 = spec.GPModule(models.loadest_spec(3))
    checkpoint.load_state(m2, ref, {})
    assert all(float(a.detach()) == float(b.detach()) for a, b in zip(m.raw_list(), m2.raw_list()))
    nested = {}
    for k, v in sd.items():
        for flat, nest in (("covar_module.kernels.0.", "covar_module.kernels.0.kernels.0."),
                           ("covar_module.kernels.1.", "covar_module.kernels.0.kernels.1."),
                           ("covar_module.kernels.2.", "covar_module.kernels.1.")):
            if k.startswith(flat):
                k = nest + k[len(flat):]
                break
        nested[k] = v
    m3 = spec.GPModule(models.loadest_spec(3))
    checkpoint.load_state(m3, nested)
    assert all(float(a.detach()) == float(b.detach()) for a, b in zip(m.raw_list(), m3.raw_list()))
    # round-1 native layout still loads; a foreign state dict fails with the missing key named
    m4 = spec.GPModule(models.loadest_spec(3))
    checkpoint.load_state(m4, m.state_dict())
    assert all(float(a.detach()) == float(b.detach()) for a, b in zip(m.raw_list(), m4.raw_list()))
    with pytest.raises(KeyError, match="raw_period_length"):
        checkpoint.load_state(m4, {k: v for k, v in sd.items() if "period" not in k})

    r = spec.GPModule(models.rating_spec(1.1, 1.8))
    with torch.no_grad():
        for k, p in enumerate(r.raw_list()):
            p.fill_(-0.3 + 0.07 * k)
    rsd, rlik = checkpoint.to_reference_state(r)
    assert set(rlik) == {"second_noise_covar.raw_noise"} and rlik["second_noise_covar.raw_noise"].shape == (1,)
    assert {"powerlaw.a", "powerlaw.b", "powerlaw.c", "likelihood.second_noise_covar.raw_noise",
            "covar_module.kernels.0.kernels.0.raw_b", "covar_module.kernels.1.kernels.0.sigmoid_kernel.raw_b",
            "covar_module.kernels.0.kernels.1.base_kernel.kernels.1.base_kernel.kernels.1.raw_lengthscale",
            "covar_module.kernels.1.kernels.1.base_kernel.raw_outputscale",
            "covar_module.kernels.2.base_kernel.kernels.1.base_kernel.kernels.0.raw_period_length"} <= set(rsd)
    assert len(rsd) == 20 + 2   # 20 parameters + the two extra registrations of the shared gate switch point
    r2 = spec.GPModule(models.rating_spec(1.1, 1.8))
    model_only = {k: v for k, v in rsd.items() if not k.startswith("likelihood.")}
    checkpoint.load_state(r2, model_only, rlik)   # learned noise taken from the likelihood state dict
    assert all(float(a.detach()) == float(b.detach()) for a, b in zip(r.raw_list(), r2.raw_list()))


@pytest.mark.parametrize("model,opt", [("loadest", "adam"), ("loadest", "adamw"), ("rating", "adam")])
def test_numpy_optimiser_path_matches_torch_path(model, opt, monkeypatch):
    """MarginalB200.fit's numpy optimiser path (raw parameters, Adam moments and chain rule in numpy vectors, no tensor
    per iteration) against its torch path (torch.optim.Adam / AdamW fused step on the module's tensors): same objective
    history, same final raw parameters, same optimiser state for save / resume, also across an interrupted-and-resumed fit.
    The engine is the CPU oracle stand-in (no GPU needed)."""
    from discontinuum_b200 import synthetic

    rng = np.random.default_rng(5)
    n = 40
    days = np.sort(rng.uniform(0, 3650, n))
    time = np.datetime64("2005-01-01") + (days * 86400e9).astype("timedelta64[ns]")
    if model == "loadest":
        flow = np.exp(1.0 + 0.8 * np.sin(2 * np.pi * days / 365.25) + 0.5 * rng.standard_normal(n))
        cov = {"time": time, "flow": flow}
        target = np.exp(0.3 * np.log(flow) + 0.2 * np.cos(2 * np.pi * days / 365.25) + 0.2 * rng.standard_normal(n))
        kw = {}
    else:
        stage = rng.lognormal(1.0, 0.5, n)
        cov = {"time": time, "stage": stage}
        target = 3.0 * (stage - 0.5 * stage.min()) ** 1.6 * np.exp(0.03 * rng.standard_normal(n))
        kw = dict(target_unc=rng.choice(np.array([1.02, 1.05, 1.08]), n))

    def make():
        m = models.LoadestGP() if model == "loadest" else models.RatingGP()
        fake = _FakeEngine(model, np.zeros((1, 2)), np.zeros(1), np.zeros(1))

        def bind(self=m):
            # serve the oracle on what the engine would be given (the data manager has standardised the inputs)
            fake.X, fake.y = torch.tensor(self.X), torch.tensor(self.y)
            fake.noise = torch.tensor(np.asarray(self.fixed_noise, dtype=np.float64) * np.ones(self.X.shape[0]))
            self._engine = fake
            self._factorized_at = None

        m._bind_engine = bind
        return m

    out = {}
    for path in ("torch", "numpy"):
        monkeypatch.setenv("DGP_HOST_OPT", path)
        torch.manual_seed(0)   # (rating-gp draws its initial power-law parameters from torch's generator)
        m = make()
        m.fit(cov, target, iterations=12, optimizer=opt, learning_rate=0.1, **kw)
        h1 = list(m.history)
        m.fit(cov, target, iterations=20, resume=True, **kw)          # interrupted-and-resumed: 8 more iterations
        raw = np.array([float(p.detach()) for p in m.model.raw_list()])
        st = m._last_optimizer.state_dict()["state"]
        out[path] = (np.array(h1 + list(m.history)), raw,
                     np.array([float(st[k]["exp_avg"].reshape(-1)[0]) for k in sorted(st)]),
                     np.array([float(st[k]["exp_avg_sq"].reshape(-1)[0]) for k in sorted(st)]),
                     [float(st[k]["step"]) for k in sorted(st)], m._last_optimizer.param_groups[0]["lr"])
    a, b = out["torch"], out["numpy"]
    assert len(a[0]) == len(b[0]) >= 20   # (resume continues from the last started iteration, as the reference does)
    assert np.max(np.abs(a[0] - b[0]) / np.abs(a[0])) <= 1e-10
    assert np.max(np.abs(a[1] - b[1])) <= 1e-9 * max(1.0, np.max(np.abs(a[1])))
    assert np.max(np.abs(a[2] - b[2])) <= 1e-9 * max(1e-3, np.max(np.abs(a[2])))
    assert np.max(np.abs(a[3] - b[3])) <= 1e-9 * max(1e-6, np.max(np.abs(a[3])))
    assert a[4] == b[4] and a[5] == b[5]
