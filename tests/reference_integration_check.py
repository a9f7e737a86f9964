"""Run by tests/test_reference_integration.py in a fresh process, only where the reference's sources are readable
(DISCONTINUUM_REFERENCE = its src/ directory).  INTEGRATION.md section 1, executed: the reference's OWN data mixin (its DataManager
and pipelines) and its OWN plot mixin, composed with `MarginalB200` exactly as a maintainer would,

    class LoadestGPMarginalB200(LoadestDataMixin, LoadestPlotMixin, MarginalB200): ...

then fit / predict / predict_grid / plot / contourf / plot_observations, and the same for rating-gp.  Third-party layers are
stand-ins (tests/fake_xarray.py as `xarray`, a mock matplotlib, oracle/gpytorch_standin so that the reference packages import);
the engine behind MarginalB200 is a CPU stand-in that serves NLML, gradient and predictions from the oracle (no GPU here), so
what this checks is the SURFACE: that the reference's mixins find every attribute, method, argument and container type they use.
"""
import importlib.machinery
import os
import sys
import types
from unittest.mock import MagicMock

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ["DISCONTINUUM_REFERENCE"]
sys.path[:0] = [os.path.join(ROOT, "oracle", "gpytorch_standin"), HERE, ROOT]


def _stub(name):
    m = types.ModuleType(name)
    m.__spec__ = importlib.machinery.ModuleSpec(name, loader=None, is_package=True)
    m.__path__ = []
    m.__getattr__ = lambda attr: MagicMock(name=f"{name}.{attr}")
    return m


import fake_xarray as fx  # noqa: E402

xr = _stub("xarray")
xr.DataArray, xr.Dataset = fx.DataArray, fx.Dataset
sys.modules["xarray"] = xr
for name in ["matplotlib", "matplotlib.pyplot", "matplotlib.dates", "matplotlib.ticker", "matplotlib.colors", "matplotlib.cm",
             "matplotlib.axes", "dataretrieval", "dataretrieval.nwis"]:
    sys.modules[name] = _stub(name)
sys.path.insert(0, REF)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import helpers as H  # noqa: E402
from helpers import orc  # noqa: E402
from discontinuum_b200 import data as b200_data  # noqa: E402
from discontinuum_b200.engine import MarginalB200  # noqa: E402
from discontinuum_b200.models import LOADEST_FIXED_NOISE, loadest_spec, rating_spec, stage_quantile_bounds  # noqa: E402
from discontinuum_b200.spec import GPModule  # noqa: E402

assert b200_data._xr is xr, "the adapter must see the xarray stand-in"

from loadest_gp.models.base import LoadestDataMixin  # noqa: E402  (the reference's own mixins)
from loadest_gp.plot import LoadestPlotMixin  # noqa: E402
from rating_gp.models.base import RatingDataMixin  # noqa: E402
from rating_gp.plot import RatingPlotMixin  # noqa: E402
from discontinuum.engines.base import ModelConfig  # noqa: E402


class CpuEngine:
    """libdgp's Engine surface as MarginalB200 uses it, served by the CPU oracle."""
    max_n = max_m = 1 << 30

    def __init__(self, kind):
        self.kind = kind

    def set_train(self, spec_c, X, y, noise):
        self.X, self.y, self.noise = torch.tensor(X), torch.tensor(y), torch.tensor(np.asarray(noise, dtype=np.float64))

    def _pieces(self, theta):
        if self.kind == "loadest":
            nat = H.loadest_nat_from_theta(theta, self.X.shape[1])
            return nat, orc.loadest_cov, orc.loadest_mean, None
        nat = H.rating_nat_from_theta(theta)
        return nat, orc.rating_cov, orc.rating_mean, nat["noise"]

    def nlml_grad(self, theta, jitter=0.0):
        nat, cov, mean, extra = self._pieces(theta)
        with torch.enable_grad():
            v, g, _, _ = orc.nlml_grad_closed_form(cov, mean, nat, self.X, self.y, self.noise,
                                                   extra_key=None if extra is None else "noise")
        conv = H.loadest_theta_from_nat if self.kind == "loadest" else H.rating_theta_from_nat
        return float(v), conv({k: t.numpy() for k, t in g.items()}), 0

    def factorize(self, theta, jitter=0.0):
        self.theta = np.array(theta)
        return 0.0, 0

    def predict(self, Xs, want_var=True):
        nat, cov, mean, extra = self._pieces(self.theta)
        mu, _, var = orc.predict(cov, mean, nat, self.X, self.y, self.noise, torch.tensor(Xs), extra_noise=extra, min_variance=0.0)
        return mu.numpy(), var.numpy()

    def sample(self, Xs, Z, jitter=0.0):
        nat, cov, mean, extra = self._pieces(self.theta)
        sim, _ = orc.sample(cov, mean, nat, self.X, self.y, self.noise, torch.tensor(Xs), torch.tensor(Z), extra_noise=extra,
                            jitter=max(float(jitter), 1e-8))
        return sim.numpy(), 0

    def close(self):
        pass


class _CpuBound(MarginalB200):
    kind = "loadest"

    def _bind_engine(self):
        self._engine = CpuEngine(self.kind)
        self._engine.set_train(None, self.X, self.y, self.fixed_noise)
        self._factorized_at = None


class LoadestGPMarginalB200(LoadestDataMixin, LoadestPlotMixin, _CpuBound):   # INTEGRATION.md section 1
    def __init__(self, model_config=None):
        super().__init__(model_config=model_config or ModelConfig())
        self.build_datamanager(model_config)

    def build_model(self, X, y):
        self.fixed_noise = np.full(y.shape[0], LOADEST_FIXED_NOISE)
        return GPModule(loadest_spec(X.shape[1]))


class RatingGPMarginalB200(RatingDataMixin, RatingPlotMixin, _CpuBound):
    kind = "rating"

    def __init__(self, model_config=None):
        super().__init__(model_config=model_config or ModelConfig())
        self.build_datamanager(model_config)

    def build_model(self, X, y, y_unc=None):
        self.fixed_noise = np.asarray(y_unc, dtype=np.float64)
        b_lo, b_hi = stage_quantile_bounds(X[:, 1])
        return GPModule(rating_spec(b_lo, b_hi, pl_a=0.1, pl_b=1.5, pl_c=0.4))

    def project_parameters(self, X_all):
        with torch.no_grad():
            self.model.raw["powerlaw__b"].clamp_(1.2, 2.5)
            self.model.raw["powerlaw__c"].clamp_(max=float(X_all[:, 1].min()) - 1e-6)


def main():
    rng = np.random.default_rng(1)
    n = 30
    days = np.sort(rng.uniform(0, 3650, n))
    time = np.datetime64("2000-01-01") + (days * 86400e9).astype("timedelta64[ns]")
    flow = np.exp(1.0 + 0.5 * rng.standard_normal(n))
    conc = np.exp(0.3 * np.log(flow) + 0.2 * rng.standard_normal(n))
    cov = fx.Dataset({"flow": ("time", flow)}, coords={"time": time})
    tgt = fx.DataArray(conc, coords={"time": time}, dims=("time",), attrs={"units": "mg/L", "long_name": "Concentration"}, name="conc")
    m = LoadestGPMarginalB200()
    assert type(m.dm).__module__ == "discontinuum.data_manager", "the reference's own DataManager is in charge"
    m.fit(covariates=cov, target=tgt, iterations=4)
    assert m.is_fitted and len(m.history) == 4 and m.history[-1] < m.history[0]
    target, se = m.predict(cov)
    assert isinstance(target, fx.DataArray) and isinstance(se, fx.DataArray) and target.attrs["units"] == "mg/L"
    assert target.values.shape == (n,) and np.all(target.values > 0) and np.all(se.values >= 1.0) and "time" in target.coords
    grid = m.predict_grid("flow")
    assert isinstance(grid, fx.DataArray) and grid.values.shape[1] == 18 and list(grid.dims) == ["time", "flow"]
    draws = m.sample(cov, n=6, seed=0)                                 # engines/gpytorch.py:551-593: [draw, time] in data space
    assert isinstance(draws, fx.DataArray) and draws.values.shape == (6, n) and list(draws.dims) == ["draw", "time"]
    assert np.all(draws.values > 0) and list(draws.coords["draw"].values) == list(range(6)) and draws.attrs["units"] == "mg/L"
    ax = MagicMock(name="Axes")
    assert m.plot(cov, ax=ax) is ax and ax.fill_between.called          # discontinuum/plot.py:68-119
    m.plot_observations(ax)                                            # discontinuum/plot.py:42-66
    assert m.contourf(levels=5, y_scale="log", ax=ax) is ax            # loadest_gp/plot.py:51-86 (as tests/test_loadest_gp.py:84)
    print("loadest: fit / predict / predict_grid / sample / plot / plot_observations / contourf ok; objective", m.history[0], "->", m.history[-1])

    stage = rng.lognormal(1.0, 0.5, n)
    q = 3.0 * (stage - 0.5 * stage.min()) ** 1.6 * np.exp(0.03 * rng.standard_normal(n))
    gse = rng.choice(np.array([1.02, 1.05, 1.08]), n)
    cov = fx.Dataset({"stage": ("time", stage)}, coords={"time": time})
    tgt = fx.DataArray(q, coords={"time": time}, dims=("time",), attrs={"units": "cfs", "long_name": "Discharge"}, name="discharge")
    unc = fx.DataArray(gse, coords={"time": time}, dims=("time",), name="gse")
    r = RatingGPMarginalB200()
    r.fit(covariates=cov, target=tgt, target_unc=unc, iterations=3)
    target, se = r.predict(cov)
    assert isinstance(target, fx.DataArray) and np.all(np.isfinite(target.values)) and np.all(se.values >= 1.0)
    ax = MagicMock(name="Axes")
    assert r.plot(cov, ax=ax) is ax
    print("rating: fit / predict / plot ok; objective", r.history[0], "->", r.history[-1])
    done = ["plot"]
    for name, args in (("plot_rating", (cov,)), ("plot_stage", (cov,)), ("plot_discharge", (cov,)), ("plot_observed_rating", ()),
                       ("plot_ratings_in_time", ())):      # rating_gp/plot.py:39-287 (plot_ratings_in_time predicts 5 x 250 points)
        getattr(r, name)(*args, ax=ax)
        done.append(name)
    print("rating plot mixin methods run:", done)
    print("INTEGRATION OK")


if __name__ == "__main__":
    main()
