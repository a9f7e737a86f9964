"""ctypes binding of libdgp.so (include/dgp.h) -- the only way Python reaches the CUDA engine.

There is no fallback: if the shared library is missing or no B200 is visible, loading / creating
an engine raises.  Arrays cross the boundary as raw pointers: numpy float64 arrays (host) or
torch CUDA float64 tensors (device).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence, Tuple

import numpy as np

MAX_TERMS, MAX_FACTORS, MAX_FDIMS, MAX_COLS, MAX_THETA = 8, 3, 4, 8, 48
ABI_VERSION = 2
BATCH_MAX_SITES = 32
BATCH_PREDICT_CHUNK = 1024  # grid rows of every site per launch of dgp_batch_predict (csrc/dgp_batch.cuh)

RBF, MATERN32, MATERN52, PERIODIC = 0, 1, 2, 3
GATE_NONE, GATE_SIGMOID, GATE_INV_SIGMOID = 0, 1, 2
COL_COPY, COL_LOG, COL_GATE = 0, 1, 2
MEAN_ZERO, MEAN_CONST, MEAN_POWERLAW = 0, 1, 2


class DgpCol(C.Structure):
    _fields_ = [("kind", C.c_int32), ("src", C.c_int32), ("theta", C.c_int32), ("pad_", C.c_int32), ("aux", C.c_double)]


class DgpFactor(C.Structure):
    _fields_ = [("kind", C.c_int32), ("ndims", C.c_int32), ("col", C.c_int32 * MAX_FDIMS), ("ls", C.c_int32 * MAX_FDIMS),
                ("period", C.c_int32), ("pad_", C.c_int32)]


class DgpTerm(C.Structure):
    _fields_ = [("scale", C.c_int32), ("gate", C.c_int32), ("gate_col", C.c_int32), ("nfactors", C.c_int32),
                ("factor", DgpFactor * MAX_FACTORS)]


class DgpSpec(C.Structure):
    _fields_ = [("abi", C.c_int32), ("ndim", C.c_int32), ("ncols", C.c_int32), ("nterms", C.c_int32),
                ("ntheta", C.c_int32), ("noise_theta", C.c_int32), ("mean_kind", C.c_int32), ("mean_col", C.c_int32),
                ("mean_theta", C.c_int32 * 4), ("col", DgpCol * MAX_COLS), ("term", DgpTerm * MAX_TERMS)]


class DgpFluxReduce(C.Structure):
    _fields_ = [("y_mean", C.c_double), ("y_scale", C.c_double), ("log_transform", C.c_int32), ("ngroups", C.c_int32),
                ("weight", C.c_void_p), ("group_start", C.c_void_p)]


# every symbol include/dgp.h declares: (name, restype, argtypes)
_P = C.c_void_p
_SIGNATURES = [
    ("dgp_create", C.c_int, [C.POINTER(_P), C.c_int, C.c_int, C.c_int, _P]),
    ("dgp_destroy", C.c_int, [_P]),
    ("dgp_last_error", C.c_char_p, [_P]),
    ("dgp_abi_version", C.c_int, []),
    ("dgp_workspace_bytes", C.c_size_t, [C.c_int, C.c_int]),
    ("dgp_set_train", C.c_int, [_P, C.POINTER(DgpSpec), _P, _P, _P, C.c_int, C.c_int]),
    ("dgp_covmat", C.c_int, [_P, _P, _P, C.c_int]),
    ("dgp_cross_covmat", C.c_int, [_P, _P, _P, C.c_int, C.c_int, _P, C.c_int]),
    ("dgp_nlml", C.c_int, [_P, _P, C.c_double, _P]),
    ("dgp_nlml_grad", C.c_int, [_P, _P, C.c_double, _P, _P]),
    ("dgp_nlml_grad_launch", C.c_int, [_P, _P, C.c_double]),
    ("dgp_nlml_grad_wait", C.c_int, [_P, _P, _P]),
    ("dgp_nlml_grad_ready", C.c_int, [_P]),
    ("dgp_factorize", C.c_int, [_P, _P, C.c_double, _P]),
    ("dgp_predict", C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P]),
    ("dgp_mean_functional_grad", C.c_int, [_P, _P, C.c_int, _P, _P, _P]),
    ("dgp_sample", C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_double, _P, C.c_int]),
    ("dgp_sample_ex", C.c_int, [_P, _P, C.c_int, _P, C.c_ulonglong, C.c_int, C.c_double, C.POINTER(DgpFluxReduce), _P, C.c_int]),
    ("dgp_reserve", C.c_int, [_P, C.c_int, C.c_int, C.c_int]),
    ("dgp_dist_dims", C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_longlong)]),
    ("dgp_dist_begin", C.c_int, [_P, _P, C.c_int, C.c_int, _P, C.c_ulonglong, C.c_double, C.c_int, C.c_int, _P, _P, _P, C.POINTER(_P)]),
    ("dgp_dist_vt_rows", C.c_int, [_P, C.c_int, C.c_int]),
    ("dgp_dist_sigma", C.c_int, [_P]),
    ("dgp_dist_panel_factor", C.c_int, [_P, C.c_int, _P, _P]),
    ("dgp_dist_panel_unpack", C.c_int, [_P, C.c_int, _P]),
    ("dgp_dist_trail", C.c_int, [_P, C.c_int, C.c_int, C.c_int]),
    ("dgp_dist_draws_partial", C.c_int, [_P]),
    ("dgp_dist_finish", C.c_int, [_P, _P]),
    ("dgp_dist_end", C.c_int, [_P]),
    ("dgp_get_alpha", C.c_int, [_P, _P, C.c_int]),
    ("dgp_get_chol", C.c_int, [_P, _P, C.c_int]),
    ("dgp_set_debug_kinv", C.c_int, [_P, C.c_int]),
    ("dgp_get_kinv", C.c_int, [_P, _P, C.c_int]),
    ("dgp_get_linv", C.c_int, [_P, _P, C.c_int]),
    ("dgp_get_uinv", C.c_int, [_P, _P, C.c_int]),
    ("dgp_gemm_nt", C.c_int, [_P, _P, C.c_longlong, _P, C.c_longlong, _P, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int]),
    ("dgp_batch_create", C.c_int, [C.POINTER(_P), C.c_int, C.c_int, C.c_int, _P]),
    ("dgp_batch_destroy", C.c_int, [_P]),
    ("dgp_batch_last_error", C.c_char_p, [_P]),
    ("dgp_batch_workspace_bytes", C.c_size_t, [C.c_int, C.c_int]),
    ("dgp_batch_set_train", C.c_int, [_P, C.POINTER(DgpSpec), C.c_int, _P, _P, _P, _P]),
    ("dgp_batch_nlml_grad", C.c_int, [_P, _P, _P, _P, _P, _P]),
    ("dgp_batch_nlml_grad_launch", C.c_int, [_P, _P, _P]),
    ("dgp_batch_nlml_grad_ready", C.c_int, [_P]),
    ("dgp_batch_nlml_grad_wait", C.c_int, [_P, _P, _P, _P]),
    ("dgp_batch_factorize", C.c_int, [_P, _P, _P, _P, _P]),
    ("dgp_batch_predict", C.c_int, [_P, _P, _P, _P, _P]),
    ("dgp_batch_mean_functional_grad", C.c_int, [_P, _P, _P, _P, _P, _P]),
    ("dgp_batch_get_alpha", C.c_int, [_P, C.c_int, _P]),
    ("dgp_batch_launch_count", C.c_longlong, [_P]),
    ("dgp_batch_set_timing", C.c_int, [_P, C.c_int]),
    ("dgp_batch_last_timing", C.c_int, [_P, _P]),
    ("dgp_launch_count", C.c_longlong, [_P]),
    ("dgp_last_timing", C.c_int, [_P, _P]),
    ("dgp_set_timing", C.c_int, [_P, C.c_int]),
]
EXPORTED_SYMBOLS = [s[0] for s in _SIGNATURES]

_LIB: Optional[C.CDLL] = None


def library_path() -> str:
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "libdgp.so")


def load_library() -> C.CDLL:
    """dlopen libdgp.so and bind every declared symbol; raises if the library was not built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: build the CUDA engine first (python -c 'import __graft_entry__ as g; g.build()'). "
            "discontinuum_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    for name, res, args in _SIGNATURES:
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.dgp_abi_version() != ABI_VERSION:
        raise RuntimeError("libdgp.so ABI version mismatch")
    _LIB = lib
    return lib


class DgpError(RuntimeError):
    pass


def _ptr(a) -> Tuple[int, int]:
    """(address, on_device) of a numpy array or a torch tensor."""
    if isinstance(a, np.ndarray):
        if a.dtype != np.float64 or not a.flags["C_CONTIGUOUS"]:
            raise TypeError("expected a C-contiguous float64 array")
        return a.ctypes.data, 0
    import torch

    if isinstance(a, torch.Tensor):
        if a.dtype != torch.float64 or not a.is_contiguous():
            raise TypeError("expected a contiguous float64 tensor")
        return a.data_ptr(), 1 if a.is_cuda else 0
    raise TypeError(type(a))


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


class BatchEngine:
    """One libdgp batch handle (dgp_batch_*): up to `max_sites` independent sites sharing one covariance spec, evaluated
    by ONE launch sequence per call (NLML + gradient of every site; or factorisation, then posterior prediction of every
    site on its own grid).  Host arrays in, host arrays out."""

    def __init__(self, max_sites: int, max_n: int, device: int = 0, stream: int = 0):
        self.lib = load_library()
        self._h = _P()
        rc = self.lib.dgp_batch_create(C.byref(self._h), int(device), int(max_sites), int(max_n), _P(stream) if stream else None)
        if rc != 0:
            msg = self.lib.dgp_batch_last_error(None)
            self._h = _P()
            raise DgpError(f"dgp_batch_create failed ({rc}): {msg.decode() if msg else ''}")
        self.max_sites, self.max_n, self.device = int(max_sites), int(max_n), int(device)
        self.nsites = 0
        self.ntheta = 0
        self.ns: Sequence[int] = ()

    def _check(self, rc: int, what: str) -> int:
        if rc < 0:
            msg = self.lib.dgp_batch_last_error(self._h)
            raise DgpError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
        return rc

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.dgp_batch_destroy(self._h)
            self._h = _P()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def set_train(self, spec: DgpSpec, sites):
        """sites: sequence of (X[n, ndim], y[n], noise[n]) host arrays, one per site."""
        data = [(_f64(X), _f64(y), _f64(nz)) for X, y, nz in sites]
        G = len(data)
        for X, y, nz in data:
            if X.ndim != 2 or X.shape[1] != spec.ndim or y.shape[0] != X.shape[0] or nz.shape[0] != X.shape[0]:
                raise ValueError("BatchEngine.set_train: X[n, ndim], y[n], noise[n] expected for every site")
        ns = (C.c_int * G)(*[int(d[0].shape[0]) for d in data])
        px = (_P * G)(*[d[0].ctypes.data for d in data])
        py = (_P * G)(*[d[1].ctypes.data for d in data])
        pn = (_P * G)(*[d[2].ctypes.data for d in data])
        self._check(self.lib.dgp_batch_set_train(self._h, C.byref(spec), G, ns, px, py, pn), "dgp_batch_set_train")
        self.nsites, self.ntheta = G, int(spec.ntheta)
        self.ns = [int(v) for v in ns]
        self._keep = spec

    def _args(self, theta, jitter):
        th = _f64(theta)
        if th.shape != (self.nsites, self.ntheta):
            raise ValueError(f"theta must be [{self.nsites}, {self.ntheta}], got {th.shape}")
        jit = None
        if jitter is not None:
            jit = _f64(jitter).reshape(-1)
            if jit.shape[0] != self.nsites:
                raise ValueError("jitter must have one entry per site")
        return th, jit

    def nlml_grad(self, theta, jitter=None):
        """(nlml[G], grad[G, P], info[G]) of every site at theta[G, P] (natural parameters)."""
        self.nlml_grad_launch(theta, jitter)
        return self.nlml_grad_wait()

    def nlml_grad_launch(self, theta, jitter=None):
        th, jit = self._args(theta, jitter)
        self._check(self.lib.dgp_batch_nlml_grad_launch(self._h, th.ctypes.data, jit.ctypes.data if jit is not None else None),
                    "dgp_batch_nlml_grad_launch")

    def nlml_grad_ready(self) -> bool:
        return self._check(self.lib.dgp_batch_nlml_grad_ready(self._h), "dgp_batch_nlml_grad_ready") == 1

    def nlml_grad_wait(self):
        val = np.zeros(self.nsites)
        grad = np.zeros((self.nsites, self.ntheta))
        info = np.zeros(self.nsites, dtype=np.int32)
        self._check(self.lib.dgp_batch_nlml_grad_wait(self._h, val.ctypes.data, grad.ctypes.data, info.ctypes.data),
                    "dgp_batch_nlml_grad_wait")
        return val, grad, info

    def factorize(self, theta, jitter=None):
        """(nlml[G], info[G]): factorise every site at theta[G, P] (+ jitter[G]) for predict (Engine.factorize per site)."""
        th, jit = self._args(theta, jitter)
        val = np.zeros(self.nsites)
        info = np.zeros(self.nsites, dtype=np.int32)
        self._check(self.lib.dgp_batch_factorize(self._h, th.ctypes.data, jit.ctypes.data if jit is not None else None,
                                                 val.ctypes.data, info.ctypes.data), "dgp_batch_factorize")
        return val, info

    def predict(self, grids, want_var: bool = True):
        """Posterior mean and latent variance of every site on its own grid (Engine.predict per site, bit for bit).
        grids: length-G sequence of Xs[m_s, ndim] host arrays, or None to skip a site.  Returns [(mu, var)] per site: var is
        None when want_var is false, (None, None) for a skipped site.  Needs factorize of every predicted site first."""
        if len(grids) != self.nsites:
            raise ValueError(f"predict: {self.nsites} grids (or None) expected, got {len(grids)}")
        G = self.nsites
        xs, out = [], []
        for Xs in grids:
            if Xs is None:
                xs.append(None)
                out.append((None, None))
                continue
            Xs = _f64(Xs)
            if Xs.ndim != 2 or Xs.shape[1] != self._keep.ndim:
                raise ValueError("predict: Xs[m, ndim] expected for every site")
            xs.append(Xs)
            m = int(Xs.shape[0])
            out.append((np.empty(m), np.empty(m) if want_var else None))
        ms = (C.c_int * G)(*[0 if x is None else int(x.shape[0]) for x in xs])
        px = (_P * G)(*[None if x is None or x.shape[0] == 0 else x.ctypes.data for x in xs])
        pm = (_P * G)(*[None if o[0] is None or o[0].shape[0] == 0 else o[0].ctypes.data for o in out])
        pv = (_P * G)(*[None if o[1] is None or o[1].shape[0] == 0 else o[1].ctypes.data for o in out])
        self._check(self.lib.dgp_batch_predict(self._h, ms, px, pm, pv if want_var else None), "dgp_batch_predict")
        return out

    def mean_functional_grad(self, points, c):
        """(val[G], grad[G, P]): F_s = sum_p c[s][p] mu_s(points[s][p]) and dF_s/dtheta_s of every site at the theta of its
        last successful nlml_grad / factorize (Engine.mean_functional_grad per site, bit for bit).  points[s] / c[s] None:
        site skipped (val 0, grad zeros).  At most BATCH_PREDICT_CHUNK points per site."""
        if len(points) != self.nsites or len(c) != self.nsites:
            raise ValueError(f"mean_functional_grad: {self.nsites} point sets and weight vectors (or None) expected")
        G = self.nsites
        xs, cs = [], []
        for Xs, cv in zip(points, c):
            if Xs is None or cv is None:
                xs.append(None)
                cs.append(None)
                continue
            Xs, cv = _f64(Xs), _f64(cv).reshape(-1)
            if Xs.ndim != 2 or Xs.shape[1] != self._keep.ndim or cv.shape[0] != Xs.shape[0]:
                raise ValueError("mean_functional_grad: points[m, ndim] and c[m] expected for every site")
            xs.append(Xs)
            cs.append(cv)
        ms = (C.c_int * G)(*[0 if x is None else int(x.shape[0]) for x in xs])
        px = (_P * G)(*[None if x is None or x.shape[0] == 0 else x.ctypes.data for x in xs])
        pc = (_P * G)(*[None if v is None or v.shape[0] == 0 else v.ctypes.data for v in cs])
        val = np.zeros(G)
        grad = np.zeros((G, self.ntheta))
        self._check(self.lib.dgp_batch_mean_functional_grad(self._h, ms, px, pc, val.ctypes.data, grad.ctypes.data),
                    "dgp_batch_mean_functional_grad")
        return val, grad

    def alpha(self, site: int) -> np.ndarray:
        a = np.empty(self.ns[site])
        self._check(self.lib.dgp_batch_get_alpha(self._h, int(site), a.ctypes.data), "dgp_batch_get_alpha")
        return a

    def set_timing(self, on: bool):
        self._check(self.lib.dgp_batch_set_timing(self._h, 1 if on else 0), "dgp_batch_set_timing")

    def last_timing(self) -> Sequence[float]:
        ms = (C.c_double * 4)()
        self.lib.dgp_batch_last_timing(self._h, ms)
        return list(ms)

    @property
    def launches(self) -> int:
        return int(self.lib.dgp_batch_launch_count(self._h))


class Engine:
    """One libdgp handle: the resident training set of one site and its factorisation workspace."""

    def __init__(self, max_n: int, max_m: int = 2048, device: int = 0, stream: int = 0):
        self.lib = load_library()
        self._h = _P()
        rc = self.lib.dgp_create(C.byref(self._h), int(device), int(max_n), int(max_m), _P(stream) if stream else None)
        if rc != 0:
            msg = self.lib.dgp_last_error(None)
            self._h = _P()
            raise DgpError(f"dgp_create failed ({rc}): {msg.decode() if msg else ''}")
        self.max_n, self.max_m, self.device = int(max_n), int(max_m), int(device)
        self.stream = int(stream)  # 0: the handle created its own stream
        self.n = 0
        self.ntheta = 0
        self._keep = None

    # -- plumbing
    def _check(self, rc: int, what: str) -> int:
        if rc < 0:
            msg = self.lib.dgp_last_error(self._h)
            raise DgpError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
        return rc

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.dgp_destroy(self._h)
            self._h = _P()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    # -- data
    def set_train(self, spec: DgpSpec, X, y, noise):
        if isinstance(X, np.ndarray) or not hasattr(X, "data_ptr"):
            X, y, noise = _f64(X), _f64(y), _f64(noise)
        n = int(X.shape[0])
        if X.ndim != 2 or X.shape[1] != spec.ndim or y.shape[0] != n or noise.shape[0] != n:
            raise ValueError("set_train: X[n, ndim], y[n], noise[n] expected")
        (px, dx), (py, dy), (pn, dn) = _ptr(X), _ptr(y), _ptr(noise)
        if not (dx == dy == dn):
            raise ValueError("set_train: X, y, noise must live on the same side")
        self._check(self.lib.dgp_set_train(self._h, C.byref(spec), px, py, pn, n, dx), "dgp_set_train")
        self.n, self.ntheta, self.ndim = n, int(spec.ntheta), int(spec.ndim)
        self._keep = spec

    def _theta(self, theta) -> np.ndarray:
        th = _f64(theta).reshape(-1)
        if th.shape[0] != self.ntheta:
            raise ValueError(f"theta has {th.shape[0]} entries, spec.ntheta = {self.ntheta}")
        return th

    # -- hot path
    def nlml(self, theta, jitter: float = 0.0) -> Tuple[float, int]:
        th = self._theta(theta)
        out = C.c_double(0.0)
        info = self._check(self.lib.dgp_nlml(self._h, th.ctypes.data, float(jitter), C.addressof(out)), "dgp_nlml")
        return out.value, info

    def nlml_grad(self, theta, jitter: float = 0.0) -> Tuple[float, np.ndarray, int]:
        th = self._theta(theta)
        out = C.c_double(0.0)
        grad = np.zeros(self.ntheta)
        info = self._check(self.lib.dgp_nlml_grad(self._h, th.ctypes.data, float(jitter), C.addressof(out), grad.ctypes.data),
                           "dgp_nlml_grad")
        return out.value, grad, info

    def nlml_grad_launch(self, theta, jitter: float = 0.0):
        th = self._theta(theta)
        self._check(self.lib.dgp_nlml_grad_launch(self._h, th.ctypes.data, float(jitter)), "dgp_nlml_grad_launch")

    def nlml_grad_ready(self) -> bool:
        """Non-blocking: has the evaluation enqueued by nlml_grad_launch finished?"""
        return self._check(self.lib.dgp_nlml_grad_ready(self._h), "dgp_nlml_grad_ready") == 1

    def nlml_grad_wait(self) -> Tuple[float, np.ndarray, int]:
        out = C.c_double(0.0)
        grad = np.zeros(self.ntheta)
        info = self._check(self.lib.dgp_nlml_grad_wait(self._h, C.addressof(out), grad.ctypes.data), "dgp_nlml_grad_wait")
        return out.value, grad, info

    def factorize(self, theta, jitter: float = 0.0) -> Tuple[float, int]:
        th = self._theta(theta)
        out = C.c_double(0.0)
        info = self._check(self.lib.dgp_factorize(self._h, th.ctypes.data, float(jitter), C.addressof(out)), "dgp_factorize")
        return out.value, info

    def predict(self, Xs, want_var: bool = True):
        on_dev = hasattr(Xs, "data_ptr") and Xs.is_cuda
        if not on_dev:
            Xs = _f64(Xs)
        m = int(Xs.shape[0])
        if Xs.ndim != 2 or Xs.shape[1] != self.ndim:
            raise ValueError("predict: Xs[m, ndim] expected")
        if on_dev:
            import torch

            mu = torch.empty(m, dtype=torch.float64, device=Xs.device)
            var = torch.empty(m, dtype=torch.float64, device=Xs.device) if want_var else None
        else:
            mu = np.empty(m)
            var = np.empty(m) if want_var else None
        self._check(self.lib.dgp_predict(self._h, _ptr(Xs)[0], m, 1 if on_dev else 0, _ptr(mu)[0],
                                         _ptr(var)[0] if want_var else None), "dgp_predict")
        return mu, var

    def mean_functional_grad(self, Xs, c) -> Tuple[float, np.ndarray]:
        """F = sum_p c[p] mu(Xs[p]) and dF/dtheta at the theta of the last nlml_grad / factorize."""
        Xs, c = _f64(Xs), _f64(c).reshape(-1)
        if Xs.ndim != 2 or Xs.shape[1] != self.ndim or c.shape[0] != Xs.shape[0]:
            raise ValueError("mean_functional_grad: Xs[m, ndim], c[m] expected")
        val = C.c_double(0.0)
        grad = np.zeros(self.ntheta)
        self._check(self.lib.dgp_mean_functional_grad(self._h, Xs.ctypes.data, int(Xs.shape[0]), c.ctypes.data,
                                                      C.addressof(val), grad.ctypes.data), "dgp_mean_functional_grad")
        return val.value, grad

    def sample(self, Xs, Z, jitter: float = 0.0):
        """(draws[S, m], info): info > 0 means the posterior covariance (+ jitter) was not positive definite.  With Z a CUDA
        tensor, Xs and the draws are CUDA tensors on its device too (nothing of size S x m crosses PCIe)."""
        on_dev = hasattr(Z, "data_ptr") and Z.is_cuda
        if not on_dev and hasattr(Xs, "data_ptr") and Xs.is_cuda:
            raise ValueError("sample: Xs is a CUDA tensor but Z is not; pass Z on the same device to sample there")
        if on_dev:
            import torch

            Xs = torch.as_tensor(Xs, dtype=torch.float64, device=Z.device).contiguous()
        else:
            Xs, Z = _f64(Xs), _f64(Z)
        S, m = Z.shape
        if Xs.ndim != 2 or Xs.shape[0] != m:
            raise ValueError("sample: Z[S, m] and Xs[m, ndim] expected")
        out = torch.empty((S, m), dtype=torch.float64, device=Z.device) if on_dev else np.empty((S, m))
        info = self._check(self.lib.dgp_sample(self._h, _ptr(Xs)[0], m, _ptr(Z)[0], S, float(jitter), _ptr(out)[0],
                                               1 if on_dev else 0), "dgp_sample")
        return out, info

    def sample_ex(self, Xs, S: int, Z=None, seed: int = 0, jitter: float = 0.0, flux: Optional[dict] = None):
        """Draws with device-generated normals (Z=None -> Philox stream `seed`) and / or the grouped flux reduction.
        flux = {"y_mean", "y_scale", "log_transform", "weight"[m], "group_start"[G+1]} -> returns [S, G] instead of [S, m]."""
        Xs = _f64(Xs)
        m = int(Xs.shape[0])
        zp = None
        if Z is not None:
            Z = _f64(Z)
            if Z.shape != (S, m):
                raise ValueError("sample_ex: Z[S, m] expected")
            zp = Z.ctypes.data
        red = None
        if flux is not None:
            w = _f64(flux["weight"]).reshape(-1)
            gs = np.ascontiguousarray(np.asarray(flux["group_start"], dtype=np.int32))
            if w.shape[0] != m:
                raise ValueError("sample_ex: weight[m] expected")
            red = DgpFluxReduce(float(flux["y_mean"]), float(flux["y_scale"]), int(flux.get("log_transform", 1)),
                                int(gs.shape[0] - 1), w.ctypes.data, gs.ctypes.data)
            out = np.empty((S, gs.shape[0] - 1))
        else:
            out = np.empty((S, m))
        info = self._check(self.lib.dgp_sample_ex(self._h, Xs.ctypes.data, m, zp, int(seed), int(S), float(jitter),
                                                  C.byref(red) if red is not None else None, out.ctypes.data, 0), "dgp_sample_ex")
        return out, info

    def reserve(self, max_m_sample: int, max_S: int = 1, max_groups: int = 0):
        """Size the sampling workspace ahead of time (sample / sample_ex / dist_* then allocate nothing); 0 releases it."""
        self._check(self.lib.dgp_reserve(self._h, int(max_m_sample), int(max_S), int(max_groups)), "dgp_reserve")

    # -- distributed sampling primitives (multisite.sample_sharded drives them)
    def dist_dims(self, m: int, S: int, world: int) -> dict:
        d = (C.c_longlong * 6)()
        self._check(self.lib.dgp_dist_dims(self._h, int(m), int(S), int(world), d), "dgp_dist_dims")
        return dict(mpad=int(d[0]), npad=int(d[1]), Spad=int(d[2]), panel_cols=int(d[3]), npanels=int(d[4]), rows_per_rank=int(d[5]))

    def dist_begin(self, Xs, S: int, Z, seed: int, jitter: float, rank: int, world: int, VT, Od, mu):
        """VT / Od / mu: CUDA float64 torch tensors owned by the caller (see include/dgp.h).  Returns a token."""
        Xs = _f64(Xs)
        zp = None
        if Z is not None:
            Z = _f64(Z)
            zp = Z.ctypes.data
        tok = _P()
        self._check(self.lib.dgp_dist_begin(self._h, Xs.ctypes.data, int(Xs.shape[0]), int(S), zp, int(seed), float(jitter),
                                            int(rank), int(world), VT.data_ptr(), Od.data_ptr(), mu.data_ptr(),
                                            C.byref(tok)), "dgp_dist_begin")
        return tok

    def dist_call(self, name: str, tok, *args) -> int:
        return self._check(getattr(self.lib, "dgp_dist_" + name)(tok, *args), "dgp_dist_" + name)

    # -- parity / debug
    def covmat(self, theta) -> np.ndarray:
        th = self._theta(theta)
        K = np.empty((self.n, self.n))
        self._check(self.lib.dgp_covmat(self._h, th.ctypes.data, K.ctypes.data, 0), "dgp_covmat")
        return K

    def cross_covmat(self, theta, Xs) -> np.ndarray:
        th, Xs = self._theta(theta), _f64(Xs)
        K = np.empty((Xs.shape[0], self.n))
        self._check(self.lib.dgp_cross_covmat(self._h, th.ctypes.data, Xs.ctypes.data, Xs.shape[0], 0, K.ctypes.data, 0),
                    "dgp_cross_covmat")
        return K

    def alpha(self) -> np.ndarray:
        a = np.empty(self.n)
        self._check(self.lib.dgp_get_alpha(self._h, a.ctypes.data, 0), "dgp_get_alpha")
        return a

    def _square_out(self, out):
        """(buffer, address, on_device) of an [n, n] result: a new numpy array, or the caller's numpy array or contiguous
        float64 tensor (a CUDA tensor is filled on the device)."""
        if out is None:
            out = np.empty((self.n, self.n))
        if tuple(out.shape) != (self.n, self.n):
            raise ValueError(f"out must be [{self.n}, {self.n}], got {tuple(out.shape)}")
        return (out,) + _ptr(out)

    def chol(self, out=None):
        """L [n, n], lower triangular, of the last evaluation."""
        L, p, dev = self._square_out(out)
        self._check(self.lib.dgp_get_chol(self._h, p, dev), "dgp_get_chol")
        return L

    def set_debug_kinv(self, on: bool):
        self._check(self.lib.dgp_set_debug_kinv(self._h, 1 if on else 0), "dgp_set_debug_kinv")

    def kinv(self, out=None):
        """Ky^-1 [n, n] (lower triangle valid) of the last nlml_grad with set_debug_kinv(True)."""
        Ki, p, dev = self._square_out(out)
        self._check(self.lib.dgp_get_kinv(self._h, p, dev), "dgp_get_kinv")
        return Ki

    def linv(self, out=None):
        """T = L^-1 [n, n], lower triangular, of the last successful factorize."""
        T, p, dev = self._square_out(out)
        self._check(self.lib.dgp_get_linv(self._h, p, dev), "dgp_get_linv")
        return T

    def uinv(self, out=None):
        """U = L^-T [n, n], upper triangular, of the last nlml_grad or factorize (the LAUUM's operand)."""
        U, p, dev = self._square_out(out)
        self._check(self.lib.dgp_get_uinv(self._h, p, dev), "dgp_get_uinv")
        return U

    def gemm_nt(self, A, B, Cm, mode: int = 0):
        """Cm (=, +=, -=) A @ B.T on CUDA float64 tensors (row-major, contiguous)."""
        M, K = A.shape
        N = B.shape[0]
        self._check(self.lib.dgp_gemm_nt(self._h, A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), Cm.data_ptr(),
                                         Cm.stride(0), M, N, K, int(mode)), "dgp_gemm_nt")

    def set_timing(self, on: bool):
        self._check(self.lib.dgp_set_timing(self._h, 1 if on else 0), "dgp_set_timing")

    def last_timing(self) -> Sequence[float]:
        ms = (C.c_double * 4)()
        self.lib.dgp_last_timing(self._h, ms)
        return list(ms)

    @property
    def launches(self) -> int:
        return int(self.lib.dgp_launch_count(self._h))
