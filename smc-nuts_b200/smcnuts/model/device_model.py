"""Device-resident target models with the reference's duck-typed target API.

Replaces smcnuts/model/bridgestan.py:StanModel (reference): `.dim`, `.constrained_dim`, `.param_names`,
`.logpdf(x, phi)`, `.logpdfgrad(x, phi)`, `.constrain(x)`.  The densities are the fused CUDA device
functions of csrc/models.cuh; phi is a kernel argument (the reference rewrites the data JSON on disk and
reloads the Stan model whenever phi changes, bridgestan.py:122-146).

numpy in -> numpy out (host buffers are copied through the device); torch CUDA tensors stay on the device.
"""
import ctypes
import json
import math
from pathlib import Path

import numpy as np

from .. import _cabi, _device as dev

DATA_DIR = Path(__file__).resolve().parents[1] / "data"


class DeviceModel:
    """A built-in model living on the GPU.  `name` in {"arma", "PRMwCD", "gauss"}."""

    def __init__(self, name, host_blob, dim, param_names=None, constrained=True):
        if name not in _cabi.MODEL_KINDS:
            raise ValueError(f"unknown device model {name!r}; built-in models: {sorted(_cabi.MODEL_KINDS)} "
                             "(arbitrary Python/BridgeStan targets cannot run on the device path)")
        self.name = name
        self.dim = int(dim)
        blob = np.ascontiguousarray(host_blob, dtype=np.float64)
        h = ctypes.c_void_p()
        dev.device()
        _cabi.call("smcb_model_create", _cabi.MODEL_KINDS[name], blob.ctypes.data, blob.size, self.dim, ctypes.byref(h))
        self._h = h
        assert _cabi.lib().smcb_model_dim(h) == self.dim
        if constrained:
            # presence of `constrained_dim` selects the constrained estimator branch (estimate.py:25-28)
            self.constrained_dim = self.dim
            self.constrain_kind = _cabi.CONSTRAIN_EXP_LAST
        else:
            self.constrain_kind = _cabi.CONSTRAIN_NONE
        self.param_names = param_names or [f"x.{i + 1}" for i in range(self.dim)]

    @property
    def handle(self):
        return self._h

    def __del__(self):
        try:
            if self._h:
                _cabi.lib().smcb_model_destroy(self._h)
        except Exception:
            pass

    # ---- diagonal metric of the NUTS proposal (README.md:66-67 "future updates" of the reference; identity by default)
    metric_scale = None      # host array [dim] or None
    _scale_dev = None

    def set_metric_scale(self, scale):
        """NUTS on this model then uses the mass matrix diag(1 / scale^2), i.e. identity-metric NUTS on z = x / scale
        (csrc/models.cuh::ScaledModel).  None restores the reference's identity metric."""
        if scale is None:
            _cabi.call("smcb_model_set_scale", self._h, None)
            self.metric_scale = self._scale_dev = None
            return
        sc = np.ascontiguousarray(dev.to_numpy(scale), dtype=np.float64).reshape(self.dim)
        _cabi.call("smcb_model_set_scale", self._h, sc.ctypes.data)
        self.metric_scale, self._scale_dev = sc, dev.to_device(sc)

    # ---- device-native entry points (torch CUDA tensors)
    def split(self, x, grad_phi=None):
        """(A, B[, grad]) with A = log prior + log Jacobian, B = log likelihood; grad = d(A + grad_phi*B)/dx."""
        xd = dev.to_device(x).reshape(-1, self.dim)
        N = xd.shape[0]
        A, B = dev.empty(N), dev.empty(N)
        g = dev.empty(N, self.dim) if grad_phi is not None else None
        _cabi.call("smcb_logp_grad", self._h, dev.ptr(xd), N, float(grad_phi if grad_phi is not None else 1.0),
                   dev.ptr(A), dev.ptr(B), dev.ptr(g), dev.stream_ptr())
        return (A, B, g) if grad_phi is not None else (A, B)

    @staticmethod
    def combine(A, B, phi):
        out = dev.empty(A.shape[0])
        _cabi.call("smcb_combine_logp", dev.ptr(A), dev.ptr(B), float(phi), A.shape[0], dev.ptr(out), dev.stream_ptr())
        return out

    # ---- reference API (bridgestan.py:28-120)
    def logpdf(self, x, phi=1.0, adjust_transform=True):
        single = getattr(x, "ndim", 2) == 1
        A, B = self.split(x)
        lp = self.combine(A, B, phi)
        if single:
            return float(lp[0].item())
        return dev.like_input(lp, x)

    def logpdfgrad(self, x, phi=1.0, adjust_transform=True):
        single = getattr(x, "ndim", 2) == 1
        _, _, g = self.split(x, grad_phi=phi)
        g = dev.like_input(g, x)
        return g[0] if single else g

    def constrain(self, x, include_tparams=True, include_gqs=True):
        """Identity except exp() on the last coordinate for arma / PRMwCD (sigma, Gamma); host-side helper
        only -- the estimators fuse this transform into the moment kernel."""
        if dev.is_host(x):
            c = np.array(x, dtype=np.float64, copy=True)
            if self.constrain_kind == _cabi.CONSTRAIN_EXP_LAST:
                c[..., -1] = np.exp(c[..., -1])
            return c
        c = x.clone()
        if self.constrain_kind == _cabi.CONSTRAIN_EXP_LAST:
            c[..., -1] = c[..., -1].exp()
        return c


def arma_model(y=None):
    """ARMA(1,1) of stan_models/arma/arma.stan with the shipped arma.json data (T = 200)."""
    if y is None:
        y = json.loads((DATA_DIR / "arma" / "arma.json").read_text())["y"]
    return DeviceModel("arma", np.asarray(y, dtype=np.float64), 4, ["mu", "beta", "theta", "sigma"])


def prmwcd_model(data=None):
    """Poisson regression with exponential-power prior of stan_models/PRMwCD/PRMwCD.stan (repaired JSON)."""
    if data is None:
        data = json.loads((DATA_DIR / "PRMwCD" / "PRMwCD.json").read_text())
    no, m, c = int(data["N"]), int(data["M"]), int(data["Clength"])
    if (m, c) != (12, 11):
        raise ValueError("the PRMwCD device function is specialised to M = 12, Clength = 11")
    y = np.asarray(data["y"], dtype=np.float64)
    lg = np.array([math.lgamma(v + 1.0) for v in y])
    X = np.asarray(data["Xkernel"], dtype=np.float64)
    assert X.size == no * c
    blob = np.concatenate([[float(data["q"])], y, lg, X])
    return DeviceModel("PRMwCD", blob, 13, [f"Beta.{i}" for i in range(1, 13)] + ["Gamma"])


def gauss_model(dim=100, rho=0.9, precision=None):
    """Synthetic correlated Gaussian (BASELINE.json config 4): Sigma_ij = rho^|i-j|, dense precision."""
    if precision is None:
        idx = np.arange(dim)
        precision = np.linalg.inv(rho ** np.abs(idx[:, None] - idx[None, :]))
    P = np.asarray(precision, dtype=np.float64)
    # the kernels read P as given: the plain one forms -P x, the tensor-core one -P'x; with P symmetric both are the
    # gradient of B = -x'Px/2 (and this is the matrix oracle.models.GaussTarget uses)
    P = 0.5 * (P + P.T)
    return DeviceModel("gauss", P.ravel(), P.shape[0], constrained=False)


def make_model(name, **kw):
    return {"arma": arma_model, "PRMwCD": prmwcd_model, "gauss": gauss_model}[name](**kw)
