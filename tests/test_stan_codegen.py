"""Generic Stan-model ingestion (SURVEY.md section 8 f3; reference: smcnuts/model/bridgestan.py:13-26 hands any Stan
program to BridgeStan).  CPU: the generated model struct is compiled with g++ and checked against the oracle densities,
an independent scipy.stats restatement and finite differences.  GPU: the generated model runs through the NUTS / SMC
kernels as a plug-in and is compared with the hand-written arma device function."""
import ctypes
import importlib.util
import json
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import smc_oracle as O

ROOT = Path(__file__).resolve().parents[1]
STAN = ROOT / "tests" / "stan"
CSRC = ROOT / "smc-nuts_b200" / "csrc"
DATA = ROOT / "smc-nuts_b200" / "smcnuts" / "data"
# programs of the original SMC-NUTS project (stan_models/<name>/<name>.stan), stored as <name>.stan
REF_STAN = ROOT / "tests" / "golden" / "reference_stan"


def _codegen():
    spec = importlib.util.spec_from_file_location("smcb_stan_codegen", ROOT / "smc-nuts_b200/smcnuts/model/stan_codegen.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


SC = _codegen()
HOST_HARNESS = r'''
#include "common.cuh"
#include "models.cuh"
#include "model_gen.h"
extern "C" void gen_logp(const double* x, long N, double phi, const double* blob, double* A, double* B, double* g) {
    smcb::ModelDesc d{}; d.data = blob; d.dim = GenModel::DMAX;
    GenModel m(d, blob);
    for (long i = 0; i < N; ++i) {
        double xv[GenModel::DMAX], gv[GenModel::DMAX];
        for (int k = 0; k < GenModel::DMAX; ++k) xv[k] = x[i * GenModel::DMAX + k];
        m.eval(xv, phi, A[i], B[i], gv);
        for (int k = 0; k < GenModel::DMAX; ++k) g[i * GenModel::DMAX + k] = gv[k];
    }
}
'''


class HostModel:
    """The generated struct compiled for the host (the same text nvcc compiles for the device)."""

    def __init__(self, src, tmp_path):
        tmp_path.mkdir(parents=True, exist_ok=True)
        (tmp_path / "model_gen.h").write_text(src.text)
        (tmp_path / "host.cpp").write_text(HOST_HARNESS)
        so = tmp_path / "libgen.so"
        subprocess.run(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-std=c++17", f"-I{CSRC}", f"-I{tmp_path}",
                        str(tmp_path / "host.cpp"), "-o", str(so)], check=True, capture_output=True)
        self.lib = ctypes.CDLL(str(so))
        self.lib.gen_logp.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_double] + [ctypes.c_void_p] * 4
        self.blob = np.array(src.blob if src.blob else [0.0])
        self.dim = src.dim

    def split(self, x, phi=1.0):
        x = np.ascontiguousarray(x, dtype=np.float64)
        n = len(x)
        A, B, g = np.empty(n), np.empty(n), np.empty((n, self.dim))
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
        self.lib.gen_logp(p(x), n, float(phi), p(self.blob), p(A), p(B), p(g))
        return A, B, g


def _arma_data():
    return {"T": 200, "y": json.loads((ROOT / "smc-nuts_b200/smcnuts/data/arma/arma.json").read_text())["y"]}


def test_generated_arma_matches_oracle(tmp_path):
    src = SC.generate((STAN / "arma11.stan").read_text(), _arma_data())
    assert src.dim == 4 and src.param_names == ["mu", "beta", "theta", "sigma"]
    assert [t[0] for t in src.transforms] == ["none", "none", "none", "lower"]
    h = HostModel(src, tmp_path)
    rng = np.random.default_rng(0)
    x = rng.normal(size=(300, 4)) * 0.5
    t = O.COracleTarget("arma")
    A, B, g = h.split(x, 0.6)
    Ao, Bo, _, _ = t.split(x, grads=False)
    np.testing.assert_allclose(A, Ao, rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(B, Bo, rtol=1e-12)
    np.testing.assert_allclose(g, t.logpdfgrad(x, 0.6), rtol=1e-10, atol=1e-9)


@pytest.mark.parametrize("name", ["arma", pytest.param("PRMwCD", marks=pytest.mark.skip(
    reason="the original PRMwCD.stan is not stored in tests/golden/reference_stan"))])
def test_reference_stan_programs_translate_to_the_oracle_densities(tmp_path, name):
    """The mechanical translation of the reference's own .stan text agrees with the hand restatement of the oracle:
    an independent pin of the model arithmetic (BridgeStan itself is not installable offline)."""
    src = SC.generate((REF_STAN / f"{name}.stan").read_text(), SC.load_data(DATA / name / f"{name}.json"))
    h = HostModel(src, tmp_path)
    t = O.COracleTarget(name)
    assert src.dim == t.dim
    rng = np.random.default_rng(1)
    x = rng.normal(size=(400, src.dim)) * 0.7
    for phi in (0.0, 0.37, 1.0):
        A, B, g = h.split(x, phi)
        Ao, Bo, _, _ = t.split(x, grads=False)
        np.testing.assert_allclose(A, Ao, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(B, Bo, rtol=1e-12, atol=1e-10)
        np.testing.assert_allclose(g, t.logpdfgrad(x, phi), rtol=1e-9, atol=1e-8)


def _logistic_data(rng):
    return {"N": 30, "K": 3, "y": rng.integers(0, 2, 30).tolist(), "X": rng.normal(size=90).tolist()}


def test_generated_logistic_matches_scipy_restatement_and_finite_differences(tmp_path):
    from scipy import stats
    from scipy.special import expit
    rng = np.random.default_rng(2)
    data = _logistic_data(rng)
    src = SC.generate((STAN / "logistic.stan").read_text(), data)
    assert src.dim == 6 and src.param_names == ["alpha", "w.1", "w.2", "w.3", "tau", "rho"]
    assert [t[0] for t in src.transforms] == ["none"] * 4 + ["lower", "both"]
    h = HostModel(src, tmp_path)
    X, y = np.array(data["X"]).reshape(30, 3), np.array(data["y"])
    x = rng.normal(size=(50, 6)) * 0.8

    def restated(u):
        alpha, w, tau, s = u[0], u[1:4], np.exp(u[4]), expit(u[5])
        rho = -1.0 + 3.0 * s
        # `~` statements: Stan drops the parameter-free terms (here: the exponential's log rate, the Student-t's
        # normaliser, the N(0, tau) 2 pi constants and the whole constant uniform density); Jacobians are kept
        prior = -1.5 * tau + (stats.t.logpdf(alpha, 4, 0, 2.5) - stats.t.logpdf(0.0, 4, 0, 2.5)) \
            + np.sum(-np.log(tau) - 0.5 * (w / tau) ** 2)
        jac = u[4] + np.log(3.0) + np.log(s) + np.log1p(-s)
        eta = alpha + rho + X @ w
        return prior + jac, np.sum(stats.bernoulli.logpmf(y, expit(eta)))

    A, B, g = h.split(x, 0.7)
    ref = np.array([restated(u) for u in x])
    np.testing.assert_allclose(A, ref[:, 0], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(B, ref[:, 1], rtol=1e-12, atol=1e-12)
    eps = 1e-6
    for k in range(6):
        xp, xm = x.copy(), x.copy()
        xp[:, k] += eps; xm[:, k] -= eps
        Ap, Bp, _ = h.split(xp, 0.7)
        Am, Bm, _ = h.split(xm, 0.7)
        fd = ((Ap + 0.7 * Bp) - (Am + 0.7 * Bm)) / (2 * eps)
        np.testing.assert_allclose(g[:, k], fd, rtol=2e-6, atol=2e-6)


def test_generated_mixed_program_matches_a_numpy_restatement_and_finite_differences(tmp_path):
    """Every parameter bound kind, local arrays, compound assignments on a loop-carried local, seven densities."""
    from scipy import stats
    from scipy.special import expit, gammaln
    rng = np.random.default_rng(4)
    N = 12
    data = {"N": N, "t": rng.normal(size=N).tolist(), "y": rng.lognormal(size=N).tolist(), "k": rng.integers(0, 6, N).tolist()}
    src = SC.generate((STAN / "mixed.stan").read_text(), data)
    assert src.dim == 6 and [t[0] for t in src.transforms] == ["lower", "upper", "both", "none", "lower", "lower"]
    h = HostModel(src, tmp_path)
    t, y, k = np.array(data["t"]), np.array(data["y"]), np.array(data["k"])

    def restated(u):
        a, b, p, c = np.exp(u[0]), 3.0 - np.exp(u[1]), expit(u[2]), u[3]
        s = 0.5 + np.exp(u[4:6])
        jac = u[0] + u[1] + np.log(p) + np.log1p(-p) + u[4] + u[5]
        # `~` statements drop their parameter-free terms
        A = (-np.log(a) - 0.5 * ((np.log(a) - 0.2) / 0.7) ** 2) \
            + stats.norm.logpdf(b, 1, 2) + stats.laplace.logpdf(c, 0, 1.5) \
            + (1.5 * np.log(p) + 0.5 * np.log1p(-p)) + np.sum(2 * np.log(s) - 2 * s) + jac
        acc, B = 0.0, 0.0
        for n in range(N):
            m = a * np.exp(-t[n] ** 2 / s[0]) + s[1] ** 1.5 * p
            acc = (acc + 0.1 * m) * 0.9
            sd = 0.3 + expit(c)
            B += stats.lognorm.logpdf(y[n], sd, scale=np.exp(np.log(m) + 0.01 * acc))
            eta = np.logaddexp(b, c) - 2.0
            B += k[n] * eta - np.exp(eta) - gammaln(k[n] + 1.0)
        A += -0.5 * acc * acc / 100.0
        return A, B

    x = rng.normal(size=(40, 6)) * 0.6
    A, B, g = h.split(x, 0.45)
    ref = np.array([restated(u) for u in x])
    np.testing.assert_allclose(A, ref[:, 0], rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(B, ref[:, 1], rtol=1e-11, atol=1e-11)
    eps = 1e-6
    for j in range(6):
        xp, xm = x.copy(), x.copy()
        xp[:, j] += eps; xm[:, j] -= eps
        Ap, Bp, _ = h.split(xp, 0.45)
        Am, Bm, _ = h.split(xm, 0.45)
        np.testing.assert_allclose(g[:, j], ((Ap + 0.45 * Bp) - (Am + 0.45 * Bm)) / (2 * eps), rtol=5e-6, atol=5e-6)


def _fd_check(h, x, g, phi, dim, tol=5e-6):
    eps = 1e-6
    for j in range(dim):
        xp, xm = x.copy(), x.copy()
        xp[:, j] += eps; xm[:, j] -= eps
        Ap, Bp, _ = h.split(xp, phi)
        Am, Bm, _ = h.split(xm, phi)
        np.testing.assert_allclose(g[:, j], ((Ap + phi * Bp) - (Am + phi * Bm)) / (2 * eps), rtol=tol, atol=tol)


def _regression_data(rng, N=9, K=3):
    return {"N": N, "K": K, "X": rng.normal(size=(N, K)).tolist(), "y": rng.normal(size=N).tolist()}


def test_generated_regression_with_matrix_product_and_transformed_blocks(tmp_path):
    """matrix * vector, transformed data (folded integer, real scalar, rep_vector), transformed parameters with a vector
    initialiser, an elementwise product inside a density argument, generated quantities skipped."""
    from scipy import stats
    rng = np.random.default_rng(7)
    data = _regression_data(rng)
    src = SC.generate((STAN / "regression.stan").read_text(), data)
    assert src.dim == 5 and src.param_names == ["alpha", "beta.1", "beta.2", "beta.3", "sigma"]
    h = HostModel(src, tmp_path)
    X, y = np.array(data["X"]), np.array(data["y"])

    def restated(u):
        alpha, beta, sigma = u[0], u[1:4], np.exp(u[4])
        A = np.sum(-0.5 * beta ** 2) - 0.5 * (alpha / 5.0) ** 2 - sigma + u[4] - 0.5 * np.sum(np.diff(beta) ** 2)
        mu = alpha + X @ beta
        return A, np.sum(stats.norm.logpdf(y, mu * 1.0, sigma))

    x = rng.normal(size=(40, 5)) * 0.7
    A, B, g = h.split(x, 0.6)
    ref = np.array([restated(u) for u in x])
    np.testing.assert_allclose(A, ref[:, 0], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(B, ref[:, 1], rtol=1e-12, atol=1e-12)
    _fd_check(h, x, g, 0.6, 5)


def _containers_data(rng, robust, N=8, K=3):
    trials = rng.integers(1, 9, N)
    return {"N": N, "K": K, "x": rng.normal(size=(N, K)).tolist(), "z": rng.integers(0, 2, N).tolist(),
            "trials": trials.tolist(), "wins": rng.binomial(trials, 0.4).tolist(), "t": rng.normal(size=N).tolist(),
            "robust": robust}


@pytest.mark.parametrize("robust", [0, 1])
def test_generated_container_expressions_match_a_numpy_restatement(tmp_path, robust):
    """row_vector * vector, .* and ./, mean / sum / dot_self / dot_product, exp of a vector, densities of vector
    expressions (in `target +=` and in `~`), if / else on a data flag and on parameter values, four more densities."""
    from scipy import stats
    from scipy.special import expit
    rng = np.random.default_rng(11)
    data = _containers_data(rng, robust)
    src = SC.generate((STAN / "containers.stan").read_text(), data)
    assert src.dim == 6
    h = HostModel(src, tmp_path)
    X, z, t = np.array(data["x"]), np.array(data["z"]), np.array(data["t"])
    trials, wins = np.array(data["trials"]), np.array(data["wins"])

    def restated(u):
        b, tau, c, p = u[0:3], np.exp(u[3]), u[4], expit(u[5])
        jac = u[3] + np.log(p) + np.log1p(-p)
        zc = (c - 0.5) / 1.5
        # `~` statements keep only the parameter-dependent terms
        A = np.sum(-0.5 * (b / 2.0) ** 2) + (0.5 * (np.log(tau) - np.log(2.0)) - (tau / 2.0) ** 1.5) \
            + (-zc - 2.0 * np.logaddexp(0.0, -zc)) + np.sum(wins * np.log(p) + (trials - wins) * np.log1p(-p)) + jac
        eta = X @ b + c
        loc = eta * t - eta.mean()
        B = np.sum(stats.t.logpdf(t, 4, loc, tau)) if robust else np.sum(stats.norm.logpdf(t, loc, tau))
        e2 = eta / (1.0 + tau)
        A += np.sum(z * e2 - np.logaddexp(0.0, e2))
        A += -0.5 * (b @ b) / 10 + 0.01 * np.sum(np.exp(-eta)) - 0.1 * np.sum(b ** 3)
        A += -c if (c > 0 and not tau >= 10) else c
        return A, B

    x = rng.normal(size=(60, 6)) * 0.7
    assert (x[:, 4] > 0).any() and (x[:, 4] < 0).any()
    A, B, g = h.split(x, 0.35)
    ref = np.array([restated(u) for u in x])
    np.testing.assert_allclose(A, ref[:, 0], rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(B, ref[:, 1], rtol=1e-11, atol=1e-11)
    _fd_check(h, x, g, 0.35, 6)


_EIGHT_SCHOOLS = """
data { int<lower=0> J; array[J] real y; array[J] real<lower=0> sigma; }
parameters { real mu; real<lower=0> tau; vector[J] theta_tilde; }
transformed parameters { vector[J] theta = mu + tau * theta_tilde; }
model { mu ~ normal(0, 5); tau ~ cauchy(0, 5); theta_tilde ~ std_normal(); y ~ normal(theta, sigma); }
"""
_POISSON_GLM = """
data { int N; int K; matrix[N, K] X; array[N] int<lower=0> y; real phi; }
parameters { real alpha; vector[K] beta; }
model {
  vector[N] eta;
  eta = X * beta;
  eta += alpha;
  alpha ~ normal(0, 1); beta ~ normal(0, 1);
  target += phi * poisson_log_lpmf(y | eta);
  target += sum(log1p_exp(beta)) - mean(beta);
  for (n in 1:N) target += 0.01 * normal_lpdf(y[n] | X[n] * beta + alpha, 2);
}
"""
_PROJECTIONS = """
data { int N; int K; matrix[K, N] W; row_vector[K] r0; vector[N] t; real phi; }
parameters { row_vector[K] r; real<lower=0> s; }
model {
  row_vector[N] proj = (r + r0) * W;
  vector[N] v;
  for (n in 1:N) {
    if (n <= 2) v[n] = proj[n] * 2; else v[n] = proj[n] - sum(r .* r0);
  }
  target += 0.5 * normal_lpdf(t | v ./ (1 + s), rep_vector(1.5, N)) - dot_self(r);
  target += phi * (-0.5 * dot_product(v, t) * dot_product(v, t) / 100);
  s ~ gamma(2, 2);
}
"""


@pytest.mark.parametrize("case", ["eight_schools", "poisson_glm", "projections"])
def test_generated_idiomatic_programs_match_numpy_restatements(tmp_path, case):
    """Programs written the way Stan users write them (non-centred eight schools; a Poisson GLM with matrix * vector, a
    compound whole-vector assignment and a row slice of a matrix inside a loop; row_vector * matrix with if / else on the
    loop variable and a density of a vector expression inside a larger expression)."""
    from scipy import stats
    from scipy.special import gammaln
    rng = np.random.default_rng(0)
    if case == "eight_schools":
        y, sd = np.array([28., 8., -3., 7., -1., 1., 18., 12.]), np.array([15., 10., 16., 11., 9., 11., 10., 18.])
        text, data, dim = _EIGHT_SCHOOLS, {"J": 8, "y": y.tolist(), "sigma": sd.tolist()}, 10

        def restated(u):
            mu, tau, tt = u[0], np.exp(u[1]), u[2:]
            th = mu + tau * tt
            return (-0.5 * (mu / 5) ** 2 - np.log1p((tau / 5) ** 2) + u[1] - 0.5 * np.sum(tt ** 2)
                    - 0.5 * np.sum(((y - th) / sd) ** 2)), 0.0
    elif case == "poisson_glm":
        N, K = 10, 2
        X, y = rng.normal(size=(N, K)), rng.poisson(2.0, N)
        text, data, dim = _POISSON_GLM, {"N": N, "K": K, "X": X.tolist(), "y": y.tolist()}, 3

        def restated(u):
            a, b = u[0], u[1:]
            eta = X @ b + a
            A = -0.5 * a * a - 0.5 * np.sum(b * b) + np.sum(np.logaddexp(0, b)) - b.mean() \
                + 0.01 * np.sum(stats.norm.logpdf(y, eta, 2))
            return A, np.sum(y * eta - np.exp(eta) - gammaln(y + 1.0))
    else:
        W, r0, t = rng.normal(size=(2, 5)), rng.normal(size=2), rng.normal(size=5)
        text, data, dim = _PROJECTIONS, {"N": 5, "K": 2, "W": W.tolist(), "r0": r0.tolist(), "t": t.tolist()}, 3

        def restated(u):
            r, s = u[:2], np.exp(u[2])
            proj = (r + r0) @ W
            v = np.where(np.arange(1, 6) <= 2, proj * 2, proj - np.sum(r * r0))
            A = 0.5 * np.sum(stats.norm.logpdf(t, v / (1 + s), 1.5)) - r @ r + (np.log(s) - 2 * s) + u[2]
            return A, -0.5 * (v @ t) ** 2 / 100
    src = SC.generate(text, data)
    assert src.dim == dim
    h = HostModel(src, tmp_path)
    x = np.random.default_rng(3).normal(size=(30, dim)) * 0.6
    A, B, g = h.split(x, 0.4)
    ref = np.array([restated(u) for u in x])
    np.testing.assert_allclose(A, ref[:, 0], rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(B, ref[:, 1], rtol=1e-11, atol=1e-11)
    _fd_check(h, x, g, 0.4, dim)


_SHAPES = """
data { int N; vector<lower=0>[N] w; array[N] int<lower=0> k; real phi; }
parameters { real<lower=0> a; real<lower=0> b; real<lower=1> nu; real<lower=0> disp; real m; }
model {
  a ~ gamma(2, 1); b ~ exponential(0.5); nu ~ gamma(2, 0.1); disp ~ lognormal(0, 1); m ~ student_t(nu, 0, 2);
  target += phi * gamma_lpdf(w | a, b);
  k ~ neg_binomial_2(exp(m), disp);
  target += 0.1 * neg_binomial_2_log_lpmf(k | m - 0.5, disp + 1) + 0.01 * lgamma(a + b);
}
"""


def test_generated_densities_with_parameter_dependent_shapes_use_the_digamma_series(tmp_path):
    """lgamma of parameter-dependent arguments (gamma shape, Student-t degrees of freedom, negative-binomial dispersion):
    values against scipy.stats, gradients against finite differences, the digamma series against scipy.special."""
    from scipy import stats
    from scipy.special import gammaln
    rng = np.random.default_rng(5)
    N = 9
    w, k = rng.gamma(2.0, 1.0, N), rng.poisson(3.0, N)
    src = SC.generate(_SHAPES, {"N": N, "w": w.tolist(), "k": k.tolist()})
    assert src.dim == 5
    h = HostModel(src, tmp_path)

    def nb2(kk, mu, ph):
        return np.sum(gammaln(kk + ph) - gammaln(kk + 1.0) - gammaln(ph) + kk * np.log(mu / (mu + ph)) + ph * np.log(ph / (mu + ph)))

    def restated(u):
        a, b, nu, disp, m = np.exp(u[0]), np.exp(u[1]), 1.0 + np.exp(u[2]), np.exp(u[3]), u[4]
        jac = u[0] + u[1] + u[2] + u[3]
        A = (np.log(a) - a) + (-0.5 * b) + (np.log(nu) - 0.1 * nu) + (-np.log(disp) - 0.5 * np.log(disp) ** 2) \
            + (stats.t.logpdf(m, nu, 0, 2) + np.log(2.0)) + jac
        A += nb2(k, np.exp(m), disp) + np.sum(gammaln(k + 1.0))            # `~` drops the parameter-free log k!
        A += 0.1 * nb2(k, np.exp(m - 0.5), disp + 1) + 0.01 * gammaln(a + b)
        return A, np.sum(stats.gamma.logpdf(w, a, scale=1.0 / b))

    x = rng.normal(size=(40, 5)) * 0.6
    A, B, g = h.split(x, 0.8)
    ref = np.array([restated(u) for u in x])
    np.testing.assert_allclose(A, ref[:, 0], rtol=1e-11, atol=1e-10)
    np.testing.assert_allclose(B, ref[:, 1], rtol=1e-11, atol=1e-10)
    _fd_check(h, x, g, 0.8, 5, tol=2e-5)


def test_local_arrays_become_scalars_only_when_every_read_sees_the_latest_write(tmp_path):
    """Scalar replacement of model-block arrays (values and sensitivities in registers instead of per-thread local
    memory): applied to `v[t] = ...; use v[t]`, refused when another element is read, when the write sits in a branch and
    for loop-carried reads -- and the refused program still evaluates correctly."""
    import re

    def arrays(text):
        return sorted(set(re.findall(r"double (v_\w+)\[\d+\]", SC.generate(text, {"T": 5}).text)))
    head = "data { int T; } parameters { real a; } model { vector[T] v; "
    reads_other = head + "v[1] = a; for (t in 2:T) { v[t] = v[1] + t; target += -v[t] * v[t]; } }"
    assert arrays(reads_other) == ["v_v"]
    assert arrays(head + "v[1] = a; target += -v[1] * v[1]; for (t in 2:T) { v[t] = a + t; target += -v[t] * v[t]; } }") == []
    assert arrays(head + "for (t in 1:T) { if (t < 3) v[t] = a; else v[t] = 2 * a; target += -v[t] * v[t]; } }") == ["v_v"]
    # the previous element is the latest write on entry of every trip: a rolling scalar ...
    rolling = head + "v[1] = a; for (t in 2:T) { v[t] = v[t - 1] * 0.5 + t; target += -v[t] * v[t - 1]; } }"
    assert arrays(rolling.replace(" * v[t - 1]", "")) == []
    assert arrays(rolling) == ["v_v"]            # ... unless it is read again after this trip's write
    assert arrays(head + "v[2] = a; for (t in 2:T) { v[t] = v[t - 1] * 0.5; target += -v[t]; } }") == ["v_v"]
    hr = HostModel(SC.generate(rolling.replace(" * v[t - 1]", ""), {"T": 5}), tmp_path / "r")
    h = HostModel(SC.generate(reads_other, {"T": 5}), tmp_path)
    x = np.linspace(-1.0, 1.0, 7)[:, None]
    Ar, _, gr = hr.split(x, 1.0)
    v, dv, want, dwant = x[:, 0].copy(), np.ones(7), 0.0, 0.0
    for t in range(2, 6):
        v, dv = v * 0.5 + t, dv * 0.5
        want, dwant = want - v, dwant - dv
    np.testing.assert_allclose(Ar, want, rtol=1e-14)
    np.testing.assert_allclose(gr[:, 0], dwant, rtol=1e-14)
    A, B, g = h.split(x, 1.0)
    np.testing.assert_allclose(A, -sum((x[:, 0] + t) ** 2 for t in range(2, 6)), rtol=1e-14)
    np.testing.assert_allclose(g[:, 0], -sum(2 * (x[:, 0] + t) for t in range(2, 6)), rtol=1e-14)


def test_trailing_vectorised_density_is_fused_into_the_loop_that_fills_its_vector(tmp_path):
    """`for (t in 2:T) { ...; resid[t] = ...; }  target += phi * normal_lpdf(resid | 0, sigma);` keeps no per-thread series:
    the density is applied where each element is written and the vectors reduce to rolling scalars; programs where that
    would be wrong (an argument that is a model-block local, elements written twice or not at all by the recognised
    writes) keep their arrays -- and all of them evaluate to the same numbers."""
    import re
    src = SC.generate((STAN / "arma_series.stan").read_text(), _arma_data())
    assert not re.findall(r"double v_\w+\[\d+\]", src.text)
    h = HostModel(src, tmp_path / "series")       # one directory per library: dlopen caches by path
    t = O.COracleTarget("arma")
    x = np.random.default_rng(1).normal(size=(200, 4)) * 0.7
    A, B, g = h.split(x, 0.37)
    Ao, Bo, _, _ = t.split(x, grads=False)
    np.testing.assert_allclose(A, Ao, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(B, Bo, rtol=1e-12, atol=1e-10)
    np.testing.assert_allclose(g, t.logpdfgrad(x, 0.37), rtol=1e-9, atol=1e-8)
    # not fusable: the scale is a local assigned after the loop / element 1 is never written / element 2 is written twice
    head = "data { int T; vector[T] y; } parameters { real a; real<lower=0> s; } model { vector[T] v; "
    loop = "for (t in 2:T) { v[t] = y[t] - a * v[t - 1]; } "
    variants = {
        "fused": head + "v[1] = y[1]; " + loop + "target += normal_lpdf(v | 0, s); }",
        "local scale": head + "real s2; v[1] = y[1]; " + loop + "s2 = 2 * s; target += normal_lpdf(v | 0, s2 / 2); }",
        "twice": head + "v[1] = y[1]; v[2] = 0; " + loop + "target += normal_lpdf(v | 0, s); }",
    }
    data = {"T": 6, "y": np.random.default_rng(2).normal(size=6).tolist()}
    xs = np.random.default_rng(3).normal(size=(20, 2)) * 0.5
    results = {}
    for name, text in variants.items():
        sv = SC.generate(text, data)
        assert bool(re.findall(r"double v_v\[\d+\]", sv.text)) == (name != "fused"), name
        results[name] = HostModel(sv, tmp_path / name.replace(" ", "_")).split(xs, 1.0)
    for name in ("local scale", "twice"):
        for got, want in zip(results[name], results["fused"]):
            np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-13)
    # an element that no recognised write covers: not fused either (Stan would report the NaN element at run time)
    assert re.findall(r"double v_v\[\d+\]", SC.generate(head + loop + "target += normal_lpdf(v | 0, s); }", data).text)


_FUNCTIONS = """
functions {
  real huber(real r, real k) {
    real a = fabs(r);
    real out;
    if (a <= k) out = 0.5 * r * r; else out = k * (a - 0.5 * k);
    return out;
  }
  real wsum(vector v, vector w, int n) {
    real acc = 0;
    for (i in 1:n) acc += v[i] * w[i];
    return acc / n;
  }
  real twice(real x) { return 2 * huber(x, 1.0) + fmax(x, 0.3) - fmin(x * x, 2.0); }
}
data { int N; vector[N] y; vector[N] w; real phi; }
parameters { real m; real<lower=0> s; vector[N] z; }
model {
  z ~ std_normal();
  s ~ exponential(1);
  for (n in 1:N) { target += phi * (-huber((y[n] - m) / s, 1.5)); target += -log(s); }
  target += -0.1 * wsum(z, w, N) - 0.01 * twice(m) + 0.001 * wsum(z .* z, w, N);
}
"""


def test_user_defined_functions_are_inlined(tmp_path):
    """Functions returning real: scalar arguments given as expressions, an integer size, containers bound by name and
    a container expression materialised first, if / else and a loop in the body, a function calling another one."""
    rng = np.random.default_rng(0)
    N = 5
    data = {"N": N, "y": rng.normal(size=N).tolist(), "w": rng.random(N).tolist()}
    src = SC.generate(_FUNCTIONS, data)
    y, w = np.array(data["y"]), np.array(data["w"])

    def hub(r, k):
        return 0.5 * r * r if abs(r) <= k else k * (abs(r) - 0.5 * k)

    def restated(u):
        m, s, z = u[0], np.exp(u[1]), u[2:]
        A = -0.5 * np.sum(z * z) - s + u[1] - N * np.log(s) - 0.1 * np.sum(z * w) / N \
            - 0.01 * (2 * hub(m, 1.0) + max(m, 0.3) - min(m * m, 2.0)) \
            + 0.001 * np.sum(z * z * w) / N
        return A, -sum(hub((y[n] - m) / s, 1.5) for n in range(N))
    h = HostModel(src, tmp_path)
    x = rng.normal(size=(30, 2 + N)) * 0.8
    A, B, g = h.split(x, 0.6)
    ref = np.array([restated(u) for u in x])
    np.testing.assert_allclose(A, ref[:, 0], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(B, ref[:, 1], rtol=1e-12, atol=1e-12)
    _fd_check(h, x, g, 0.6, 2 + N, tol=2e-5)


def test_generated_prm_kernel_program_matches_the_oracle(tmp_path):
    """The second shipped model re-phrased (log-rate accumulator, poisson_log, pow): against the oracle's PRMwCD density."""
    data = json.loads((ROOT / "smc-nuts_b200/smcnuts/data/PRMwCD/PRMwCD.json").read_text())
    data.pop("phi")
    src = SC.generate((STAN / "prm_kernel.stan").read_text(), data)
    t = O.COracleTarget("PRMwCD")
    assert src.dim == t.dim == 13
    h = HostModel(src, tmp_path)
    x = np.random.default_rng(1).normal(size=(200, 13)) * 0.7
    for phi in (0.0, 0.37, 1.0):
        A, B, g = h.split(x, phi)
        Ao, Bo, _, _ = t.split(x, grads=False)
        np.testing.assert_allclose(A, Ao, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(B, Bo, rtol=1e-12, atol=1e-10)
        np.testing.assert_allclose(g, t.logpdfgrad(x, phi), rtol=1e-9, atol=1e-8)


def test_builtin_device_functions_are_only_used_for_the_shipped_program_text():
    """StanModel("arma", path, ...) runs the hand-tuned device function only when the file IS the reference's program
    (comments and white space aside); an edited file of the same name goes through the generator."""
    import sys
    sys.path.insert(0, str(ROOT / "smc-nuts_b200"))
    from smcnuts.model.bridgestan import _BUILTIN_DIGESTS, program_digest
    a = "data { int T; } // c\nparameters { real mu; } /* block\n comment */ model { mu ~ normal(0, 1); }"
    assert program_digest(a) == program_digest("data{int T;}\n\nparameters{real mu;}model{mu~normal(0,1);}  # tail")
    assert program_digest(a) != program_digest(a.replace("normal(0, 1)", "normal(0, 2)"))
    assert program_digest((STAN / "arma_series.stan").read_text()) != _BUILTIN_DIGESTS["arma"]
    for name, digest in _BUILTIN_DIGESTS.items():
        if name == "PRMwCD":            # not stored (see test_reference_stan_programs_translate_to_the_oracle_densities)
            continue
        text = (REF_STAN / f"{name}.stan").read_text()
        assert program_digest(text) == digest
        assert program_digest(text.replace("2.5", "3.5").replace("1.3", "1.4")) != digest


_WHILE = """
functions {
  real newton_sqrt(real c) {      // the trip count depends on the value
    real z = c;
    real k = 0;
    while (fabs(z * z - c) > 1e-13 * c && k < 60) { z = 0.5 * (z + c / z); k += 1; }
    return z;
  }
}
data { int N; vector[N] y; }
parameters { real<lower=0> a; real m; }
model {
  real acc = 0;
  real i = 1;
  vector[N] v;
  while (i <= N - 0.5) { acc += i * m; i += 1; }
  target += -0.5 * square(newton_sqrt(1 + a) - 1.2) - 0.01 * acc * acc;
  for (n in 1:N) { v[n] = y[n] - m; while (v[n] > 1) v[n] = v[n] - 1; target += -0.5 * v[n] * v[n]; }
}
"""


def test_while_loops_with_value_dependent_trip_counts(tmp_path):
    """while: a counting loop, a wrap-into-range loop on an array element and a Newton iteration inside an inlined
    function; derivatives flow through however many trips the values take."""
    rng = np.random.default_rng(0)
    data = {"N": 4, "y": (rng.normal(size=4) * 2).tolist()}
    y = np.array(data["y"])

    def restated(u):
        a, m = np.exp(u[0]), u[1]
        acc = sum(i * m for i in (1, 2, 3))                  # i <= N - 0.5
        A = -0.5 * (np.sqrt(1 + a) - 1.2) ** 2 - 0.01 * acc * acc + u[0]
        for n in range(4):
            v = y[n] - m
            while v > 1:
                v -= 1
            A += -0.5 * v * v
        return A
    h = HostModel(SC.generate(_WHILE, data), tmp_path)
    x = rng.normal(size=(20, 2)) * 0.5
    A, B, g = h.split(x, 1.0)
    np.testing.assert_allclose(A, [restated(u) for u in x], rtol=1e-12, atol=1e-12)
    _fd_check(h, x, g, 1.0, 2, tol=2e-5)


def test_print_is_ignored_and_reject_maps_to_minus_infinity(tmp_path):
    """bridgestan.py:47-49 of the reference turns a Stan exception into logp = -inf; reject() does the same here."""
    text = ('parameters { real a; } model { print("a = ", a, " (debug)"); '
            'if (a > 1.5) reject("a too large: ", a); a ~ normal(0, 1); }')
    h = HostModel(SC.generate(text, {}), tmp_path)
    A, B, g = h.split(np.array([[0.3], [2.0]]), 1.0)
    assert A[0] == -0.5 * 0.3 ** 2 and A[1] == -np.inf and g[0, 0] == -0.3


def test_unsupported_constructs_fail_loudly_with_the_line():
    ok = "data { int N; } parameters { real a; } model { a ~ normal(0, 1); }"
    assert SC.generate(ok, {"N": 3}).dim == 1
    for bad, what in [
        ("parameters { real a; } model { a ~ normal(0, 1) T[0, ]; }", "truncation"),
        ("parameters { real a; } model { a ~ wishart(1, 2); }", "wishart"),
        ("parameters { matrix[2, 2] a; } model { }", "matrix"),
        ("functions { vector f(vector x) { return x; } } parameters { real a; } model { }", "returning real"),
        ("functions { real f(real x) { if (x > 0) return x; return -x; } } parameters { real a; } model { target += f(a); }",
         "early returns"),
        ("functions { real f(real x) { return f(x); } } parameters { real a; } model { target += f(a); }", "recursive"),
        ("data { int N; vector[N] v; } parameters { vector[N] a; } model { target += sum(a * v); }", "elementwise products"),
        ("data { int N; matrix[N, N] X; } parameters { vector[N] a; } model { vector[N] m = a; m = X * m; }", "second variable"),
        ("data { int N; } parameters { vector[N] a; } model { vector[2] m; m = a; }", "size"),
        ("data { int N; } parameters { real a; } model { a ~ normal(0, 1); }", "missing from the data"),
        ("data { real phi; } parameters { real a; } model { target += exp(phi * a); }", "phi"),
    ]:
        data = {} if "missing" in what else {"N": 3, "v": [1.0, 2.0, 3.0], "X": [[1.0, 0.0, 0.0]] * 3}
        with pytest.raises(SC.StanSubsetError, match=what):
            SC.generate(bad, data)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_generated_model_runs_the_nuts_and_smc_kernels_like_the_builtin_one():
    from smcnuts.distributions import StdNormal
    from smcnuts.model.bridgestan import StanModel
    from smcnuts.model.device_model import make_model
    from smcnuts.model.generated import GeneratedModel
    from smcnuts.proposal.nuts import NUTSProposal
    from smcnuts.smc_sampler import SMCSampler
    gen = GeneratedModel((STAN / "arma11.stan").read_text(), _arma_data(), "arma11")
    ref = make_model("arma")
    rng = np.random.default_rng(3)
    N = 4096
    x = rng.normal(size=(N, 4)) * 0.05 + np.array([0.0, 0.9, 0.0, -1.7])
    r = rng.normal(size=(N, 4))
    for phi in (0.3, 1.0):
        np.testing.assert_allclose(gen.logpdf(x, phi), ref.logpdf(x, phi), rtol=1e-11)
        np.testing.assert_allclose(gen.logpdfgrad(x, phi), ref.logpdfgrad(x, phi), rtol=1e-9, atol=1e-8)
    kg, kr = NUTSProposal(gen, StdNormal(4), 0.01, rng=10), NUTSProposal(ref, StdNormal(4), 0.01, rng=10)
    xg, _ = kg.rvs(x, r, 1.0)
    xr, _ = kr.rvs(x, r, 1.0)
    same = (kg.last["n_leapfrog"] == kr.last["n_leapfrog"]).cpu().numpy()
    assert same.mean() > 0.99, same.mean()          # same trees up to the rounding of two formulations of one density
    np.testing.assert_allclose(xg[same], xr[same], rtol=1e-6, atol=1e-8)
    assert gen.constrain_kind == ref.constrain_kind
    np.testing.assert_allclose(gen.constrain(x), ref.constrain(x), rtol=1e-15)
    # the diagonal metric goes through the plug-in as well (ScaledModel instantiated in its translation unit)
    sc = np.array([0.5, 2.0, 1.5, 0.7])
    gen.set_metric_scale(sc); ref.set_metric_scale(sc)
    try:
        kg.iteration = kr.iteration = 0
        xg2, _ = kg.rvs(x, r, 1.0)
        xr2, _ = kr.rvs(x, r, 1.0)
        same2 = (kg.last["n_leapfrog"] == kr.last["n_leapfrog"]).cpu().numpy()
        assert same2.mean() > 0.99 and not np.array_equal(xr2, xr)
        np.testing.assert_allclose(xg2[same2], xr2[same2], rtol=1e-6, atol=1e-8)
    finally:
        gen.set_metric_scale(None); ref.set_metric_scale(None)
    # whole SMC run through the reference-facing constructor, model resolved by StanModel(name, model_path, data_path)
    data_path = ROOT / "smc-nuts_b200/smcnuts/data/arma/arma.json"
    sm = StanModel("arma11", str(STAN / "arma11.stan"), str(data_path))
    out = []
    for target in (sm, ref):
        s = SMCSampler(K=6, N=2048, target=target, step_size=0.01, sample_proposal=StdNormal(4), momentum_proposal=StdNormal(4),
                       lkernel="forwardsLKernel", tempering=False, rng=10)
        s.sample(show_progress=False)
        out.append(s)
    np.testing.assert_allclose(out[0].mean_estimate[-1], out[1].mean_estimate[-1], rtol=0.05, atol=0.02)
    assert abs(out[0].leapfrogs.sum() / out[1].leapfrogs.sum() - 1.0) < 0.02


@pytest.mark.gpu
def test_generated_logistic_model_with_bounded_parameters_samples_and_constrains():
    from scipy.special import expit
    from smcnuts.distributions import StdNormal
    from smcnuts.model.generated import GeneratedModel
    from smcnuts.smc_sampler import SMCSampler
    rng = np.random.default_rng(2)
    m = GeneratedModel((STAN / "logistic.stan").read_text(), _logistic_data(rng), "logistic")
    x = rng.normal(size=(64, 6))
    c = m.constrain(x)
    np.testing.assert_allclose(c[:, :4], x[:, :4])
    np.testing.assert_allclose(c[:, 4], np.exp(x[:, 4]), rtol=1e-15)
    np.testing.assert_allclose(c[:, 5], -1.0 + 3.0 * expit(x[:, 5]), rtol=1e-13, atol=1e-15)
    s = SMCSampler(K=8, N=4096, target=m, step_size=0.05, sample_proposal=StdNormal(6), momentum_proposal=StdNormal(6),
                   lkernel="forwardsLKernel", tempering=False, rng=3)
    s.sample(show_progress=False)
    est = s.mean_estimate[-1]
    assert np.all(np.isfinite(est)) and est[4] > 0 and -1 < est[5] < 2 and s.leapfrogs.sum() > 0


@pytest.mark.gpu
def test_generated_container_programs_run_on_the_device_like_their_host_build(tmp_path):
    """The programs with container expressions, if / else and transformed blocks, compiled by nvcc as plug-ins: the device
    log density and gradient equal the g++ build of the same generated text, and a tempered SMC run on the regression
    program recovers the coefficients the data were generated from."""
    from smcnuts.distributions import StdNormal
    from smcnuts.model.generated import GeneratedModel
    from smcnuts.smc_sampler import SMCSampler
    rng = np.random.default_rng(11)
    data = _containers_data(rng, 1)
    m = GeneratedModel((STAN / "containers.stan").read_text(), data, "containers")
    h = HostModel(m.source, tmp_path)
    x = rng.normal(size=(512, 6)) * 0.7
    for phi in (0.0, 0.35, 1.0):
        A, B, g = h.split(x, phi)
        np.testing.assert_allclose(m.logpdf(x, phi), A + phi * B, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(m.logpdfgrad(x, phi), g, rtol=1e-10, atol=1e-10)
    # regression: y = 0.7 + X (1, -0.5, 0.25) + 0.3 noise, 60 observations
    N, K = 60, 3
    X = rng.normal(size=(N, K))
    truth = np.array([0.7, 1.0, -0.5, 0.25])
    y = truth[0] + X @ truth[1:] + 0.3 * rng.normal(size=N)
    reg = GeneratedModel((STAN / "regression.stan").read_text(), {"N": N, "K": K, "X": X.tolist(), "y": y.tolist()}, "regression")
    s = SMCSampler(K=40, N=4096, target=reg, step_size=0.03, sample_proposal=StdNormal(5), momentum_proposal=StdNormal(5),
                   lkernel="asymptoticLKernel", tempering=True, rng=5)
    s.sample(show_progress=False)
    assert s.phi[-1] == 1.0
    est = s.mean_estimate[-1]
    # the random-walk and N(0, 1) priors shrink a little; posterior sd of a coefficient is ~0.3 / sqrt(60) = 0.04
    np.testing.assert_allclose(est[:4], truth, atol=0.15)
    assert 0.2 < est[4] < 0.45


@pytest.mark.gpu
def test_stanmodel_with_a_rephrased_arma_file_goes_through_the_generator_and_agrees_with_the_builtin():
    from smcnuts.model.bridgestan import StanModel
    data_path = ROOT / "smc-nuts_b200/smcnuts/data/arma/arma.json"
    edited = StanModel("arma", str(STAN / "arma_series.stan"), str(data_path))     # same name, another program text
    builtin = StanModel("arma", "no_such_file.stan", str(data_path))
    assert edited.resolved == "generated" and builtin.resolved == "builtin"
    x = np.random.default_rng(3).normal(size=(256, 4)) * 0.05 + np.array([0.0, 0.9, 0.0, -1.7])
    for phi in (0.25, 1.0):
        np.testing.assert_allclose(edited.logpdf(x, phi), builtin.logpdf(x, phi), rtol=1e-11)
        np.testing.assert_allclose(edited.logpdfgrad(x, phi), builtin.logpdfgrad(x, phi), rtol=1e-9, atol=1e-8)
    np.testing.assert_allclose(edited.constrain(x), builtin.constrain(x), rtol=1e-15)
