"""simplex / ordered / positive_ordered parameters of the Stan subset, the densities they are for (dirichlet, categorical,
multinomial, log_sum_exp of a vector) and the constrained output of generated models (`constrain()` with
constrained_dim columns, estimates on the constrained scale).

CPU: the generated struct is compiled with g++ (the text nvcc compiles for the device) and checked against a torch
autograd restatement of the transforms and densities, a numerically formed Jacobian, numpy inverse transforms and
scipy.  GPU: the plug-in against the host build, constrain() into a guarded buffer, and SMC runs against exact posterior
moments (Dirichlet-multinomial) and a numerical quadrature (two-component mixture)."""
import ctypes
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from tests.test_stan_codegen import SC, CSRC, STAN, _containers_data, _logistic_data

EPS = np.finfo(np.float64).eps
HARNESS = r'''
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
extern "C" int gen_cdim() { return GenModel::CDIM; }
extern "C" void gen_constrain(const double* x, long N, double* out) {
    for (long i = 0; i < N; ++i) {
        double xv[GenModel::DMAX];
        for (int k = 0; k < GenModel::DMAX; ++k) xv[k] = x[i * GenModel::DMAX + k];
        GenModel::constrain(xv, out + i * GenModel::CDIM);
    }
}
'''


class Host:
    """A generated model built with g++: split density, gradient and constrain()."""

    def __init__(self, src, tmp_path):
        tmp_path.mkdir(parents=True, exist_ok=True)
        (tmp_path / "model_gen.h").write_text(src.text)
        (tmp_path / "host.cpp").write_text(HARNESS)
        so = tmp_path / "libgen.so"
        subprocess.run(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-std=c++17", f"-I{CSRC}", f"-I{tmp_path}",
                        str(tmp_path / "host.cpp"), "-o", str(so)], check=True, capture_output=True)
        self.lib = ctypes.CDLL(str(so))
        self.blob = np.array(src.blob if src.blob else [0.0])
        self.dim, self.cdim = src.dim, self.lib.gen_cdim()
        assert self.cdim == src.cdim

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(ctypes.c_void_p)

    def split(self, x, phi=1.0):
        x = np.ascontiguousarray(x, dtype=np.float64)
        n = len(x)
        A, B, g = np.empty(n), np.empty(n), np.empty((n, self.dim))
        self.lib.gen_logp(self._p(x), ctypes.c_long(n), ctypes.c_double(phi), self._p(self.blob), self._p(A), self._p(B),
                          self._p(g))
        return A, B, g

    def constrain(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.empty((len(x), self.cdim))
        self.lib.gen_constrain(self._p(x), ctypes.c_long(len(x)), self._p(out))
        return out


# ------------------------------------------------------------------------------------------------ torch restatements
def t_simplex(y):
    """stick-breaking (Stan <= 2.35), y [n, K-1] -> (x [n, K], log J [n])"""
    K = y.shape[1] + 1
    r = torch.ones_like(y[:, 0])
    log_r = torch.zeros_like(r)
    xs, lj = [], torch.zeros_like(r)
    for k in range(K - 1):
        u = y[:, k] - np.log(K - 1 - k)
        xs.append(r * torch.sigmoid(u))
        lj = lj + torch.nn.functional.logsigmoid(u) + torch.nn.functional.logsigmoid(-u) + log_r
        r = r * torch.sigmoid(-u)
        log_r = log_r + torch.nn.functional.logsigmoid(-u)
    return torch.stack(xs + [r], 1), lj


def t_ordered(y, positive):
    first = torch.exp(y[:, :1]) if positive else y[:, :1]
    x = torch.cumsum(torch.cat([first, torch.exp(y[:, 1:])], 1), 1)
    return x, y[:, 1:].sum(1) + (y[:, 0] if positive else 0.0)


def t_constrain(kind, y):
    return t_simplex(y) if kind == "simplex" else t_ordered(y, kind == "positive_ordered")


def n_unc(kind, K):
    return K - 1 if kind == "simplex" else K


def draw(rng, n, d):
    """mostly moderate coordinates, every row has one coordinate at +-30 and some rows are all large"""
    y = rng.normal(size=(n, d)) * 1.5
    y[np.arange(n), rng.integers(0, d, n)] = rng.choice([-30.0, 30.0], n) * rng.uniform(0.8, 1.0, n)
    y[: n // 8] = rng.uniform(-30, 30, size=(n // 8, d))
    return y


# ------------------------------------------------------------------------------------------------ CPU: the transforms
KINDS = ("simplex", "ordered", "positive_ordered")


def _plain_program(K):
    return f"""
data {{ vector[{K}] m; vector[{K}] w; real phi; }}
parameters {{ simplex[{K}] s; ordered[{K}] o; positive_ordered[{K}] p; }}
model {{
  target += normal_lpdf(s | m, 1.5) + normal_lpdf(log(p) | m, 2);
  o ~ normal(m, 3);
  target += phi * (dot_product(w, s) + dot_product(w, o) - dot_product(w, p));
}}"""


def _array_program(kind, K):
    return f"""
data {{ vector[{K}] m; array[3] vector[{K}] w; real phi; }}
parameters {{ array[3] {kind}[{K}] v; }}
model {{
  for (j in 1:3) {{
    target += normal_lpdf(v[j] | m, 1.5 + j);
    target += phi * dot_product(w[j], v[j]);
  }}
}}"""


def _reference_plain(y, K, m, w, phi):
    """A, B, grad of _plain_program by torch autograd"""
    yt = torch.tensor(y, dtype=torch.float64, requires_grad=True)
    nu = K - 1
    s, ls = t_simplex(yt[:, :nu])
    o, lo = t_ordered(yt[:, nu:nu + K], False)
    p, lp = t_ordered(yt[:, nu + K:], True)
    mt, wt = torch.tensor(m), torch.tensor(w)

    def normal(x, mu, sd, const=True):
        return (-0.5 * ((x - mu) / sd) ** 2 - ((np.log(sd) + 0.5 * np.log(2 * np.pi)) if const else 0.0)).sum(1)
    A = ls + lo + lp + normal(s, mt, 1.5) + normal(torch.log(p), mt, 2.0) + normal(o, mt, 3.0, const=False)
    B = (s * wt).sum(1) + (o * wt).sum(1) - (p * wt).sum(1)
    (g,) = torch.autograd.grad((A + phi * B).sum(), yt)
    return A.detach().numpy(), B.detach().numpy(), g.numpy()


def _reference_array(y, kind, K, m, w, phi):
    yt = torch.tensor(y, dtype=torch.float64, requires_grad=True)
    nu = n_unc(kind, K)
    mt = torch.tensor(m)
    A = B = 0.0
    for j in range(3):
        x, lj = t_constrain(kind, yt[:, j * nu:(j + 1) * nu])
        sd = 1.5 + j + 1
        A = A + lj + (-0.5 * ((x - mt) / sd) ** 2 - np.log(sd) - 0.5 * np.log(2 * np.pi)).sum(1)
        B = B + (x * torch.tensor(w[j])).sum(1)
    (g,) = torch.autograd.grad((A + phi * B).sum(), yt)
    return A.detach().numpy(), B.detach().numpy(), g.numpy()


def _close(got, ref, rtol, what):
    scale = np.maximum(np.abs(ref), 1.0)
    err = np.max(np.abs(got - ref) / scale)
    assert err <= rtol, f"{what}: max relative error {err:.3g} > {rtol}"


@pytest.mark.parametrize("K", [2, 3, 7, 16])
def test_vector_parameter_types_match_an_autograd_restatement(tmp_path, K):
    rng = np.random.default_rng(K)
    m, w = rng.normal(size=K), rng.normal(size=K)
    src = SC.generate(_plain_program(K), {"m": m.tolist(), "w": w.tolist()})
    assert src.dim == 3 * K - 1 and src.cdim == 3 * K
    assert src.param_names == [f"{n}.{i}" for n in "sop" for i in range(1, K + 1)]
    assert src.param_unc_names == ([f"s.{i}" for i in range(1, K)] + [f"{n}.{i}" for n in "op" for i in range(1, K + 1)])
    h = Host(src, tmp_path / "plain")
    y = draw(rng, 400, src.dim)
    y[:, K - 1:] = np.clip(y[:, K - 1:], -30, 5)   # ordered values of exp(30) squared in a normal density lose all digits
    for phi in (0.0, 0.45, 1.0):
        A, B, g = h.split(y, phi)
        Ar, Br, gr = _reference_plain(y, K, m, w, phi)
        _close(A, Ar, 1e-12, "A")
        _close(B, Br, 1e-12, "B")
        _close(g, gr, 1e-9, "gradient")
    for kind in KINDS:
        wa = rng.normal(size=(3, K))
        src = SC.generate(_array_program(kind, K), {"m": m.tolist(), "w": wa.tolist()})
        nu = n_unc(kind, K)
        assert src.dim == 3 * nu and src.cdim == 3 * K and src.param_names[K] == "v.2.1"
        assert src.param_unc_names[nu] == "v.2.1" and src.param_unc_names[-1] == f"v.3.{nu}"
        h = Host(src, tmp_path / kind)
        y = draw(rng, 300, src.dim)
        if kind != "simplex":
            y = np.clip(y, -30, 5)
        A, B, g = h.split(y, 0.7)
        Ar, Br, gr = _reference_array(y, kind, K, m, wa, 0.7)
        _close(A, Ar, 1e-12, f"{kind} A")
        _close(B, Br, 1e-12, f"{kind} B")
        _close(g, gr, 1e-9, f"{kind} gradient")


def _inverse(kind, x):
    """numpy inverse transforms: constrained rows [n, K] -> y [n, K or K - 1]"""
    K = x.shape[1]
    if kind == "simplex":
        r = np.cumsum(x[:, ::-1], 1)[:, ::-1]          # r_k = sum_{j >= k} x_j: the remaining stick, no cancellation
        return np.log(x[:, :-1]) - np.log(r[:, 1:]) + np.log(K - 1 - np.arange(K - 1))
    d = np.diff(x, axis=1)
    first = np.log(x[:, :1]) if kind == "positive_ordered" else x[:, :1]
    return np.concatenate([first, np.log(d)], 1)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("K", [2, 3, 7, 16])
def test_log_jacobian_and_constrained_rows(tmp_path, kind, K):
    src = SC.generate(f"parameters {{ {kind}[{K}] v; }} model {{ }}", {})
    h = Host(src, tmp_path)
    nu = src.dim
    rng = np.random.default_rng(100 + K)
    # log J against log |det| of the Jacobian of y -> (x_1 .. x_{K-1}) (simplex) or y -> x, by central differences
    y = rng.normal(size=(40, nu)) * 1.2
    A, _, _ = h.split(y)
    hstep = 1e-5
    for i in range(len(y)):
        J = np.empty((nu, nu))
        for j in range(nu):
            e = np.zeros(nu)
            e[j] = hstep
            J[:, j] = (h.constrain((y[i] + e)[None])[0, :nu] - h.constrain((y[i] - e)[None])[0, :nu]) / (2 * hstep)
        assert abs(A[i] - np.linalg.slogdet(J)[1]) <= 1e-8 * max(1.0, abs(A[i])), (i, A[i], np.linalg.slogdet(J)[1])
    # constrained rows, including coordinates at |y| = 30
    y = draw(rng, 2000, nu)
    x = h.constrain(y)
    assert x.shape == (2000, K) and np.all(np.isfinite(x))
    xr, _ = t_constrain(kind, torch.tensor(y))
    # a cumulative sum that crosses zero has only absolute accuracy, relative to the largest partial sum of the row
    assert np.all(np.abs(x - xr.numpy()) <= 1e-13 * np.maximum(np.abs(x), np.abs(x).max(1, keepdims=True) * (kind != "simplex")))
    if kind == "simplex":
        assert np.all(x >= 0.0)
        assert np.max(np.abs(x.sum(1) - 1.0)) <= 4 * EPS, np.max(np.abs(x.sum(1) - 1.0)) / EPS
        keep = np.all(x > 1e-300, 1)
        np.testing.assert_allclose(_inverse(kind, x[keep]), y[keep], rtol=1e-9, atol=1e-9)
    else:
        d = np.diff(x, axis=1)
        assert np.all(d >= 0.0)
        # strictly increasing wherever exp(y_k) is representable next to x_{k-1} (ulp of x_{k-1} below it)
        visible = np.exp(y[:, 1:]) > 2 * np.spacing(np.abs(x[:, :-1]))
        assert np.all(d[visible] > 0.0)
        if kind == "positive_ordered":
            assert np.all(x[:, 0] > 0.0)
        moderate = np.all(np.abs(y) < 8, 1)
        np.testing.assert_allclose(_inverse(kind, x[moderate]), y[moderate], rtol=1e-8, atol=1e-8)


# ------------------------------------------------------------------------------------------------ CPU: the densities
def _fd_grad(h, y, phi, step=1e-6):
    g = np.empty_like(y)
    for j in range(y.shape[1]):
        e = np.zeros(y.shape[1])
        e[j] = step
        Ap, Bp, _ = h.split(y + e, phi)
        Am, Bm, _ = h.split(y - e, phi)
        g[:, j] = ((Ap + phi * Bp) - (Am + phi * Bm)) / (2 * step)
    return g


def _simplex_np(y):
    x, lj = t_simplex(torch.tensor(y))
    return x.numpy(), lj.numpy()


def _mixture_data(rng, K, N):
    mus = np.linspace(-3, 3, K)
    return {"K": K, "N": N, "y": (rng.choice(mus, N) + rng.normal(size=N)).tolist()}


def test_mixture_program_matches_numpy_and_finite_differences(tmp_path):
    from scipy.special import logsumexp
    from scipy.stats import norm
    rng = np.random.default_rng(5)
    K, N = 3, 40
    data = _mixture_data(rng, K, N)
    src = SC.generate((STAN / "mixture.stan").read_text(), data)
    assert src.dim == 2 * K - 1 and src.cdim == 2 * K
    h = Host(src, tmp_path)
    y = rng.normal(size=(50, src.dim))
    yd = np.asarray(data["y"])
    for phi in (0.3, 1.0):
        A, B, g = h.split(y, phi)
        theta, lj_s = _simplex_np(y[:, :K - 1])
        mu = np.cumsum(np.concatenate([y[:, K - 1:K], np.exp(y[:, K:])], 1), 1)
        lj_o = y[:, K:].sum(1)
        Ar = lj_s + lj_o + (-0.5 * (mu / 10) ** 2).sum(1)          # `~`: the constants of normal(0, 10) are dropped
        lps = np.log(theta)[:, None, :] + norm.logpdf(yd[None, :, None], mu[:, None, :], 1.0)
        Br = logsumexp(lps, axis=2).sum(1)
        np.testing.assert_allclose(A, Ar, rtol=1e-12)
        np.testing.assert_allclose(B, Br, rtol=1e-12)
        np.testing.assert_allclose(g, _fd_grad(h, y, phi), rtol=1e-6, atol=1e-5)


def test_dirichlet_multinomial_and_categorical_match_scipy(tmp_path):
    from scipy.stats import dirichlet, multinomial
    rng = np.random.default_rng(6)
    K = 5
    alpha = np.array([1.0, 2.5, 0.7, 3.0, 1.0])
    counts = np.array([3, 0, 7, 2, 11])
    data = {"K": K, "alpha": alpha.tolist(), "counts": counts.tolist()}
    src = SC.generate((STAN / "dirichlet_multinomial.stan").read_text(), data)
    h = Host(src, tmp_path / "dm")
    y = rng.normal(size=(60, K - 1)) * 1.5
    theta, lj = _simplex_np(y)
    for phi in (0.0, 0.6, 1.0):
        A, B, g = h.split(y, phi)
        # `theta ~ dirichlet(alpha)` with data alpha keeps sum (alpha_k - 1) log theta_k only
        norm_const = dirichlet.logpdf(np.full(K, 1.0 / K), alpha) - ((alpha - 1) * np.log(1.0 / K)).sum()
        Ar = lj + np.array([dirichlet.logpdf(t, alpha) for t in theta]) - norm_const
        Br = np.array([multinomial.logpmf(counts, counts.sum(), t) for t in theta])
        np.testing.assert_allclose(A, Ar, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(B, Br, rtol=1e-12)
        np.testing.assert_allclose(g, _fd_grad(h, y, phi), rtol=1e-6, atol=1e-6)
    # target += keeps every constant; a parameter alpha (digamma series); categorical over an int array and an int
    prog = """
data { int K; array[6] int z; int z1; }
parameters { simplex[K] th; vector<lower=0>[K] a; }
model {
  target += dirichlet_lpdf(th | a);
  a ~ exponential(1);
  target += categorical_lpmf(z | th) + categorical_lpmf(z1 | th);
}"""
    z = [1, 3, 3, 2, 3, 1]
    src = SC.generate(prog, {"K": 3, "z": z, "z1": 2})
    h = Host(src, tmp_path / "cat")
    y = rng.normal(size=(40, 5)) * 0.8
    A, B, g = h.split(y)
    th, lj = _simplex_np(y[:, :2])
    a = np.exp(y[:, 2:])
    Ar = (lj + y[:, 2:].sum(1) + np.array([dirichlet.logpdf(t, aa) for t, aa in zip(th, a)]) - a.sum(1)
          + np.log(th[:, [zz - 1 for zz in z + [2]]]).sum(1))
    np.testing.assert_allclose(A + B, Ar, rtol=1e-11)
    np.testing.assert_allclose(g, _fd_grad(h, y, 1.0), rtol=1e-6, atol=1e-6)


def test_log_sum_exp_of_a_vector_and_vector_types_in_transformed_parameters(tmp_path):
    from scipy.special import logsumexp, softmax
    prog = """
data { int K; }
parameters { vector[K] v; }
transformed parameters { simplex[K] w = exp(v - log_sum_exp(v)); }
model { target += log_sum_exp(v) + 0.5 * w[1]; }"""
    src = SC.generate(prog, {"K": 4})
    assert src.dim == 4 and src.cdim == 4          # a transformed parameter is a plain vector: no transform, no output
    h = Host(src, tmp_path)
    v = np.random.default_rng(7).normal(size=(30, 4)) * 20
    A, B, g = h.split(v)
    w = softmax(v, axis=1)
    np.testing.assert_allclose(A + B, logsumexp(v, axis=1) + 0.5 * w[:, 0], rtol=1e-13)
    e0 = np.zeros_like(w)
    e0[:, 0] = 1.0
    np.testing.assert_allclose(g, w + 0.5 * w[:, :1] * (e0 - w), rtol=1e-10, atol=1e-12)


def test_overflow_makes_the_density_minus_infinity(tmp_path):
    src = SC.generate("parameters { positive_ordered[3] p; } model { p ~ normal(0, 1); }", {})
    h = Host(src, tmp_path)
    A, _, _ = h.split(np.array([[0.0, 800.0, 0.0], [0.0, 1.0, 2.0]]))
    assert A[0] == -np.inf and np.isfinite(A[1])


def test_scalar_programs_keep_one_value_per_coordinate():
    for name, data in (("logistic", _logistic_data(np.random.default_rng(2))),
                       ("containers", _containers_data(np.random.default_rng(11), 1))):
        src = SC.generate((STAN / f"{name}.stan").read_text(), data)
        assert src.cdim == src.dim and src.param_unc_names == src.param_names
        assert "gc[" not in src.text                  # the gradient leaves eval() as before: no pullback


def test_constrained_types_outside_the_subset_fail_loudly_with_the_line():
    for bad, what in [
        ("parameters {\n simplex<lower=0>[3] s; } model { }", "line 2: bounds on a simplex"),
        ("parameters {\n real a;\n unit_vector[3] u; } model { }", "line 3: type 'unit_vector'"),
        ("parameters {\n cholesky_factor_corr[3] L; } model { }", "line 2: type 'cholesky_factor_corr'"),
        ("parameters {\n sum_to_zero_vector[3] z; } model { }", "line 2: type 'sum_to_zero_vector'"),
        ("parameters {\n cov_matrix[3] S; } model { }", "line 2: type 'cov_matrix'"),
        ("data {\n int K;\n simplex[K] p; } parameters { real a; } model { }", "line 3: data 'p' is not a valid simplex"),
        ("data {\n int K;\n array[2] ordered[K] c; } parameters { real a; } model { }", "line 3: data 'c' is not a valid ordered"),
        ("parameters {\n simplex[1] s; } model { }", "line 2: a simplex needs at least 2"),
    ]:
        data = {"K": 3, "p": [0.2, 0.3, 0.6], "c": [[1.0, 2.0, 3.0], [1.0, 1.0, 2.0]]}
        with pytest.raises(SC.StanSubsetError, match=what):
            SC.generate(bad, data)
    ok = "data { int K; simplex[K] p; array[2] ordered[K] c; positive_ordered[K] q; } parameters { real a; } model { }"
    SC.generate(ok, {"K": 3, "p": [0.2, 0.3, 0.5], "c": [[1.0, 2.0, 3.0], [-1.0, 0.0, 2.0]], "q": [0.1, 1.0, 2.0]})


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_plugin_matches_the_host_build_and_constrains_into_a_guarded_buffer(tmp_path):
    from smcnuts import _cabi, _device as dev
    from smcnuts.model.generated import GeneratedModel
    from tests.test_gpu_dispatch import guarded
    rng = np.random.default_rng(21)
    for K in (3, 16):
        m = GeneratedModel(_plain_program(K), {"m": rng.normal(size=K).tolist(), "w": rng.normal(size=K).tolist()},
                           f"plain{K}")
        h = Host(m.source, tmp_path / f"p{K}")
        assert m.constrained_dim == 3 * K and m.dim == 3 * K - 1 and m.constrain_kind == _cabi.CONSTRAIN_MODEL
        y = draw(rng, 4096, m.dim)
        y[:, K - 1:] = np.clip(y[:, K - 1:], -30, 5)
        for phi in (0.2, 1.0):
            A, B, g = h.split(y, phi)
            ref = A + phi * B
            np.testing.assert_allclose(m.logpdf(y, phi), ref, rtol=1e-12, atol=1e-12 * np.abs(ref).max())
            gd = m.logpdfgrad(y, phi)
            assert np.max(np.abs(gd - g) / np.maximum(np.abs(g), 1.0)) <= 1e-9
        n = 1 << 20
        yb = draw(rng, n, m.dim)
        out, check = guarded(n * m.constrained_dim)
        _cabi.call("smcb_model_constrain", m.handle if hasattr(m, "handle") else m._h, dev.ptr(dev.to_device(yb)), n,
                   dev.ptr(out), dev.stream_ptr())
        check()
        got = out.view(n, m.constrained_dim).cpu().numpy()
        ref = h.constrain(yb)
        # to rounding: the device exp / log and glibc's may differ in the last bit; a simplex value carries that through
        # up to K stick factors, an ordered value only has absolute accuracy against its largest partial sum
        scale = np.abs(ref)
        for j in (1, 2):
            scale[:, j * K:(j + 1) * K] = np.abs(ref[:, j * K:(j + 1) * K]).max(1, keepdims=True)
        assert np.all(np.abs(got - ref) <= 4 * K * EPS * scale)
        assert torch.equal(m.constrain(torch.tensor(yb[:100], device="cuda")).cpu(), torch.tensor(got[:100]))
        np.testing.assert_array_equal(m.constrain(yb[:7].reshape(7, m.dim)), got[:7])


@pytest.mark.gpu
def test_existing_generated_fixtures_constrain_through_the_plugin():
    from scipy.special import expit
    from smcnuts import _cabi
    from smcnuts.model.generated import GeneratedModel
    rng = np.random.default_rng(2)
    m = GeneratedModel((STAN / "logistic.stan").read_text(), _logistic_data(rng), "logistic")
    assert m.constrain_kind == _cabi.CONSTRAIN_MODEL
    x = rng.normal(size=(64, 6)) * 3
    c = m.constrain(x)
    np.testing.assert_array_equal(c[:, :4], x[:, :4])
    np.testing.assert_allclose(c[:, 4], np.exp(x[:, 4]), rtol=1e-15)
    np.testing.assert_allclose(c[:, 5], -1.0 + 3.0 * expit(x[:, 5]), rtol=1e-13, atol=1e-15)
    mixed_data = {"N": 5, "t": rng.normal(size=5).tolist(), "y": rng.uniform(0.5, 2, 5).tolist(), "k": [1, 0, 3, 2, 1]}
    m = GeneratedModel((STAN / "mixed.stan").read_text(), mixed_data, "mixed")
    x = rng.normal(size=(64, 6)) * 3
    c = m.constrain(x)
    np.testing.assert_allclose(c[:, 0], np.exp(x[:, 0]), rtol=1e-15)
    np.testing.assert_allclose(c[:, 1], 3.0 - np.exp(x[:, 1]), rtol=1e-14, atol=1e-14)
    np.testing.assert_allclose(c[:, 2], expit(x[:, 2]), rtol=1e-13, atol=1e-16)
    np.testing.assert_array_equal(c[:, 3], x[:, 3])
    np.testing.assert_allclose(c[:, 4:], 0.5 + np.exp(x[:, 4:]), rtol=1e-15)
    m = GeneratedModel((STAN / "containers.stan").read_text(), _containers_data(rng, 1), "containers")
    x = rng.normal(size=(64, m.dim))
    c = m.constrain(x)
    assert c.shape == (64, m.dim)
    kinds = [t[0] for t in m.source.transforms]
    for j, (kind, lo, hi) in enumerate(m.source.transforms):
        ref = {"none": x[:, j], "lower": (lo or 0.0) + np.exp(x[:, j]), "upper": (hi or 0.0) - np.exp(x[:, j])}.get(kind)
        if ref is None:
            ref = lo + (hi - lo) * expit(x[:, j])
        np.testing.assert_allclose(c[:, j], ref, rtol=1e-13, atol=1e-15, err_msg=str(kinds))


def _sampler(target, K, N, lkernel, seed, step):
    from smcnuts.distributions import StdNormal
    from smcnuts.smc_sampler import SMCSampler
    return SMCSampler(K=K, N=N, target=target, step_size=step, sample_proposal=StdNormal(target.dim),
                      momentum_proposal=StdNormal(target.dim), lkernel=lkernel, tempering=True, rng=seed)


@pytest.mark.gpu
def test_dirichlet_multinomial_posterior_moments():
    from smcnuts.model.generated import GeneratedModel
    K = 5
    alpha = np.array([1.0, 2.0, 0.5, 3.0, 1.5])
    counts = np.array([12, 3, 0, 25, 8])
    m = GeneratedModel((STAN / "dirichlet_multinomial.stan").read_text(),
                       {"K": K, "alpha": alpha.tolist(), "counts": counts.tolist()}, "dm")
    s = _sampler(m, 30, 1 << 16, "forwardsLKernel", 4, 0.2)
    s.sample(show_progress=False)
    assert s.phi[-1] == 1.0
    mean, var = s.mean_estimate[-1], s.variance_estimate[-1]
    assert mean.shape == (K,) and s.variance_estimate.shape == (31, K)
    assert abs(mean.sum() - 1.0) <= 1e-12
    a = alpha + counts
    a0 = a.sum()
    exact_mean, exact_var = a / a0, a * (a0 - a) / (a0 ** 2 * (a0 + 1))
    ess = s.ess[-1]
    se = np.sqrt(var / ess)
    assert np.all(np.abs(mean - exact_mean) <= 4 * se), (mean, exact_mean, se)
    np.testing.assert_allclose(var, exact_var, rtol=0.25)


def _mixture_quadrature(y):
    """posterior means of (w1, w2, mu1, mu2) of tests/stan/mixture.stan with K = 2 by quadrature over (w1, mu1 < mu2)"""
    from scipy.special import logsumexp
    w = np.linspace(0.0005, 0.9995, 400)
    mu = np.linspace(-6, 6, 241)
    M1, M2 = np.meshgrid(mu, mu, indexing="ij")
    keep = M1 < M2
    m1, m2 = M1[keep], M2[keep]
    ll1 = -0.5 * (y[None, :] - m1[:, None]) ** 2
    ll2 = -0.5 * (y[None, :] - m2[:, None]) ** 2
    lw = np.empty((len(w), len(m1)))
    for i, wi in enumerate(w):                       # flat prior on the simplex, normal(0, 10) on mu
        lw[i] = np.logaddexp(np.log(wi) + ll1, np.log1p(-wi) + ll2).sum(1) - 0.5 * (m1 ** 2 + m2 ** 2) / 100
    p = np.exp(lw - lw.max())
    p /= p.sum()
    Wg = w[:, None]
    return np.array([(p * Wg).sum(), (p * (1 - Wg)).sum(), (p * m1).sum(), (p * m2).sum()])


@pytest.mark.gpu
def test_two_component_mixture_matches_quadrature():
    from smcnuts.model.generated import GeneratedModel
    rng = np.random.default_rng(8)
    n = 200
    y = np.where(rng.uniform(size=n) < 0.35, -1.5, 1.5) + rng.normal(size=n)
    m = GeneratedModel((STAN / "mixture.stan").read_text(), {"K": 2, "N": n, "y": y.tolist()}, "mix2")
    s = _sampler(m, 40, 1 << 16, "forwardsLKernel", 9, 0.1)
    s.sample(show_progress=False)
    assert s.phi[-1] == 1.0
    mean, var = s.mean_estimate[-1], s.variance_estimate[-1]
    exact = _mixture_quadrature(y)
    se = np.sqrt(var / s.ess[-1])
    assert np.all(np.abs(mean - exact) <= 4 * se), (mean, exact, se)


@pytest.mark.gpu
def test_asymptotic_lkernel_estimates_have_the_constrained_width():
    from smcnuts.model.generated import GeneratedModel
    K = 4
    m = GeneratedModel((STAN / "dirichlet_multinomial.stan").read_text(),
                       {"K": K, "alpha": [1.0] * K, "counts": [5, 1, 9, 3]}, "dm4")
    s = _sampler(m, 8, 4096, "asymptoticLKernel", 3, 0.2)
    s.sample(show_progress=False)
    assert s.mean_estimate.shape == (9, K) and s.variance_estimate.shape == (9, K)
    assert np.all(np.isfinite(s.mean_estimate[-1])) and abs(s.mean_estimate[-1].sum() - 1.0) < 1e-9
