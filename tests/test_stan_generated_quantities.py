"""Generated quantities of generated Stan models and the `_rng` functions of csrc/stan_rng.cuh.

CPU: the generated gq struct and the _rng functions are compiled with g++ (the text nvcc compiles for the device) and
checked against numpy / scipy restatements, KS and chi-square tests against scipy's distributions, batching and row-order
invariance, refusals and the deferred error of a block outside the subset; the generated density text is pinned to the
digests it had before generated quantities existed.  GPU: the plug-in against the host build into a guarded buffer, and
SMCSampler(generated_quantities=True) against closed-form posterior predictives."""
import ctypes
import hashlib
import json
import subprocess

import numpy as np
import pytest
from scipy import stats

from tests.test_stan_codegen import (SC, CSRC, STAN, ROOT, _arma_data, _containers_data, _logistic_data,
                                     _regression_data)

HARNESS = r'''
#include <cstring>
#include "common.cuh"
#include "models.cuh"
#include "model_gen.h"
#include "model_gq.h"
extern "C" int gen_gq_dim() { return GenModelGQ::GDIM; }
extern "C" void gen_gq(const double* x, long N, unsigned long long seed, unsigned counter, long long particle0,
                       const double* blob, double* out) {
    smcb::ModelDesc d{}; d.data = blob; d.dim = GenModelGQ::DMAX;
    GenModelGQ q(d);
    for (long i = 0; i < N; ++i) {
        double xv[GenModelGQ::DMAX];
        for (int k = 0; k < GenModelGQ::DMAX; ++k) xv[k] = x[i * GenModelGQ::DMAX + k];
        smcb::stan::Rng rng(seed, counter, (unsigned long long)(particle0 + i));
        q.generated_quantities(xv, rng, out + i * GenModelGQ::GDIM);
    }
}
'''

RNG_HARNESS = r'''
#include <cstring>
#include "stan_rng.cuh"
using namespace smcb::stan;
// draw i of `name` with arguments a[0..] from the stream of particle i
extern "C" int rng_draws(const char* name, const double* a, long n, unsigned long long seed, double* out) {
    for (long i = 0; i < n; ++i) {
        Rng g(seed, 0, (unsigned long long)i);
        double v;
        if (!strcmp(name, "normal")) v = normal_rng(a[0], a[1], g);
        else if (!strcmp(name, "std_normal")) v = std_normal_rng(g);
        else if (!strcmp(name, "student_t")) v = student_t_rng(a[0], a[1], a[2], g);
        else if (!strcmp(name, "cauchy")) v = cauchy_rng(a[0], a[1], g);
        else if (!strcmp(name, "double_exponential")) v = double_exponential_rng(a[0], a[1], g);
        else if (!strcmp(name, "logistic")) v = logistic_rng(a[0], a[1], g);
        else if (!strcmp(name, "lognormal")) v = lognormal_rng(a[0], a[1], g);
        else if (!strcmp(name, "exponential")) v = exponential_rng(a[0], g);
        else if (!strcmp(name, "gamma")) v = gamma_rng(a[0], a[1], g);
        else if (!strcmp(name, "inv_gamma")) v = inv_gamma_rng(a[0], a[1], g);
        else if (!strcmp(name, "beta")) v = beta_rng(a[0], a[1], g);
        else if (!strcmp(name, "uniform")) v = uniform_rng(a[0], a[1], g);
        else if (!strcmp(name, "bernoulli")) v = bernoulli_rng(a[0], g);
        else if (!strcmp(name, "bernoulli_logit")) v = bernoulli_logit_rng(a[0], g);
        else if (!strcmp(name, "binomial")) v = binomial_rng(a[0], a[1], g);
        else if (!strcmp(name, "poisson")) v = poisson_rng(a[0], g);
        else if (!strcmp(name, "poisson_log")) v = poisson_log_rng(a[0], g);
        else if (!strcmp(name, "neg_binomial_2")) v = neg_binomial_2_rng(a[0], a[1], g);
        else if (!strcmp(name, "categorical")) v = categorical_rng<4>(a, g);
        else return -1;
        out[i] = g.ok ? v : NAN;
    }
    return 0;
}
'''


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _compile(tmp_path, files, main):
    tmp_path.mkdir(parents=True, exist_ok=True)
    for name, text in files.items():
        (tmp_path / name).write_text(text)
    so = tmp_path / "lib.so"
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-std=c++17", f"-I{CSRC}", f"-I{tmp_path}",
                    str(tmp_path / main), "-o", str(so)], check=True, capture_output=True)
    return ctypes.CDLL(str(so))


class HostGQ:
    """The density struct and the generated-quantities struct of a program, built with g++."""

    def __init__(self, src, tmp_path):
        self.lib = _compile(tmp_path, {"model_gen.h": src.text, "model_gq.h": src.gq_text, "host.cpp": HARNESS}, "host.cpp")
        self.lib.gen_gq.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_ulonglong, ctypes.c_uint, ctypes.c_longlong,
                                    ctypes.c_void_p, ctypes.c_void_p]
        self.blob = np.array(src.blob if src.blob else [0.0])
        self.dim, self.G = src.dim, self.lib.gen_gq_dim()
        assert self.G == src.gq_dim

    def gq(self, x, seed=1, counter=0, particle0=0):
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.empty((len(x), self.G))
        self.lib.gen_gq(_p(x), len(x), seed, counter, particle0, _p(self.blob), _p(out))
        return out


_RNG_LIB = {}


def rng_draws(tmp_path_factory, name, args, n=1 << 20, seed=7):
    if "lib" not in _RNG_LIB:
        lib = _compile(tmp_path_factory.mktemp("rng"), {"rng.cpp": RNG_HARNESS}, "rng.cpp")
        lib.rng_draws.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_ulonglong, ctypes.c_void_p]
        _RNG_LIB["lib"] = lib
    a = np.ascontiguousarray(args + [0.0] * 4, dtype=np.float64)
    out = np.empty(n)
    assert _RNG_LIB["lib"].rng_draws(name.encode(), _p(a), n, seed, _p(out)) == 0
    return out


def _ppc_data(rng, N=12):
    x = rng.normal(size=N)
    return {"N": N, "x": x.tolist(), "y": (0.5 + 1.5 * x + 0.7 * rng.normal(size=N)).tolist()}


def _ppc_rows(rng, n):
    return np.column_stack([rng.normal(size=n), rng.normal(size=n), rng.normal(size=n) * 0.5])


# ------------------------------------------------------------------------------------------------ the density is unchanged
# sha256 of GeneratedSource.text for every fixture, taken from the generator before generated quantities existed
_DENSITY_DIGESTS = [
    ("arma11.stan", "420b53835f1ffa128304fb19688ba9b21c5c978ccf67d55b506dc7428f437d66"),
    ("arma_series.stan", "99d68dddc5badf82c7b4b65e99c548e5d13446483f8584dc88cc30f927e39422"),
    ("containers.stan", "eb12829ef1001df7bf53fcf6441ed83de1ce0aff45e8bdb069bb8414da5023d4"),
    ("containers.stan", "42bbd0cdfbdf336741d88cd84eab34ed52813cafdbd0be0ce34226a99d442041"),
    ("dirichlet_multinomial.stan", "f496afadd0ab0cf32edf3d20655cd0172140e784f7736337c00a12a0cb1ad6c0"),
    ("logistic.stan", "25ab10f9ca19852b3f121d2144e2f77931b913db51d3ef17410a2fd2599dd018"),
    ("mixed.stan", "744c427d5179d4570cbe5c3585c4d764d68e02822266bb5e21c2e22f1ffb5210"),
    ("mixture.stan", "6ab9c7a126b850e031c822b99cb8b0d8299af805dae42fb61fddebcf9715ca16"),
    ("prm_kernel.stan", "faf4646423c4e33a696b5672fe40a297a0c05a3a73c3f12e5f869404c72c55fd"),
    ("regression.stan", "d464eb4e0bf401efc142662dcff7df2044257f47553f7137efae3f058b596ee3"),
    ("golden/reference_stan/arma.stan", "0346e548c56a4e869f6f3e01424ab191fad2e81eb69465309e258805c841811c"),
]


def _fixture_data():
    rng = np.random.default_rng(5)
    prm = json.loads((ROOT / "smc-nuts_b200/smcnuts/data/PRMwCD/PRMwCD.json").read_text())
    prm.pop("phi")
    return [_arma_data(), _arma_data(), _containers_data(rng, 0), _containers_data(rng, 1),
            {"K": 4, "alpha": [1.0, 2.0, 0.5, 3.0], "counts": [5, 1, 9, 3]}, _logistic_data(rng),
            {"N": 5, "t": rng.normal(size=5).tolist(), "y": rng.uniform(0.5, 2, 5).tolist(), "k": [1, 0, 3, 2, 1]},
            {"K": 3, "N": 20, "y": rng.normal(size=20).tolist()}, prm, _regression_data(rng),
            SC.load_data(ROOT / "smc-nuts_b200/smcnuts/data/arma/arma.json")]


def test_density_text_is_unchanged_for_every_fixture():
    for (name, digest), data in zip(_DENSITY_DIGESTS, _fixture_data()):
        path = (ROOT / "tests" / name) if name.startswith("golden") else (STAN / name)
        src = SC.generate(path.read_text(), data)
        assert hashlib.sha256(src.text.encode()).hexdigest() == digest, name
        assert src.gq_error is None
    # with generated quantities the density text is the one of the same program without them
    data = _ppc_data(np.random.default_rng(1))
    text = (STAN / "ppc.stan").read_text()
    bare = text[:text.index("generated quantities")]
    assert SC.generate(text, data).text == SC.generate(bare, data).text
    assert SC.generate(text, data).digest != SC.generate(bare, data).digest


# ------------------------------------------------------------------------------------------------ deterministic values
def test_deterministic_generated_quantities_match_numpy(tmp_path):
    rng = np.random.default_rng(3)
    N = 12
    data = _ppc_data(rng, N)
    src = SC.generate((STAN / "ppc.stan").read_text(), data)
    assert src.gq_names == ([f"y_rep.{i}" for i in range(1, N + 1)] + [f"log_lik.{i}" for i in range(1, N + 1)]
                            + ["k_rep", "cv"])
    assert src.gq_dim == 2 * N + 2 and src.param_names == ["alpha", "beta", "sigma"] and src.cdim == src.dim == 3
    h = HostGQ(src, tmp_path / "ppc")
    x = _ppc_rows(rng, 500)
    out = h.gq(x)
    a, b, s = x[:, 0:1], x[:, 1:2], np.exp(x[:, 2:3])
    mu = a + b * np.array(data["x"])[None, :]
    ll = stats.norm.logpdf(np.array(data["y"])[None, :], mu, s)
    np.testing.assert_allclose(out[:, N:2 * N], ll, rtol=1e-13, atol=1e-13 * np.abs(ll).max())
    np.testing.assert_allclose(out[:, -1], s[:, 0] / (np.abs(a[:, 0]) + 1), rtol=1e-13)
    assert np.all(out[:, 2 * N] == np.round(out[:, 2 * N])) and np.all(out[:, 2 * N] >= 0)
    # y_rep is normal(mu, sigma): standardised, the draws of all rows and elements are N(0, 1)
    z = ((out[:, :N] - mu) / s).ravel()
    assert stats.kstest(z, "norm").pvalue > 1e-4

    rd = _regression_data(rng)
    reg = SC.generate((STAN / "regression.stan").read_text(), rd)
    assert reg.gq_names == ["s2"]
    hr = HostGQ(reg, tmp_path / "reg")
    xr = rng.normal(size=(300, reg.dim))
    np.testing.assert_allclose(hr.gq(xr)[:, 0], np.exp(xr[:, -1]) ** 2, rtol=1e-13)


def test_gq_value_only_code_covers_containers_functions_and_densities(tmp_path):
    """Transformed data, container expressions, user functions, _lpmf by value, vectorised draws into arrays of int,
    nested arrays of vectors (BridgeStan's names), categorical_rng of an expression, a while loop and reject."""
    prog = """
functions {
  real twice(real z) { return 2 * z; }
}
data { int<lower=1> N; vector[N] t; array[N] int k; }
transformed data { vector[N] t2 = t .* t; }
parameters { real<lower=0> lam; simplex[3] th; }
model { k ~ poisson(lam); }
generated quantities {
  real lp = poisson_lpmf(k | lam) + twice(sum(t2));
  array[N] int k_rep = poisson_rng(rep_vector(lam, N) .* t2);
  array[2] vector[3] w;
  real c = categorical_rng(th .* th / dot_self(th));
  int steps = 0;
  for (i in 1:2) w[i] = th * i;
  while (steps < 3) steps += 1;
  if (lam > 100) reject("too large");
}
"""
    rng = np.random.default_rng(2)
    N = 5
    t = rng.uniform(0.5, 2, N)
    k = rng.integers(0, 5, N)
    src = SC.generate(prog, {"N": N, "t": t.tolist(), "k": k.tolist()})
    assert src.gq_error is None, src.gq_error
    assert src.gq_names == (["lp"] + [f"k_rep.{i}" for i in range(1, N + 1)]
                            + [f"w.{i}.{j}" for i in (1, 2) for j in (1, 2, 3)] + ["c", "steps"])
    h = HostGQ(src, tmp_path / "c")
    x = rng.normal(size=(400, 3))
    x[0, 0] = 5.0                                                            # lam > 100: rejected, the row is NaN
    out = h.gq(x)
    assert np.all(np.isnan(out[0]))
    out, x = out[1:], x[1:]
    lam = np.exp(x[:, 0])
    lp = stats.poisson.logpmf(k[None, :], lam[:, None]).sum(1) + 2 * np.sum(t * t)
    np.testing.assert_allclose(out[:, 0], lp, rtol=1e-13)
    assert np.all(out[:, 1:N + 1] == np.round(out[:, 1:N + 1]))
    y = x[:, 1:]
    z1 = 1 / (1 + np.exp(-(y[:, 0] - np.log(2))))
    z2 = 1 / (1 + np.exp(-y[:, 1]))
    th = np.column_stack([z1, (1 - z1) * z2, (1 - z1) * (1 - z2)])
    np.testing.assert_allclose(out[:, 1 + N:4 + N], th, rtol=1e-13)
    np.testing.assert_allclose(out[:, 4 + N:7 + N], 2 * th, rtol=1e-13)
    assert set(np.unique(out[:, -2])) <= {1.0, 2.0, 3.0} and np.all(out[:, -1] == 3)


# ------------------------------------------------------------------------------------------------ distributions
def _ks(draws, dist):
    return stats.kstest(draws, dist.cdf).pvalue


def _chi2(draws, dist):
    """chi-square over bins of at least ~50 expected draws each (edges at quantiles of the reference distribution)"""
    n = len(draws)
    edges = np.unique(dist.ppf(np.linspace(0, 1, 201)[1:-1]))
    edges = edges[np.isfinite(edges)]
    cdf = np.concatenate([[0.0], dist.cdf(edges), [1.0]])
    expected = n * np.diff(cdf)
    observed = np.bincount(np.searchsorted(edges, draws, side="left"), minlength=len(expected))
    keep = expected > 0
    assert observed[~keep].sum() == 0
    expected, observed = expected[keep], observed[keep]
    if len(expected) < 2:
        return 1.0
    return stats.chisquare(observed, expected * observed.sum() / expected.sum()).pvalue


def _moments_ok(draws, dist, var_check=True):
    n = len(draws)
    m, v, _, k = dist.stats(moments="mvsk")
    m, v, k = float(m), float(v), float(k)
    assert abs(draws.mean() - m) <= 5 * np.sqrt(v / n) + 1e-300, (draws.mean(), m)
    if var_check and np.isfinite(k):
        # 5 first-order standard errors of the sample variance, plus the square of the mean's 5 standard errors (its
        # second-order term, which alone remains when the kurtosis is -2: a fair Bernoulli)
        assert abs(draws.var() - v) <= 5 * np.sqrt((k + 2) * v * v / n) + 25 * v / n, (draws.var(), v)


# (Stan function, arguments, scipy distribution, check the variance)
CONTINUOUS = [
    ("normal", [1.5, 2.0], stats.norm(1.5, 2.0), True),
    ("normal", [-1e3, 1e-3], stats.norm(-1e3, 1e-3), True),
    ("std_normal", [], stats.norm(), True),
    ("student_t", [3.0, 1.0, 2.0], stats.t(3.0, 1.0, 2.0), False),
    ("student_t", [30.0, 0.0, 1.0], stats.t(30.0, 0.0, 1.0), True),
    ("student_t", [0.5, 0.0, 1.0], stats.t(0.5, 0.0, 1.0), None),
    ("cauchy", [2.0, 0.5], stats.cauchy(2.0, 0.5), None),
    ("double_exponential", [1.0, 2.0], stats.laplace(1.0, 2.0), True),
    ("logistic", [-1.0, 0.5], stats.logistic(-1.0, 0.5), True),
    ("lognormal", [0.3, 0.4], stats.lognorm(0.4, scale=np.exp(0.3)), True),
    ("exponential", [2.5], stats.expon(scale=0.4), True),
    ("exponential", [1e-3], stats.expon(scale=1e3), True),
    ("gamma", [1e-3, 1.0], stats.gamma(1e-3), True),
    ("gamma", [0.5, 2.0], stats.gamma(0.5, scale=0.5), True),
    ("gamma", [1.0, 1.0], stats.gamma(1.0), True),
    ("gamma", [50.0, 0.1], stats.gamma(50.0, scale=10.0), True),
    ("inv_gamma", [3.0, 2.0], stats.invgamma(3.0, scale=2.0), False),
    ("inv_gamma", [6.0, 0.5], stats.invgamma(6.0, scale=0.5), True),
    ("beta", [0.5, 0.5], stats.beta(0.5, 0.5), True),
    ("beta", [2.0, 5.0], stats.beta(2.0, 5.0), True),
    ("beta", [0.3, 4.0], stats.beta(0.3, 4.0), True),
    ("uniform", [-2.0, 3.0], stats.uniform(-2.0, 5.0), True),
]


@pytest.mark.parametrize("name,args,dist,var", CONTINUOUS, ids=[f"{c[0]}{c[1]}" for c in CONTINUOUS])
def test_continuous_rng_functions_pass_ks_against_scipy(tmp_path_factory, name, args, dist, var):
    """2^20 draws, one per particle stream, seed 7; KS p-value above 1e-4 and the moments within 5 standard errors."""
    d = rng_draws(tmp_path_factory, name, args)
    assert np.all(np.isfinite(d)) or name in ("inv_gamma",)
    if name == "gamma" and args[0] < 0.1:
        # about half of the Gamma(0.001) draws lie below the smallest double: they come back as 0, and are compared
        # through a randomised probability transform (uniform below the cdf at half the smallest subnormal)
        from scipy.special import gammaln
        f0 = np.exp(args[0] * (np.log(np.nextafter(0, 1)) - np.log(2.0)) - gammaln(args[0] + 1))
        u = dist.cdf(d)
        zero = d == 0
        assert 0.4 < zero.mean() < 0.55
        u[zero] = np.random.default_rng(0).uniform(0, f0, zero.sum())
        assert stats.kstest(u, "uniform").pvalue > 1e-4
    else:
        assert _ks(d, dist) > 1e-4
    if var is not None:
        _moments_ok(d, dist, var)


DISCRETE = ([("poisson", [lam], stats.poisson(lam)) for lam in (0.0, 1e-3, 9.99, 10.0, 1e3, 1e7)]
            + [("binomial", [n, p], stats.binom(n, p)) for n in (0, 1, 20, 10000) for p in (0.0, 1e-4, 0.5, 1.0)]
            + [("binomial", [10000, 0.97], stats.binom(10000, 0.97)), ("binomial", [40, 0.2], stats.binom(40, 0.2))]
            + [("bernoulli", [0.3], stats.bernoulli(0.3)), ("bernoulli_logit", [-2.0], stats.bernoulli(1 / (1 + np.exp(2.0)))),
               ("poisson_log", [np.log(30.0)], stats.poisson(30.0)), ("poisson_log", [np.log(2.0)], stats.poisson(2.0)),
               ("neg_binomial_2", [5.0, 2.0], stats.nbinom(2.0, 2.0 / 7.0)),
               ("neg_binomial_2", [1e3, 0.5], stats.nbinom(0.5, 0.5 / 1000.5)),
               ("categorical", [0.1, 0.2, 0.3, 0.4], stats.rv_discrete(values=([1, 2, 3, 4], [0.1, 0.2, 0.3, 0.4])))])


@pytest.mark.parametrize("name,args,dist", DISCRETE, ids=[f"{c[0]}{c[1]}" for c in DISCRETE])
def test_discrete_rng_functions_pass_chi_square_against_scipy(tmp_path_factory, name, args, dist):
    """2^20 draws, seed 7; chi-square p-value above 1e-4 over quantile bins, integer values, moments within 5 SE."""
    d = rng_draws(tmp_path_factory, name, args)
    assert np.all(np.isfinite(d)) and np.all(d == np.round(d))
    m, v = float(dist.mean()), float(dist.var())
    if v == 0.0:
        assert np.all(d == m)
        return
    assert _chi2(d, dist) > 1e-4
    _moments_ok(d, dist)


@pytest.mark.parametrize("name,args", [
    ("normal", [0.0, -1.0]), ("normal", [np.inf, 1.0]), ("normal", [0.0, 0.0]), ("normal", [np.nan, 1.0]),
    ("student_t", [0.0, 0.0, 1.0]), ("cauchy", [0.0, -2.0]), ("exponential", [0.0]), ("gamma", [-1.0, 1.0]),
    ("gamma", [1.0, np.inf]), ("inv_gamma", [1.0, 0.0]), ("beta", [0.0, 1.0]), ("uniform", [1.0, 1.0]),
    ("lognormal", [0.0, np.nan]), ("logistic", [0.0, 0.0]), ("double_exponential", [0.0, -1.0]),
    ("bernoulli", [1.5]), ("bernoulli_logit", [np.nan]), ("binomial", [-1.0, 0.5]), ("binomial", [3.5, 0.5]),
    ("binomial", [10.0, 1.1]), ("poisson", [-1.0]), ("poisson", [2.0 ** 30]), ("poisson", [np.nan]),
    ("poisson_log", [31 * np.log(2.0)]), ("neg_binomial_2", [0.0, 1.0]), ("neg_binomial_2", [1e12, 1e3]),
    ("categorical", [0.5, 0.5, 0.5, -0.5]), ("categorical", [0.3, 0.3, 0.3, 0.3])])
def test_invalid_arguments_give_nan(tmp_path_factory, name, args):
    d = rng_draws(tmp_path_factory, name, args, n=64)
    assert np.all(np.isnan(d))


# ------------------------------------------------------------------------------------------------ reproducibility
def test_draws_do_not_depend_on_batching_or_row_order(tmp_path):
    rng = np.random.default_rng(4)
    data = _ppc_data(rng, 12)
    h = HostGQ(SC.generate((STAN / "ppc.stan").read_text(), data), tmp_path / "ppc")
    x = _ppc_rows(rng, 1000)
    full = h.gq(x, seed=99, counter=3)
    two = np.concatenate([h.gq(x[:377], seed=99, counter=3), h.gq(x[377:], seed=99, counter=3, particle0=377)])
    assert np.array_equal(full.view(np.uint64), two.view(np.uint64))
    for i in rng.permutation(1000)[:200]:
        assert np.array_equal(h.gq(x[i:i + 1], seed=99, counter=3, particle0=int(i))[0].view(np.uint64),
                              full[i].view(np.uint64))
    assert not np.array_equal(full[:, :12], h.gq(x, seed=99, counter=4)[:, :12])        # another call: other draws
    assert not np.array_equal(full[:, :12], h.gq(x, seed=98, counter=3)[:, :12])
    np.testing.assert_array_equal(full[:, 12:24], h.gq(x, seed=98, counter=4)[:, 12:24])  # deterministic columns


# ------------------------------------------------------------------------------------------------ refusals and deferral
BASE = """
data { int N; vector[N] y; }
parameters { real mu; real<lower=0> s; }
model { y ~ normal(mu, s); }
"""


def test_target_in_gq_and_rng_outside_gq_are_refused_with_the_line():
    data = {"N": 3, "y": [0.1, 0.2, 0.3]}
    src = SC.generate(BASE + "generated quantities {\n  real a = mu;\n  target += a;\n}\n", data)
    assert src.gq_error is not None and "line 7" in src.gq_error and src.gq_dim == 0
    src = SC.generate(BASE + "generated quantities {\n  real a = mu;\n  y ~ normal(a, 1);\n}\n", data)
    assert "line 7" in src.gq_error
    src = SC.generate(BASE + "generated quantities {\n  real a = phi;\n}\n", {**data})
    assert "line 6" in src.gq_error
    with pytest.raises(SC.StanSubsetError, match="line 5.*only allowed in generated quantities"):
        SC.generate(BASE.replace("y ~ normal(mu, s);", "real z;\n  z = normal_rng(mu, s);"), data)
    with pytest.raises(SC.StanSubsetError, match="line 4.*only allowed in generated quantities"):
        SC.generate(BASE.replace("real<lower=0> s; }", "real<lower=0> s; }\ntransformed parameters { real z = normal_rng(0, 1); }"),
                    data)


def test_redeclarations_in_gq_are_refused_with_the_line_and_sibling_scopes_are_not():
    data = {"N": 3, "y": [0.1, 0.2, 0.3]}
    tp = BASE.replace("model {", "transformed parameters {\n  vector[2] m = rep_vector(mu, 2);\n}\nmodel {")
    src = SC.generate(tp + "generated quantities {\n  real m = 2;\n}\n", data)       # a transformed parameter
    assert "line 9" in src.gq_error and "already declared" in src.gq_error and src.gq_dim == 0
    src = SC.generate(BASE + "generated quantities {\n  real a = mu;\n  {\n    real a = 1;\n  }\n}\n", data)
    assert "line 8" in src.gq_error and "already declared" in src.gq_error
    src = SC.generate(BASE + "generated quantities {\n  real a = mu;\n  int a = 1;\n}\n", data)
    assert "line 7" in src.gq_error
    src = SC.generate(BASE + "generated quantities {\n  real a = 0;\n  { real r = mu; a += r; }\n"
                      "  { real r = s; a += r; }\n  for (i in 1:2) { real r = i; a += r; }\n}\n", data)
    assert src.gq_error is None and src.gq_names == ["a"]


def test_more_generated_quantities_than_a_row_of_shared_memory_holds_are_deferred():
    data = {"N": 3, "y": [0.1, 0.2, 0.3]}
    src = SC.generate(BASE + "generated quantities {\n  array[24577] real z;\n}\n", data)
    assert "24577 generated quantities" in src.gq_error and src.gq_dim == 0
    src = SC.generate(BASE + "generated quantities {\n  array[24576] real z;\n}\n", data)
    assert src.gq_error is None and src.gq_dim == 24576


def test_a_gq_block_outside_the_subset_keeps_the_density_and_defers_its_error(tmp_path):
    data = {"N": 3, "y": [0.1, 0.2, 0.3]}
    for gq, line in (("  matrix[2, 2] W = wishart_rng(4, S);\n", 6), ("  cov_matrix[2] W;\n", 6),
                     ("  real a = mu;\n  real b = wishart_rng(4, a);\n", 7)):
        src = SC.generate(BASE + "generated quantities {\n" + gq + "}\n", data)
        assert src.gq_error is not None and f"line {line}" in src.gq_error, (gq, src.gq_error)
        assert src.text == SC.generate(BASE, data).text and src.gq_dim == 0
        assert "GDIM = 0" in src.gq_text


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_plugin_matches_the_host_build_into_a_guarded_buffer(tmp_path):
    from smcnuts import _cabi, _device as dev
    from smcnuts.model.generated import GeneratedModel
    from tests.test_gpu_dispatch import guarded
    rng = np.random.default_rng(31)
    N = 12
    data = _ppc_data(rng, N)
    m = GeneratedModel((STAN / "ppc.stan").read_text(), data, "ppc")
    h = HostGQ(m.source, tmp_path / "ppc")
    assert m.gq_dim == 2 * N + 2 and m.gq_names == m.source.gq_names
    n = (1 << 20) - 37                                             # a partial last block of 64 rows
    x = _ppc_rows(rng, n)
    out, check = guarded(n * m.gq_dim)
    _cabi.call("smcb_model_generated_quantities", m._h, dev.ptr(dev.to_device(x)), n, 1234, 5, 0, dev.ptr(out),
               dev.stream_ptr())
    check()
    got = out.view(n, m.gq_dim).cpu().numpy()
    ref = h.gq(x, seed=1234, counter=5)
    det = slice(N, 2 * N)
    np.testing.assert_allclose(got[:, det], ref[:, det], rtol=1e-13, atol=1e-13 * np.abs(ref[:, det]).max())
    np.testing.assert_allclose(got[:, -1], ref[:, -1], rtol=1e-13)
    # draws: equal to rounding of the device exp / log / cos; a rounding difference may flip a rare accept / reject
    draws = np.concatenate([got[:, :N], got[:, 2 * N:2 * N + 1]], 1)
    rdraws = np.concatenate([ref[:, :N], ref[:, 2 * N:2 * N + 1]], 1)
    same = np.abs(draws - rdraws) <= 1e-12 * np.maximum(np.abs(rdraws), 1.0)
    assert same.mean() >= 0.999, same.mean()
    # host in -> host out, device in -> device out; batching with particle0 reproduces the rows
    np.testing.assert_array_equal(m.generated_quantities(x[:9], seed=1234, counter=5), got[:9])
    xd = dev.to_device(x[100:300])
    gd = m.generated_quantities(xd, seed=1234, counter=5, particle0=100)
    assert gd.is_cuda and np.array_equal(gd.cpu().numpy(), got[100:300])
    assert m.generated_quantities(x[:7].reshape(7, 1, 3), seed=1).shape == (7, 1, m.gq_dim)
    # invalid arguments: NaN rows
    bad = GeneratedModel(BASE + "generated quantities {\n  real z = normal_rng(mu, -s);\n}\n",
                         {"N": 3, "y": [0.1, 0.2, 0.3]}, "bad")
    assert np.all(np.isnan(bad.generated_quantities(rng.normal(size=(64, 2)))))
    # deferred error
    w = GeneratedModel(BASE + "generated quantities {\n  real a = mu;\n  real b = wishart_rng(4, a);\n}\n",
                       {"N": 3, "y": [0.1, 0.2, 0.3]}, "wish")
    assert np.isfinite(w.logpdf(rng.normal(size=(4, 2)), 1.0)).all()
    from smcnuts.model.stan_codegen import StanSubsetError
    with pytest.raises(StanSubsetError, match="line 7"):
        w.generated_quantities(rng.normal(size=(4, 2)))
    from smcnuts.model.device_model import make_model
    assert _cabi.lib().smcb_model_gq_dim(make_model("arma")._h) == 0          # built-in models have none


@pytest.mark.gpu
def test_wide_rows_are_staged_for_fewer_particles_per_block(tmp_path):
    """G = 601: 42 rows of a block fit in shared memory (the other 22 threads idle); 1000 rows end in a partial block."""
    from smcnuts import _cabi, _device as dev
    from smcnuts.model.generated import GeneratedModel
    from tests.test_gpu_dispatch import guarded
    prog = BASE + """generated quantities {
  array[300] real z;
  array[300] int k;
  real e = exp(mu);
  for (i in 1:300) {
    z[i] = normal_rng(mu * i, s);
    k[i] = poisson_rng(s * i);
  }
}
"""
    data = {"N": 3, "y": [0.1, 0.2, 0.3]}
    m = GeneratedModel(prog, data, "wide")
    h = HostGQ(m.source, tmp_path / "wide")
    assert m.gq_dim == 601
    rng = np.random.default_rng(40)
    n = 1000
    x = np.column_stack([rng.normal(size=n), rng.normal(size=n) * 0.3])
    out, check = guarded(n * m.gq_dim)
    _cabi.call("smcb_model_generated_quantities", m._h, dev.ptr(dev.to_device(x)), n, 77, 1, 5, dev.ptr(out),
               dev.stream_ptr())
    check()
    got = out.view(n, m.gq_dim).cpu().numpy()
    ref = h.gq(x, seed=77, counter=1, particle0=5)
    np.testing.assert_allclose(got[:, -1], np.exp(x[:, 0]), rtol=1e-13)
    same = np.abs(got - ref) <= 1e-12 * np.maximum(np.abs(ref), 1.0)
    assert same.mean() >= 0.999, same.mean()
    assert np.all(got[:, 300:600] == np.round(got[:, 300:600]))


def _run(m, K, N, seed, step):
    from smcnuts.distributions import StdNormal
    from smcnuts.smc_sampler import SMCSampler
    s = SMCSampler(K=K, N=N, target=m, step_size=step, sample_proposal=StdNormal(m.dim), momentum_proposal=StdNormal(m.dim),
                   lkernel="forwardsLKernel", tempering=True, rng=seed, generated_quantities=True)
    s.sample(show_progress=False)
    assert s.phi[-1] == 1.0
    return s


@pytest.mark.gpu
def test_sampler_posterior_predictive_of_a_normal_mean():
    """y_i ~ N(theta, 1), theta ~ N(0, 10^2): the predictive of a new y is N(post mean, post var + 1)."""
    from smcnuts.model.generated import GeneratedModel
    prog = """
data { int N; vector[N] y; real phi; }
parameters { real theta; }
model { theta ~ normal(0, 10); target += phi * normal_lpdf(y | theta, 1); }
generated quantities {
  array[300] real y_new;
  real t2 = theta;
  for (i in 1:300) y_new[i] = normal_rng(theta, 1);
}
"""
    rng = np.random.default_rng(12)
    y = 1.3 + rng.normal(size=20)
    m = GeneratedModel(prog, {"N": 20, "y": y.tolist()}, "nmean")
    s = _run(m, 20, 1 << 16, 5, 0.3)
    pv = 1 / (1 / 100 + 20)
    pm = pv * y.sum()
    # G = 301 > 256: the weighted moments are reduced in column blocks
    assert s.gq_draws.shape == (s.samples.n_local, 301) and s.gq_draws.is_cuda
    assert m.gq_names[:2] == ["y_new.1", "y_new.2"] and m.gq_names[-1] == "t2"
    mean, var = s.gq_mean_estimate, s.gq_variance_estimate
    assert mean.shape == var.shape == (301,) and s.leapfrogs.sum() > 0 and s.run_time > 0
    ess = s.ess[-1]
    np.testing.assert_allclose(mean[-1], s.mean_estimate[-1][0], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(var[-1], s.variance_estimate[-1][0], rtol=1e-10)
    se_m = np.sqrt((pv + 1) / ess)
    assert np.all(np.abs(mean[:300] - pm) <= 5 * se_m), (mean, pm, se_m)
    # predictive variance = posterior variance + sigma^2, on the particle approximation: the weighted variance of theta
    # (whose own error is the sampler's, not the draws') plus the variance of the N(0, 1) noise, within 5 standard errors
    # of a weighted variance of unit normal draws
    se_v = np.sqrt(2 / ess)
    assert np.all(np.abs(var[:300] - (var[-1] + 1)) <= 5 * se_v), (var, var[-1] + 1, se_v)
    assert abs(var[:300].mean() - (pv + 1)) <= 0.05 * (pv + 1), (var[:300].mean(), pv + 1)
    # the blocks reduce what one launch per column would: the moments of each column against a host restatement
    w = s.samples.wn.cpu().numpy()
    d = s.gq_draws.cpu().numpy()
    mw = w @ d
    np.testing.assert_allclose(mean, mw, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(var, w @ (d - mw) ** 2, rtol=1e-8, atol=1e-12)


@pytest.mark.gpu
def test_sampler_posterior_predictive_of_a_poisson_gamma_model():
    """k_i ~ Poisson(lam), lam ~ Gamma(a, b): the predictive of a new count is negative binomial with r = a + sum k and
    p = (b + n) / (b + n + 1)."""
    from smcnuts.model.generated import GeneratedModel
    prog = """
data { int N; array[N] int k; real phi; }
parameters { real<lower=0> lam; }
model { lam ~ gamma(3, 0.5); target += phi * poisson_lpmf(k | lam); }
generated quantities { int k_new = poisson_rng(lam); }
"""
    rng = np.random.default_rng(13)
    k = rng.poisson(4.0, size=15)
    m = GeneratedModel(prog, {"N": 15, "k": k.tolist()}, "pg")
    s = _run(m, 20, 1 << 16, 6, 0.2)
    r, p = 3 + k.sum(), (0.5 + 15) / (0.5 + 15 + 1)
    nb = stats.nbinom(r, p)
    ess = s.ess[-1]
    mean, var = s.gq_mean_estimate[0], s.gq_variance_estimate[0]
    assert np.all(s.gq_draws.cpu().numpy() == np.round(s.gq_draws.cpu().numpy()))
    assert abs(mean - nb.mean()) <= 5 * np.sqrt(nb.var() / ess), (mean, nb.mean())
    kurt = float(nb.stats(moments="k"))
    assert abs(var - nb.var()) <= 5 * nb.var() * np.sqrt((kurt + 2) / ess), (var, nb.var())
