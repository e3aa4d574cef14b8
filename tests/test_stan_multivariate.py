"""Multivariate normal densities, cholesky_decompose, add_diag and gp_exp_quad_cov in generated Stan models.

CPU: the generated struct is built with g++ (the text nvcc compiles for the device) and checked against scipy's
multivariate_normal (data covariances) and a torch autograd restatement with torch.linalg.cholesky (covariances built
from parameters) at K, N in {1, 2, 3, 7, 16, 32}; the propto drops of `~`; -inf for non-symmetric, indefinite and NaN
matrices; the folding of data covariances at generation time; the per-thread size budget; refusals with their line; and
multi_normal(_cholesky)_rng in generated quantities (KS of the marginals, sample covariance, NaN rows, batching).
GPU: the plug-in against the host build into guarded buffers, and SMCSampler against closed-form or quadrature posteriors.
"""
import math

import numpy as np
import pytest
import torch
from scipy import stats

from tests.test_stan_codegen import SC, STAN, HostModel
from tests.test_stan_generated_quantities import HostGQ

SIZES = (1, 2, 3, 7, 16, 32)


def _gp_data(rng, N):
    x = np.sort(rng.uniform(-3, 3, N))
    return {"N": N, "x": x.tolist(), "y": (np.sin(x) + 0.3 * rng.normal(size=N)).tolist()}


def _gp_torch(u, data, phi):
    """A, B and grad(A + phi B) of tests/stan/gp.stan at unconstrained rows u (log rho, log alpha, log sigma)"""
    xs = torch.tensor(data["x"], dtype=torch.float64)
    y = torch.tensor(data["y"], dtype=torch.float64)
    A, B, G = [], [], []
    for row in u:
        t = torch.tensor(row, dtype=torch.float64, requires_grad=True)
        rho, alpha, sigma = torch.exp(t)
        Kx = alpha ** 2 * torch.exp(-(xs[:, None] - xs[None, :]) ** 2 / (2 * rho ** 2)) + sigma ** 2 * torch.eye(len(xs),
                                                                                                              dtype=torch.float64)
        L = torch.linalg.cholesky(Kx)
        z = torch.linalg.solve_triangular(L, y[:, None], upper=False)[:, 0]
        b = -0.5 * len(xs) * math.log(2 * math.pi) - torch.log(torch.diagonal(L)).sum() - 0.5 * (z ** 2).sum()
        a = t.sum() - 6.0 * torch.log(rho) - 5.0 / rho - 0.5 * alpha ** 2 - 0.5 * sigma ** 2
        (a + phi * b).backward()
        A.append(a.item()), B.append(b.item()), G.append(t.grad.numpy().copy())
    return np.array(A), np.array(B), np.array(G)


def _close(got, ref, tol, what):
    err = np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1.0))
    assert err <= tol, (what, err)


@pytest.mark.parametrize("N", SIZES)
def test_gp_regression_matches_a_torch_cholesky_restatement(tmp_path, N):
    rng = np.random.default_rng(100 + N)
    data = _gp_data(rng, N)
    src = SC.generate((STAN / "gp.stan").read_text(), data)
    assert src.dim == 3 and src.param_names == ["rho", "alpha", "sigma"]
    assert "#pragma unroll 1" in src.text
    h = HostModel(src, tmp_path / "gp")
    u = np.column_stack([rng.normal(0, 0.5, 40), rng.normal(0, 0.5, 40), rng.normal(-1, 0.3, 40)])
    phi = 0.37
    A, B, g = h.split(u, phi)
    rA, rB, rg = _gp_torch(u, data, phi)
    _close(A, rA, 1e-12, "A")
    _close(B, rB, 1e-9, "B")
    _close(g, rg, 1e-8, "grad")


def _mvn_data(rng, K, N):
    Q = rng.normal(size=(K, K))
    Sigma = Q @ Q.T / K + 0.5 * np.eye(K)
    Q0 = rng.normal(size=(K, K))
    Sigma0 = 2.0 * (Q0 @ Q0.T / K + np.eye(K))
    y = rng.multivariate_normal(np.linspace(-1, 1, K), Sigma, size=N)
    return {"K": K, "N": N, "y": y.tolist(), "Sigma": Sigma.tolist(), "mu0": np.zeros(K).tolist(), "Sigma0": Sigma0.tolist()}


@pytest.mark.parametrize("K", SIZES)
def test_data_covariance_matches_scipy_and_is_factored_at_generation_time(tmp_path, K):
    rng = np.random.default_rng(200 + K)
    N = 4
    data = _mvn_data(rng, K, N)
    src = SC.generate((STAN / "mvn.stan").read_text(), data)
    # both covariances are data: their factors are in the blob, and eval() factors nothing
    for name in ("Sigma", "Sigma0"):
        fac = np.linalg.cholesky(np.array(data[name])).ravel()
        blob = np.array(src.blob)
        assert any(np.array_equal(blob[o:o + K * K], fac) for o in range(len(blob) - K * K + 1)), name
    assert "sqrt(" not in src.text and "ok = false" not in src.text
    h = HostModel(src, tmp_path / "mvn")
    mu = rng.normal(size=(30, K))
    phi = 0.61
    A, B, g = h.split(mu, phi)
    S, S0, y = np.array(data["Sigma"]), np.array(data["Sigma0"]), np.array(data["y"])
    rB = np.array([stats.multivariate_normal(m, S).logpdf(y).sum() for m in mu])
    # `~` drops -K/2 log 2 pi and -log det of the data Sigma0: only the quadratic form is left
    rA = -0.5 * np.einsum("ni,ij,nj->n", mu, np.linalg.inv(S0), mu)
    rg = -mu @ np.linalg.inv(S0) + phi * (y.sum(0)[None, :] - N * mu) @ np.linalg.inv(S)
    _close(A, rA, 1e-11, "A")
    _close(B, rB, 1e-11, "B")
    _close(g, rg, 1e-10, "grad")


MEANS = """
data { int K; int N; array[N] vector[K] y; matrix[K, K] S; }
transformed data { matrix[K, K] L = cholesky_decompose(S); }
parameters { array[N] vector[K] m; vector[K] c; }
model {
  target += multi_normal_cholesky_lpdf(y | m, L);
  target += multi_normal_cholesky_lpdf(y | c, L);
  y[1] ~ multi_normal_cholesky(c, L);
}
"""


def test_arrays_of_vectors_with_shared_and_per_element_means(tmp_path):
    rng = np.random.default_rng(3)
    K, N = 3, 5
    Q = rng.normal(size=(K, K))
    S = Q @ Q.T + np.eye(K)
    y = rng.normal(size=(N, K))
    src = SC.generate(MEANS, {"K": K, "N": N, "y": y.tolist(), "S": S.tolist()})
    assert "sqrt(" not in src.text                    # L is transformed data of a data matrix: folded
    h = HostModel(src, tmp_path / "means")
    x = rng.normal(size=(20, (N + 1) * K))
    A, B, g = h.split(x, 1.0)
    ref = []
    for row in x:
        m, c = row[:N * K].reshape(N, K), row[N * K:]
        full = sum(stats.multivariate_normal(m[n], S).logpdf(y[n]) for n in range(N))
        full += stats.multivariate_normal(c, S).logpdf(y).sum()
        # under `~` with a data factor only the quadratic form is kept
        d = y[0] - c
        full += -0.5 * d @ np.linalg.solve(S, d)
        ref.append(full)
    _close(A, np.array(ref), 1e-11, "A")
    assert np.all(B == 0)


PROPTO = """
data { int K; vector[K] y; array[K] real xd; }
parameters { real<lower=0> s; }
model {
  matrix[K, K] L = cholesky_decompose(add_diag(gp_exp_quad_cov(xd, 1.0, 1.0), s));
  STMT
}
"""


def test_tilde_drops_the_constant_and_keeps_the_log_determinant_of_a_parameter_factor(tmp_path):
    rng = np.random.default_rng(4)
    K = 4
    y = rng.normal(size=K)
    u = rng.normal(size=(10, 1))
    out = {}
    for key, stmt in (("target", "target += multi_normal_cholesky_lpdf(y | rep_vector(0, K), L);"),
                      ("tilde", "y ~ multi_normal_cholesky(rep_vector(0, K), L);")):
        src = SC.generate(PROPTO.replace("STMT", stmt), {"K": K, "y": y.tolist(), "xd": np.linspace(0, 1, K).tolist()})
        out[key] = HostModel(src, tmp_path / key).split(u)
    (At, _, gt), (Ad, _, gd) = out["target"], out["tilde"]
    np.testing.assert_allclose(At - Ad, -0.5 * K * math.log(2 * math.pi) + np.zeros(len(u)), rtol=1e-12)
    np.testing.assert_allclose(gt, gd, rtol=1e-12)
    xd = np.linspace(0, 1, K)
    for row, a in zip(u, At):
        s = math.exp(row[0])
        S = np.exp(-0.5 * (xd[:, None] - xd[None, :]) ** 2) + s * np.eye(K)
        np.testing.assert_allclose(a, stats.multivariate_normal(np.zeros(K), S).logpdf(y) + row[0], rtol=1e-11)


def _ar1_data(rng, K, N):
    S = 1.3 ** 2 * 0.6 ** np.abs(np.subtract.outer(np.arange(K), np.arange(K)))
    return {"K": K, "N": N, "y": rng.multivariate_normal(np.zeros(K), S, size=N).tolist()}


def _ar1_torch(u, data, phi):
    y = torch.tensor(data["y"], dtype=torch.float64)
    K = data["K"]
    lag = torch.tensor(np.abs(np.subtract.outer(np.arange(K), np.arange(K))), dtype=torch.float64)
    A, B, G = [], [], []
    for row in u:
        t = torch.tensor(row, dtype=torch.float64, requires_grad=True)
        s, r, m = torch.exp(t[0]), t[1], t[2:]
        S = s ** 2 * torch.where(lag == 0, torch.ones_like(lag), r ** lag)
        L = torch.linalg.cholesky(S)
        z = torch.linalg.solve_triangular(L, (y - m).T, upper=False)
        b = -0.5 * y.numel() * math.log(2 * math.pi) - len(y) * torch.log(torch.diagonal(L)).sum() - 0.5 * (z ** 2).sum()
        a = t[0] - t[0] - 0.5 * t[0] ** 2 - 0.5 * r ** 2 - 0.5 * (m ** 2).sum() / 9.0
        (a + phi * b).backward()
        A.append(a.item()), B.append(b.item()), G.append(t.grad.numpy().copy())
    return np.array(A), np.array(B), np.array(G)


@pytest.mark.parametrize("K", (1, 2, 3, 7, 16))
def test_parameter_covariance_matches_torch_and_is_minus_infinity_where_not_positive_definite(tmp_path, K):
    rng = np.random.default_rng(300 + K)
    data = _ar1_data(rng, K, 6)
    src = SC.generate((STAN / "ar1_cov.stan").read_text(), data)
    h = HostModel(src, tmp_path / "ar1")
    u = np.column_stack([rng.normal(0, 0.3, 60), rng.uniform(-1.5, 1.5, 60), rng.normal(size=(60, K))])
    phi = 0.8
    A, B, g = h.split(u, phi)
    # lognormal(0, 1) of s under `~`: -log s - log(s)^2 / 2; with the Jacobian log s the first cancels
    bad = np.abs(u[:, 1]) >= 1.0
    if K == 1:
        bad[:] = False                                 # r^0 = 1: a 1 x 1 covariance is s^2 whatever r is
    assert np.all(A[bad] == -np.inf)
    good = ~bad
    rA, rB, rg = _ar1_torch(u[good], data, phi)
    _close(A[good], rA, 1e-12, "A")
    _close(B[good], rB, 1e-9, "B")
    _close(g[good], rg, 1e-7, "grad")


CHOL = """
parameters { real a; real b; real c; real d; }
model {
  matrix[2, 2] M;
  M[1, 1] = a; M[1, 2] = b; M[2, 1] = c; M[2, 2] = d;
  matrix[2, 2] L = cholesky_decompose(M);
  target += L[1, 1] + L[2, 1] + L[2, 2] + L[1, 2];
}
"""


def test_cholesky_decompose_checks_symmetry_positive_definiteness_and_finiteness(tmp_path):
    h = HostModel(SC.generate(CHOL, {}), tmp_path / "chol")
    rows = np.array([[4.0, 2.0, 2.0, 5.0],              # SPD: L = [[2, 0], [1, 2]]
                     [4.0, 2.0, 2.0 + 5e-9, 5.0],       # asymmetric within 1e-8: accepted, lower triangle read
                     [4.0, 2.0, 2.0 + 2e-8, 5.0],       # beyond 1e-8
                     [1.0, 2.0, 2.0, 1.0],              # indefinite
                     [4.0, np.nan, np.nan, 5.0],
                     [np.nan, 2.0, 2.0, 5.0],
                     [4.0, 2.0, 2.0, np.inf],
                     [0.0, 0.0, 0.0, 1.0]])            # singular
    A, _, g = h.split(rows)
    assert A[0] == 5.0 and abs(A[1] - (2.0 + (2.0 + 5e-9) / 2.0 + math.sqrt(5.0 - ((2.0 + 5e-9) / 2) ** 2))) < 1e-15
    assert np.all(A[2:] == -np.inf)
    # d/da (sqrt a + c / sqrt a + sqrt(d - c^2 / a)) at (4, 2, 5): 1/4 - 2/16 + (4/16) / (2 * 2)
    np.testing.assert_allclose(g[0], [0.25 - 0.125 + 0.0625, 0.0, 0.5 - 0.25, 0.25], rtol=1e-14, atol=1e-15)


def test_non_positive_definite_data_covariances_are_refused_with_their_line():
    bad = np.array([[1.0, 2.0], [2.0, 1.0]])
    data = {"K": 2, "N": 1, "y": [[0.0, 0.0]], "Sigma": bad.tolist(), "mu0": [0.0, 0.0], "Sigma0": np.eye(2).tolist()}
    with pytest.raises(SC.StanSubsetError, match=r"line 17: data 'Sigma' is not a symmetric positive definite"):
        SC.generate((STAN / "mvn.stan").read_text(), data)
    data["Sigma"], data["Sigma0"] = np.eye(2).tolist(), [[1.0, 0.5], [0.4, 1.0]]
    with pytest.raises(SC.StanSubsetError, match=r"line 16: data 'Sigma0'"):
        SC.generate((STAN / "mvn.stan").read_text(), data)
    with pytest.raises(SC.StanSubsetError, match=r"line 3: data 'S'"):
        SC.generate(MEANS, {"K": 2, "N": 1, "y": [[0.0, 0.0]], "S": [[1.0, 0.0], [0.0, np.nan]]})


BUDGET = """
data { int n; array[n] real x; }
parameters { real<lower=0> a; real<lower=0> b; real<lower=0> c; }
model {
  a ~ normal(0, 1);
  matrix[n, n] M = cholesky_decompose(add_diag(gp_exp_quad_cov(x, a, b), c));
  target += M[n, n];
}
"""


def test_matrix_locals_are_refused_past_the_per_thread_budget():
    assert SC._Gen.MAX_MATRIX_BYTES == 32768
    # 32 x 32 entries, each a value and 3 tangents: 32768 bytes, exactly the budget
    SC.generate(BUDGET, {"n": 32, "x": np.linspace(0, 1, 32).tolist()})
    with pytest.raises(SC.StanSubsetError, match=r"line 6: matrix locals take 34848 bytes a thread up to 'M' \(33 x 33, 4"):
        SC.generate(BUDGET, {"n": 33, "x": np.linspace(0, 1, 33).tolist()})
    # without tangents: 64 x 64 values
    nodeps = BUDGET.replace("gp_exp_quad_cov(x, a, b), c)", "gp_exp_quad_cov(x, 1.0, 2.0), 0.5)")
    SC.generate(nodeps, {"n": 64, "x": np.linspace(0, 1, 64).tolist()})
    with pytest.raises(SC.StanSubsetError, match=r"line 6: matrix locals take 33800 bytes"):
        SC.generate(nodeps, {"n": 65, "x": np.linspace(0, 1, 65).tolist()})


REFUSE = """
data {{ int K; vector[K] y; matrix[K, K] S; matrix[K, 3] R; array[K] real x; vector[K] xv; }}
parameters {{ real m; }}
model {{
  {stmt}
}}
"""


@pytest.mark.parametrize("stmt,msg", [
    ("matrix[K, 3] L = cholesky_decompose(R);", "cholesky_decompose takes a square matrix"),
    ("target += multi_normal_lpdf(y | rep_vector(m, 3), S);", "the location has 3 elements, the matrix is 4 x 4"),
    ("target += multi_normal_cholesky_lpdf(y | rep_vector(m, K), R);", "takes a square matrix"),
    ("target += multi_normal_lpdf(x | rep_vector(m, K), S);", "the outcome must be a vector or an array of vectors"),
    ("matrix[K, K] G = gp_exp_quad_cov(xv, 1.0, m);", r"gp_exp_quad_cov\(x, alpha, rho\) takes x as array"),
    ("matrix[K, K] G = gp_exp_quad_cov(x, 1.0);", "gp_exp_quad_cov takes 3 argument"),
    ("matrix[K, K] G = gp_exp_quad_cov(x, y, m);", r"gp_exp_quad_cov\(x, alpha, rho\)"),
    ("matrix[K, K] G = add_diag(S, rep_vector(m, 3));", "add_diag adds a real or a vector of size 4"),
])
def test_matrix_functions_outside_their_signatures_are_refused_with_the_line(stmt, msg):
    data = {"K": 4, "y": [0.0] * 4, "S": np.eye(4).tolist(), "R": np.zeros((4, 3)).tolist(), "x": [0.0, 1, 2, 3],
            "xv": [0.0] * 4}
    with pytest.raises(SC.StanSubsetError, match=f"line 5: .*{msg}"):
        SC.generate(REFUSE.format(stmt=stmt), data)


GQ = """
data { int K; vector[K] m; matrix[K, K] S; vector[K] y; }
transformed data { matrix[K, K] L = cholesky_decompose(S); }
parameters { real a; real r; }
model { a ~ normal(0, 1); r ~ normal(0, 1); }
generated quantities {
  vector[K] y1 = multi_normal_rng(m + a, S);
  array[2] vector[K] y2;
  y2[2] = multi_normal_cholesky_rng(m, L);
  y2[1] = multi_normal_cholesky_rng(m, L);
  real ll = multi_normal_cholesky_lpdf(y | m + a, L);
  real ll2 = multi_normal_lpdf(y | m, add_diag(S, r));
}
"""


def _gq_data(K):
    Q = np.random.default_rng(K).normal(size=(K, K))
    S = Q @ Q.T / K + 0.3 * np.eye(K)
    return {"K": K, "m": np.linspace(-1, 2, K).tolist(), "S": S.tolist(), "y": np.linspace(0, 1, K).tolist()}, S


@pytest.mark.parametrize("K", (1, 3, 7))
def test_multi_normal_draws_and_densities_in_generated_quantities(tmp_path, K):
    data, S = _gq_data(K)
    src = SC.generate(GQ, data)
    assert src.gq_error is None and src.gq_dim == 3 * K + 2
    h = HostGQ(src, tmp_path / "gq")
    n = 1 << 20
    x = np.zeros((n, 2))
    out = h.gq(x, seed=5)
    m = np.array(data["m"])
    for block in (out[:, :K], out[:, K:2 * K], out[:, 2 * K:3 * K]):
        for i in range(K):
            assert stats.kstest(block[:, i], stats.norm(m[i], math.sqrt(S[i, i])).cdf).pvalue > 1e-4
        c = np.cov(block.T).reshape(K, K)
        se = np.sqrt((S * S + np.outer(np.diag(S), np.diag(S))) / n)
        assert np.all(np.abs(c - S) <= 4 * se)
    # two calls draw independently; the second element of y2 was drawn first
    assert not np.array_equal(out[:, K:2 * K], out[:, 2 * K:3 * K])
    # the densities by value
    xs = np.random.default_rng(1).normal(size=(50, 2))
    v = h.gq(xs)
    y = np.array(data["y"])
    for row, o in zip(xs, v):
        Sr = S + row[1] * np.eye(K)
        if np.all(np.linalg.eigvalsh(Sr) > 0):
            np.testing.assert_allclose(o[-2], stats.multivariate_normal(m + row[0], S).logpdf(y), rtol=1e-12)
            np.testing.assert_allclose(o[-1], stats.multivariate_normal(m, Sr).logpdf(y), rtol=1e-10)
        else:
            assert np.all(np.isnan(o))                   # not positive definite: the whole row is NaN
    assert np.isnan(v[:, -1]).any() and not np.isnan(v[:, -1]).all()


NAN_GQ = """
data { int K; }
parameters { real a; real r; }
transformed parameters {
  matrix[K, K] S;
  for (i in 1:K) for (j in 1:K) S[i, j] = pow(r, abs(i - j));
}
model { a ~ normal(0, 1); }
generated quantities {
  vector[K] y = multi_normal_rng(rep_vector(inv(a), K), S);
}
"""


def test_invalid_draw_arguments_make_the_row_nan_and_draws_do_not_depend_on_batching(tmp_path):
    K = 3
    src = SC.generate(NAN_GQ, {"K": K})
    assert src.gq_error is None and src.gq_names == ["y.1", "y.2", "y.3"]
    h = HostGQ(src, tmp_path / "nan")
    rng = np.random.default_rng(9)
    x = np.column_stack([rng.uniform(0.5, 2, 1000), rng.uniform(-1.5, 1.5, 1000)])
    x[::7, 0] = 0.0                                    # mu = 1 / 0: not finite
    out = h.gq(x, seed=11, counter=2)
    bad = (x[:, 0] == 0.0) | (np.abs(x[:, 1]) >= 1.0)
    assert np.all(np.isnan(out[bad])) and np.all(np.isfinite(out[~bad]))
    two = np.concatenate([h.gq(x[:377], seed=11, counter=2), h.gq(x[377:], seed=11, counter=2, particle0=377)])
    assert np.array_equal(out.view(np.uint64), two.view(np.uint64))
    for i in rng.permutation(1000)[:100]:
        assert np.array_equal(h.gq(x[i:i + 1], seed=11, counter=2, particle0=int(i))[0].view(np.uint64),
                              out[i].view(np.uint64))
    # a draw is mu + L z, z the particle's first K standard normals: with S = I (r = 0) it is mu + z
    x0 = np.array([[1.0, 0.0], [2.0, 0.0]])
    z = h.gq(x0, seed=11, counter=2) - 1.0 / x0[:, :1]
    z2 = h.gq(np.array([[4.0, 0.0], [0.5, 0.0]]), seed=11, counter=2) - np.array([[0.25], [2.0]])
    np.testing.assert_allclose(z, z2, rtol=0, atol=1e-15)


def test_rng_is_refused_outside_generated_quantities():
    prog = "data { int K; matrix[K, K] S; }\nparameters { real a; }\nmodel {\n  vector[K] v = multi_normal_rng(rep_vector(a, K), S);\n}\n"
    with pytest.raises(SC.StanSubsetError, match="line 4.*only allowed in generated quantities"):
        SC.generate(prog, {"K": 2, "S": np.eye(2).tolist()})


# ------------------------------------------------------------------------------------------------ GPU
def _logp_grad_guarded(m, x):
    from smcnuts import _cabi, _device as dev
    from tests.test_gpu_dispatch import guarded
    n = len(x)
    A, ca = guarded(n)
    B, cb = guarded(n)
    g, cg = guarded(n * m.dim)
    _cabi.call("smcb_logp_grad", m._h, dev.ptr(dev.to_device(x)), n, 0.45, dev.ptr(A), dev.ptr(B), dev.ptr(g),
               dev.stream_ptr())
    ca(), cb(), cg()
    return A.cpu().numpy(), B.cpu().numpy(), g.view(n, m.dim).cpu().numpy()


def _agree(got, ref, tol, what):
    fin = np.isfinite(ref)
    assert np.array_equal(fin, np.isfinite(got)), what
    assert np.array_equal(got[~fin], ref[~fin]), what
    err = np.abs(got[fin] - ref[fin]) / np.maximum(np.abs(ref[fin]), 1.0)
    assert err.max() <= tol, (what, err.max())


@pytest.mark.gpu
def test_plugin_matches_the_host_build_into_guarded_buffers(tmp_path):
    from smcnuts.model.generated import GeneratedModel
    rng = np.random.default_rng(41)
    gp = GeneratedModel((STAN / "gp.stan").read_text(), _gp_data(rng, 20), "gp20")
    ar = GeneratedModel((STAN / "ar1_cov.stan").read_text(), _ar1_data(rng, 5, 8), "ar1")
    n = (1 << 16) + 13
    for m, x in ((gp, np.column_stack([rng.normal(0, 0.5, n), rng.normal(0, 0.5, n), rng.normal(-1, 0.3, n)])),
                 (ar, np.column_stack([rng.normal(0, 0.3, n), rng.uniform(-1.5, 1.5, n), rng.normal(size=(n, 5))]))):
        h = HostModel(m.source, tmp_path / m.name)
        A, B, g = _logp_grad_guarded(m, x)
        rA, rB, rg = h.split(x, 0.45)
        _agree(A, rA, 1e-12, "A")
        ok = np.isfinite(rA)
        _agree(B[ok], rB[ok], 1e-10, "B")
        _agree(g[ok], rg[ok], 1e-8, "grad")
        if m is ar:
            assert np.array_equal(~ok, np.abs(x[:, 1]) >= 1.0)


@pytest.mark.gpu
def test_plugin_generated_quantities_match_the_host_build(tmp_path):
    from smcnuts import _cabi, _device as dev
    from smcnuts.model.generated import GeneratedModel
    from tests.test_gpu_dispatch import guarded
    data, _ = _gq_data(7)
    m = GeneratedModel(GQ, data, "mvngq")
    h = HostGQ(m.source, tmp_path / "gq")
    n = (1 << 18) - 37
    x = np.random.default_rng(2).normal(size=(n, 2))
    out, check = guarded(n * m.gq_dim)
    _cabi.call("smcb_model_generated_quantities", m._h, dev.ptr(dev.to_device(x)), n, 1234, 5, 0, dev.ptr(out),
               dev.stream_ptr())
    check()
    got = out.view(n, m.gq_dim).cpu().numpy()
    ref = h.gq(x, seed=1234, counter=5)
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    fin = ~np.isnan(ref)
    same = np.abs(got[fin] - ref[fin]) <= 1e-12 * np.maximum(np.abs(ref[fin]), 1.0)
    assert same.mean() >= 0.999, same.mean()


def _sampler(m, K, N, seed, step, gq=False):
    from smcnuts.distributions import StdNormal
    from smcnuts.smc_sampler import SMCSampler
    s = SMCSampler(K=K, N=N, target=m, step_size=step, sample_proposal=StdNormal(m.dim), momentum_proposal=StdNormal(m.dim),
                   lkernel="forwardsLKernel", tempering=True, rng=seed, generated_quantities=gq)
    s.sample(show_progress=False)
    assert s.phi[-1] == 1.0
    return s


@pytest.mark.gpu
def test_sampler_posterior_of_a_multivariate_normal_mean():
    from smcnuts.model.generated import GeneratedModel
    K, N = 3, 10
    data = _mvn_data(np.random.default_rng(6), K, N)
    m = GeneratedModel((STAN / "mvn.stan").read_text(), data, "mvn3")
    s = _sampler(m, 20, 1 << 16, 7, 0.2)
    S, S0, y = np.array(data["Sigma"]), np.array(data["Sigma0"]), np.array(data["y"])
    P = np.linalg.inv(S0) + N * np.linalg.inv(S)
    V = np.linalg.inv(P)
    mean_exact = V @ (np.linalg.inv(S) @ y.sum(0))
    mean, var, ess = s.mean_estimate[-1], s.variance_estimate[-1], s.ess[-1]
    assert np.all(np.abs(mean - mean_exact) / np.sqrt(np.diag(V) / ess) < 4), (mean, mean_exact)
    # the ESS counts correlated particles as independent, which understates the error of a variance estimate: relative
    np.testing.assert_allclose(var, np.diag(V), rtol=0.1)


def _gp_quadrature(data):
    """posterior means and variances of (rho, alpha, sigma) of gp.stan on a log-scale grid, batched Cholesky in numpy"""
    x, y = np.array(data["x"]), np.array(data["y"])
    lr, la, ls = (np.linspace(lo, hi, 72) for lo, hi in ((-2.5, 2.5), (-3.0, 2.0), (-3.5, 1.0)))
    R, Al, Sg = (np.exp(v) for v in np.meshgrid(lr, la, ls, indexing="ij"))
    r, a, s = R.ravel(), Al.ravel(), Sg.ravel()
    d2 = (x[:, None] - x[None, :]) ** 2
    Kx = a[:, None, None] ** 2 * np.exp(-d2[None] / (2 * r[:, None, None] ** 2)) + s[:, None, None] ** 2 * np.eye(len(x))
    L = np.linalg.cholesky(Kx)
    z = np.linalg.solve(L, np.broadcast_to(y, (len(r), len(x)))[..., None])[..., 0]
    ll = -np.log(np.diagonal(L, axis1=1, axis2=2)).sum(1) - 0.5 * (z ** 2).sum(1)
    # priors on the constrained scale with the log-scale Jacobian: inv_gamma(5, 5), half normals
    lp = ll - 6 * np.log(r) - 5 / r - 0.5 * a ** 2 - 0.5 * s ** 2 + np.log(r) + np.log(a) + np.log(s)
    w = np.exp(lp - lp.max())
    w /= w.sum()
    th = np.column_stack([r, a, s])
    mean = w @ th
    return mean, w @ (th - mean) ** 2


@pytest.mark.gpu
def test_sampler_gp_hyperparameters_match_quadrature():
    from smcnuts.model.generated import GeneratedModel
    data = _gp_data(np.random.default_rng(10), 10)
    m = GeneratedModel((STAN / "gp.stan").read_text(), data, "gp10")
    s = _sampler(m, 30, 1 << 16, 11, 0.2)
    mean, var, ess = s.mean_estimate[-1], s.variance_estimate[-1], s.ess[-1]
    qm, qv = _gp_quadrature(data)
    # within a tenth of a posterior standard deviation (the ESS of the final particles overstates their independence)
    assert np.all(np.abs(mean - qm) <= 0.1 * np.sqrt(qv)), (mean, qm, ess)
    np.testing.assert_allclose(var, qv, rtol=0.25)


@pytest.mark.gpu
def test_sampler_posterior_predictive_of_a_multivariate_normal():
    from smcnuts.model.generated import GeneratedModel
    K, N = 3, 10
    data = _mvn_data(np.random.default_rng(12), K, N)
    prog = (STAN / "mvn.stan").read_text().replace("parameters {", "transformed data {\n  matrix[K, K] L = "
                                                   "cholesky_decompose(Sigma);\n}\nparameters {")
    prog += "generated quantities {\n  vector[K] y_rep = multi_normal_cholesky_rng(mu, L);\n}\n"
    m = GeneratedModel(prog, data, "mvnppc")
    s = _sampler(m, 20, 1 << 16, 13, 0.2, gq=True)
    w = s.samples.wn.cpu().numpy()
    d = s.gq_draws.cpu().numpy()
    xs = s.samples.x.cpu().numpy()
    mu_mean = w @ xs
    mu_cov = (xs - mu_mean).T @ (w[:, None] * (xs - mu_mean))
    S = np.array(data["Sigma"])
    ess = s.ess[-1]
    pm = s.gq_mean_estimate
    assert np.all(np.abs(pm - mu_mean) <= 4 * np.sqrt(np.diag(S + mu_cov) / ess)), (pm, mu_mean)
    dm = w @ d
    cov = (d - dm).T @ (w[:, None] * (d - dm))
    target = S + mu_cov
    se = np.sqrt((target * target + np.outer(np.diag(target), np.diag(target))) / ess)
    assert np.all(np.abs(cov - target) <= 4 * se), (cov, target)
