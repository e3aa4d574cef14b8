"""Cost of the constrained vector parameter types of generated models (fixed inputs).

    python tools/constrained_time.py [log2N_nuts] [log2N_constrain] [reps]

1. NUTS grad-evals/s of the K-component normal mixture (tests/stan/mixture.stan: simplex[K] weights, ordered[K] means)
   against the same density written with unconstrained parameters and the stick-breaking / cumulative-exp transforms and
   their log-Jacobians spelled out in `transformed parameters` (every transformed value then carries sensitivities for all
   earlier coordinates: K^2 doubles a thread, where the built-in types pull the gradient back in O(K)).
2. smcb_model_constrain at N rows for CDIM = 3 and 16 (simplex[CDIM]): bytes moved (N (dim + CDIM) 8) over kernel time.
   Four input / output pairs are used in turn, so that the working set exceeds the 126 MB L2 of a B200.
"""
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "smc-nuts_b200"))
from smcnuts import _cabi, _device as dev  # noqa: E402
from smcnuts.distributions import StdNormal  # noqa: E402
from smcnuts.model.generated import GeneratedModel  # noqa: E402
from smcnuts.proposal.nuts import NUTSProposal  # noqa: E402

BY_HAND = """
data { int<lower=1> K; int<lower=1> N; array[N] real y; real phi; }
parameters { vector[K - 1] ys; vector[K] yo; }
transformed parameters {
  vector[K] theta;
  vector[K] mu;
  {
    real r = 1;
    for (k in 1:(K - 1)) {
      theta[k] = r * inv_logit(ys[k] - log(K - k));
      r = r * inv_logit(log(K - k) - ys[k]);
    }
    theta[K] = r;
  }
  mu[1] = yo[1];
  for (k in 2:K) mu[k] = mu[k - 1] + exp(yo[k]);
}
model {
  for (k in 1:(K - 1))
    target += -log1p_exp(log(K - k) - ys[k]) - (K - k) * log1p_exp(ys[k] - log(K - k));
  for (k in 2:K) target += yo[k];
  mu ~ normal(0, 10);
  for (n in 1:N) {
    vector[K] lps = log(theta);
    for (k in 1:K)
      lps[k] += normal_lpdf(y[n] | mu[k], 1);
    target += phi * log_sum_exp(lps);
  }
}
"""

lg = int(sys.argv[1]) if len(sys.argv) > 1 else 18
lgc = int(sys.argv[2]) if len(sys.argv) > 2 else 20
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 2
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"device: {smi}", flush=True)


def timed(fn, n):
    fn()
    ts = []
    for _ in range(n):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); out = fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return min(ts), out


N = 1 << lg
rng = np.random.default_rng(0)
for K in (3, 16):
    n_obs = 100
    y = (rng.choice(np.linspace(-4, 4, K), n_obs) + rng.normal(size=n_obs)).tolist()
    data = {"K": K, "N": n_obs, "y": y}
    models = [("simplex / ordered types", GeneratedModel((ROOT / "tests/stan/mixture.stan").read_text(), data, f"mix{K}")),
              ("transforms by hand", GeneratedModel(BY_HAND, data, f"mix{K}_hand"))]
    D = models[0][1].dim
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    x0 = torch.randn(N, D, dtype=torch.float64, device="cuda", generator=g) * 0.3
    x0[:, K - 1] -= 2.0                   # the first mean; the others follow at exp(~0) spacing
    lp = [m.logpdf(x0[:4096], 1.0) for _, m in models]
    dlp = float((lp[0] - lp[1]).abs().max() / lp[0].abs().max())
    for name, m in models:
        k = NUTSProposal(m, StdNormal(D), 0.02, rng=10)
        x = x0
        for it in range(2):
            x = k.transition(x, StdNormal(D, seed=10).rvs(N, iteration=it), 1.0, iteration=it)["x_new"]
        r = StdNormal(D, seed=10).rvs(N, iteration=2)
        t, o = timed(lambda: k.transition(x, r, 1.0, iteration=2), reps)
        nl = int(o["n_leapfrog"].sum().item())
        print(f"mixture K={K:2d} {name:26s} N=2^{lg}: {t:9.3f} ms  {nl / t / 1e6:7.3f} G grad-evals/s "
              f"(mean {nl / N:.1f} leapfrogs; max rel. logp difference of the two phrasings {dlp:.1e})", flush=True)

NC = 1 << lgc
for C in (3, 16):
    m = GeneratedModel(f"parameters {{ simplex[{C}] s; }} model {{ s ~ dirichlet(rep_vector(2, {C})); }}", {}, f"simplex{C}")
    xs = [torch.randn(NC, m.dim, dtype=torch.float64, device="cuda") for _ in range(4)]
    outs = [torch.empty(NC, C, dtype=torch.float64, device="cuda") for _ in range(4)]
    it = [0]

    def run():
        i = it[0] % 4
        it[0] += 1
        _cabi.call("smcb_model_constrain", m._h, dev.ptr(xs[i]), NC, dev.ptr(outs[i]), dev.stream_ptr())
        return outs[i]
    for _ in range(4):
        run()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_launch = 200
    a.record()
    for _ in range(n_launch):
        run()
    b.record(); torch.cuda.synchronize()
    t = a.elapsed_time(b) / n_launch
    nbytes = NC * (m.dim + C) * 8
    print(f"smcb_model_constrain CDIM={C:2d} dim={m.dim:2d} N=2^{lgc}: {t * 1e3:8.1f} us  {nbytes / t / 1e9:6.2f} TB/s "
          f"({100 * nbytes / t / 1e9 / 7.7:.0f} % of the 7.7 TB/s data-sheet HBM bandwidth)", flush=True)
