"""Cost of the matrix functions of generated models (fixed inputs).

    python tools/gp_time.py [log2N] [reps]

1. NUTS grad-evals/s at N = 2^log2N particles of tests/stan/gp.stan (cholesky_decompose, add_diag, gp_exp_quad_cov,
   multi_normal_cholesky_lpdf) with 8, 16 and 32 observations, against the same density with the covariance, its
   Cholesky factor and the forward solve written out in Stan loops (the only form the subset had before).  The
   written-out form keeps two N x N matrices with tangents, past the generator's per-thread budget at 32 observations:
   it is generated with the budget lifted for this comparison only.
2. For each build: registers, stack frame and spills of the plug-in's NUTS kernel (ptxas -v) and the nvcc wall time.
3. multi_normal_lpdf with a data covariance (factored when the model is generated) against the same density with the
   factor computed in the model block in every evaluation (K = 16, 20 observations).
The card's name, power limit and maximum SM clock are read in the same run.
"""
import re
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "smc-nuts_b200"))
from smcnuts.distributions import StdNormal  # noqa: E402
from smcnuts.model import generated, stan_codegen  # noqa: E402
from smcnuts.model.generated import GeneratedModel  # noqa: E402
from smcnuts.proposal.nuts import NUTSProposal  # noqa: E402

BY_HAND = """
data { int<lower=1> N; array[N] real x; vector[N] y; real phi; }
parameters { real<lower=0> rho; real<lower=0> alpha; real<lower=0> sigma; }
model {
  matrix[N, N] K;
  matrix[N, N] L;
  vector[N] z;
  real ld = 0;
  real q = 0;
  for (i in 1:N)
    for (j in 1:N)
      K[i, j] = square(alpha) * exp(-0.5 * square(x[i] - x[j]) / square(rho));
  for (n in 1:N) K[n, n] += square(sigma);
  for (j in 1:N) {
    real s = K[j, j];
    for (k in 1:(j - 1)) s -= square(L[j, k]);
    L[j, j] = sqrt(s);
    for (i in (j + 1):N) {
      real t = K[i, j];
      for (k in 1:(j - 1)) t -= L[i, k] * L[j, k];
      L[i, j] = t / L[j, j];
    }
  }
  for (i in 1:N) {
    real t = y[i];
    for (j in 1:(i - 1)) t -= L[i, j] * z[j];
    z[i] = t / L[i, i];
    ld += log(L[i, i]);
    q += square(z[i]);
  }
  rho ~ inv_gamma(5, 5);
  alpha ~ std_normal();
  sigma ~ std_normal();
  target += phi * (-0.9189385332046727 * N - ld - 0.5 * q);
}
"""

MVN_IN_MODEL = """
data { int<lower=1> K; int<lower=1> N; array[N] vector[K] y; matrix[K, K] Sigma; vector[K] mu0; matrix[K, K] Sigma0;
       real phi; }
parameters { vector[K] mu; }
model {
  matrix[K, K] L = cholesky_decompose(Sigma);
  mu ~ multi_normal(mu0, Sigma0);
  target += phi * multi_normal_cholesky_lpdf(y | mu, L);
}
"""

lg = int(sys.argv[1]) if len(sys.argv) > 1 else 18
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"device: {smi}", flush=True)


def ptxas(src):
    """nvcc wall time and ptxas' registers / stack frame / spills of the NUTS kernel of the plug-in of `src`"""
    work = Path(tempfile.mkdtemp(prefix="gp_time."))
    try:
        (work / "model_gen.cuh").write_text(src.text)
        (work / "model_gq.cuh").write_text(src.gq_text)
        (work / "plugin.cu").write_text(f'#define SMCB_PLUGIN_TU 1\n#include "nuts_plugin.cuh"\n#include "model_gen.cuh"\n'
                                        f'#include "model_gq.cuh"\nSMCB_DEFINE_PLUGIN({src.struct_name})\n'
                                        f'SMCB_DEFINE_PLUGIN_GQ({src.struct_name}GQ)\n')
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        t0 = time.time()
        r = subprocess.run([nvcc, *generated.NVCC_FLAGS, "-Xptxas", "-v", f"-I{generated.CSRC}", f"-I{work}",
                            str(work / "plugin.cu"), "-o", str(work / "model.so")], capture_output=True, text=True)
        wall = time.time() - t0
        if r.returncode:
            raise RuntimeError(r.stderr)
        lines = r.stderr.splitlines()
        for i, ln in enumerate(lines):
            if "Compiling entry function" in ln and "nuts" in ln.lower():
                info = " ".join(lines[i + 1:i + 4])
                regs = re.search(r"Used (\d+) registers", info)
                stack = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores", info)
                return wall, int(regs.group(1)), int(stack.group(1)), int(stack.group(2))
        raise RuntimeError("no NUTS kernel in the ptxas output")
    finally:
        shutil.rmtree(work, ignore_errors=True)


def rate(m, x0, step):
    D = m.dim
    k = NUTSProposal(m, StdNormal(D), step, rng=10)
    x = x0
    for it in range(2):
        x = k.transition(x, StdNormal(D, seed=10).rvs(x0.shape[0], iteration=it), 1.0, iteration=it)["x_new"]
    r = StdNormal(D, seed=10).rvs(x0.shape[0], iteration=2)
    ts, nl = [], 0
    for _ in range(reps):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); o = k.transition(x, r, 1.0, iteration=2); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
        nl = int(o["n_leapfrog"].sum().item())
    t = min(ts)
    return t, nl / t / 1e6, nl / x0.shape[0]


def report(label, src, m, x0, step):
    wall, regs, stack, spill = ptxas(src)
    frame_gb = stack * 148 * 2048 / 1e9
    t, g, mean_l = rate(m, x0, step)
    print(f"{label:34s} N=2^{lg}: {t:9.2f} ms {g:8.4f} G grad-evals/s (mean {mean_l:5.1f} leapfrogs) | NUTS kernel "
          f"{regs} registers, {stack} B stack frame ({frame_gb:.1f} GB at 148 x 2048 threads), {spill} B spill stores | "
          f"nvcc {wall:.0f} s", flush=True)
    return t


N = 1 << lg
rng = np.random.default_rng(0)
for n_obs in (8, 16, 32):
    x = np.sort(rng.uniform(-3, 3, n_obs))
    data = {"N": n_obs, "x": x.tolist(), "y": (np.sin(x) + 0.3 * rng.normal(size=n_obs)).tolist()}
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    x0 = torch.randn(N, 3, dtype=torch.float64, device="cuda", generator=g) * 0.2
    x0[:, 2] -= 1.0
    gp = GeneratedModel((ROOT / "tests/stan/gp.stan").read_text(), data, f"gp{n_obs}")
    saved = stan_codegen._Gen.MAX_MATRIX_BYTES
    stan_codegen._Gen.MAX_MATRIX_BYTES = 1 << 30
    try:
        hand = GeneratedModel(BY_HAND, data, f"gp{n_obs}_hand")
    finally:
        stan_codegen._Gen.MAX_MATRIX_BYTES = saved
    lp = [float(mm.logpdf(x0[:4096], 1.0).sub(gp.logpdf(x0[:4096], 1.0)).abs().max()) for mm in (hand,)]
    print(f"gp.stan, {n_obs} observations (max |logp difference| of the two forms {lp[0]:.1e})", flush=True)
    report("  matrix functions", gp.source, gp, x0, 0.1)
    report("  written out in Stan loops", hand.source, hand, x0, 0.1)

K, n_obs = 16, 20
Q = rng.normal(size=(K, K))
Sigma = Q @ Q.T / K + 0.5 * np.eye(K)
data = {"K": K, "N": n_obs, "y": rng.multivariate_normal(np.zeros(K), Sigma, size=n_obs).tolist(), "Sigma": Sigma.tolist(),
        "mu0": np.zeros(K).tolist(), "Sigma0": (2 * np.eye(K)).tolist()}
g = torch.Generator(device="cuda"); g.manual_seed(2)
x0 = torch.randn(N, K, dtype=torch.float64, device="cuda", generator=g) * 0.2
folded = GeneratedModel((ROOT / "tests/stan/mvn.stan").read_text(), data, "mvn16")
inmodel = GeneratedModel(MVN_IN_MODEL, data, "mvn16_model")
d = float(folded.logpdf(x0[:4096], 1.0).sub(inmodel.logpdf(x0[:4096], 1.0)).abs().max())
print(f"multi_normal, K = {K}, {n_obs} observations (max |logp difference| {d:.1e})", flush=True)
report("  data covariance factored once", folded.source, folded, x0, 0.1)
report("  factored in the model block", inmodel.source, inmodel, x0, 0.1)
