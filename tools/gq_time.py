"""Cost of generated quantities (fixed inputs).

    python tools/gq_time.py [log2N] [K] [reps]

1. smcb_model_generated_quantities on N = 2^log2N rows of tests/stan/ppc.stan with 100 observations: per particle 100
   y_rep draws (normal_rng), 100 log_lik values, a poisson_rng count and a derived value (G = 202).  Rows/s and bytes/s,
   bytes = N (dim + G) 8 (the rows read and written), over the kernel time from CUDA events.  Four input / output pairs
   are used in turn, so that the working set exceeds the 126 MB L2 of a B200.
2. Its share of one SMC run: SMCSampler(K, N, generated_quantities=True) on the same model, the wall time of the whole
   run against the time of the one generated-quantities evaluation that finish() adds.
The card's name, power limit and SM clock are read in the same run.
"""
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "smc-nuts_b200"))
from smcnuts import _cabi, _device as dev  # noqa: E402
from smcnuts.distributions import StdNormal  # noqa: E402
from smcnuts.model.generated import GeneratedModel  # noqa: E402
from smcnuts.smc_sampler import SMCSampler  # noqa: E402

lg = int(sys.argv[1]) if len(sys.argv) > 1 else 20
K = int(sys.argv[2]) if len(sys.argv) > 2 else 10
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 20
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"device: {smi}")

rng = np.random.default_rng(0)
n_obs = 100
xs = rng.normal(size=n_obs)
data = {"N": n_obs, "x": xs.tolist(), "y": (0.5 + 1.5 * xs + 0.7 * rng.normal(size=n_obs)).tolist()}
m = GeneratedModel((ROOT / "tests" / "stan" / "ppc.stan").read_text(), data, "ppc100")
G, D, N = m.gq_dim, m.dim, 1 << lg
print(f"ppc.stan, {n_obs} observations: dim {D}, gq_dim {G}")
# staging of csrc/nuts_plugin.cuh (GqLayout): ROWS particles of a 64-thread block, S = max(D, G) | 1 doubles a row; the
# CTAs an SM holds by shared memory (228 KB an SM, 1 KB reserved a block on sm_100)
S = max(D, G) | 1
rows = min(64, (200 * 1024 // 8) // S)
smem = 8 * rows * S
print(f"staging: {rows} rows a block, {smem / 1024:.1f} KB shared memory a block, {228 * 1024 // (smem + 1024)} CTAs "
      f"({2 * (228 * 1024 // (smem + 1024))} warps) an SM by shared memory")

xs_d = [dev.to_device(np.column_stack([rng.normal(0.5, 0.1, N), rng.normal(1.5, 0.1, N), rng.normal(-0.4, 0.1, N)]))
        for _ in range(4)]
outs = [dev.empty(N, G) for _ in range(4)]


def gq(i, n=N):
    _cabi.call("smcb_model_generated_quantities", m._h, dev.ptr(xs_d[i % 4]), n, 7, 0, 0, dev.ptr(outs[i % 4]),
               dev.stream_ptr())


for i in range(8):
    gq(i)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for i in range(reps):
    gq(i)
e1.record()
torch.cuda.synchronize()
t = e0.elapsed_time(e1) * 1e-3 / reps
nbytes = N * (D + G) * 8
print(f"gq kernel, N = 2^{lg}: {t * 1e3:.3f} ms/call, {N / t / 1e6:.1f} M rows/s, {nbytes / t / 1e12:.3f} TB/s "
      f"({nbytes / 1e9:.2f} GB a call)")
assert np.isfinite(outs[(reps - 1) % 4][:1000].cpu().numpy()).all()
del xs_d, outs

# one SMC run with generated quantities at the end
s = SMCSampler(K=K, N=N, target=m, step_size=0.05, sample_proposal=StdNormal(D), momentum_proposal=StdNormal(D),
               lkernel="forwardsLKernel", tempering=True, rng=3, generated_quantities=True)
torch.cuda.synchronize()
t0 = time.time()
s.sample(show_progress=False)
torch.cuda.synchronize()
run = time.time() - t0
x_final, t_gq = s.samples.x, []
for _ in range(5):
    torch.cuda.synchronize()
    a = time.time()
    m.generated_quantities(x_final, seed=s.seed)
    torch.cuda.synchronize()
    t_gq.append(time.time() - a)
t_g = float(np.median(t_gq))
print(f"SMC run, K = {K}, N = 2^{lg}: {run:.3f} s wall; generated quantities of the final particles {t_g * 1e3:.3f} ms "
      f"= {100 * t_g / run:.2f} % of the run; leapfrogs {int(s.leapfrogs.sum())}")
print(f"posterior predictive mean of y_rep.1 {s.gq_mean_estimate[0]:.4f}, k_rep {s.gq_mean_estimate[2 * n_obs]:.4f}")
