"""bench.py -- leapfrog grad-evals/s (and SMC iters/s) of the SMC-NUTS particle hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload arma|PRMwCD|gauss]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

A "step" is one SMC iteration (normalise -> estimate -> ESS -> resample -> NUTS propose -> temper -> reweight,
/root/reference/smcnuts/smc_sampler.py:109-140) over the whole particle set.  Default workload is
BASELINE.json configs[1]: arma, N = 2^20 particles IN TOTAL (sharded over the N GPUs: strong scaling, as the metric
"... at N=2^20 particles, 1/2/4/8 B200" states), forward-proposal L-kernel, fp64.  `--scaling weak` keeps 2^20 particles
per GPU instead.  Prints ONE JSON line.  With more than one rank the warm-up also runs a small sharded case that rank 0
repeats unsharded: `sharded_check` reports whether the leapfrog counts are identical and the largest relative
difference of the estimates.

`value`  : leapfrog gradient evaluations per second over the K timed steps, inputs resident in HBM,
           timed with CUDA events between barriers, max over ranks.
`e2e`    : the same metric through the reference-facing plugin call NUTSProposal.rvs(x_host, r_host, phi) with
           pinned HOST buffers: H2D of x and r, the transition, D2H of x_new and r_new, every step.
`roofline`: the NUTS kernel's algorithmic FP64 FLOPs / its CUDA-event time, against the FP64 FMA peak measured
           live on this GPU by smcb_probe_fp64 (MEASURED_PEAKS.json carries no FP64 figure).
`cpu_baseline`: the oracle's C port of the same NUTS transition on this box's host cores (OpenMP, all cores) on a
           bounded sample of the SAME particle state.
`--impl reference`: the oracle port of the whole SMC iteration (the reference is pure Python + BridgeStan, which is
           not installable offline and cannot travel) on the host cores, bounded particle count, same metric.
`--dump-outputs DIR`: after the timed steps, what the last timed step returned to its caller is written as DIR/<name>.npy
           (rank 0's shard when sharded): the SMC iteration's particles, log-weights and estimates (`smc_*`) and the
           last NUTSProposal.rvs call's results (`e2e_*`; `micro_*` for the micro workload).  As in the reference's
           bookkeeping, smc_x / smc_logw are the particle set AFTER the step's move and reweighting, while
           smc_mean_estimate, smc_variance_estimate, smc_ess and smc_log_likelihood describe the set the step started
           from.  Every array is float64, counters (leapfrogs, resampled) and `sample_rows` included.  All inputs derive
           from fixed seeds, so two builds run with the same arguments can be compared array for array.  At most 64 MB
           in all: when the per-particle arrays are larger, the same seeded sample of rows is taken from each and its
           indices are `sample_rows.npy`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "smc-nuts_b200"))

WORKLOADS = {
    # name: (model, model kwargs, step size, lkernel, tempering, log2 particles per GPU, FLOP per fused value+grad)
    "arma": ("arma", {}, 0.01, "forwardsLKernel", False, 20, 3900.0),
    # PRMwCD: 100 x (22 eta + 24 gradient + 6) = 5.2 kFLOP plus 100 exp; an fp64 exp costs 12 FMA-pipe instructions in
    # the table-driven csrc/common.cuh::fast_exp (libdevice: ~25) = 24 FLOP-slots, so 7.6 kFLOP of FP64-pipe work per
    # evaluation (round-1 lines before the table exp counted 20 instructions per exp = 9.2 kFLOP)
    "PRMwCD": ("PRMwCD", {}, 0.01, "asymptoticLKernel", True, 20, 7600.0),
    "gauss": ("gauss", {"dim": 100}, 0.1, "GaussianApproxLKernel", False, 22, 20200.0),
}


# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the NUTS kernel, from `ncu --set full` captures under
# profiles/ (keyed by workload and particles per GPU); not measured live -> "traffic_live": false in the line
TRAFFIC = {
    ("arma", 1 << 20): (514807552, "ncu --set full capture of round 2 (profiles/r2_nuts_arma_details.csv, tools/r2_final.sh): 125.0 MB read "
                                    "+ 389.8 MB written (algorithmic: 222 MB of particle rows and scalars; the rest is the per-lane tree "
                                    "workspace leaving L2)"),
    ("gauss", 1 << 18): (16656124000, "ncu --set full capture of round 2 (profiles/r2_nuts_gauss100_details.csv): 3.29 GB read + 13.36 GB "
                                       "written at N = 2^18 (algorithmic 0.84 GB: the 10 KB per-lane tree records do not fit in L2)"),
    ("PRMwCD", 1 << 17): (1948797000, "ncu --set full capture of round 2 (profiles/r2_nuts_prm_group_details.csv): 0.18 GB read + 1.76 GB "
                                       "written at N = 2^17"),
}


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled every 100 ms while the timed regions run: through NVML in this process
    (nvidia_ml_py; a query costs microseconds), falling back to one `nvidia-smi` subprocess per sample (the recipe's
    clocks line) -- spawning that five times a second next to the host-driven e2e pipeline perturbed it measurably."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()
        self.nvml = None
        if os.environ.get("SMCB_BENCH_NVIDIA_SMI") != "1":
            try:
                import pynvml
                pynvml.nvmlInit()
                # NVML enumerates all devices: map torch's index through CUDA_VISIBLE_DEVICES when it is a plain index list
                vis = [v.strip() for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip()]
                if vis and index < len(vis) and vis[index].startswith(("GPU-", "MIG-")):
                    self.handle = pynvml.nvmlDeviceGetHandleByUUID(vis[index].encode())
                else:
                    phys = int(vis[index]) if vis and index < len(vis) and vis[index].isdigit() else index
                    self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
                self.nvml = pynvml
            except Exception:
                self.nvml = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        try:
            power = n.nvmlDeviceGetPowerUsage(h) / 1000.0
        except Exception:
            power = float("nan")
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        bits = [n.nvmlClocksThrottleReasonHwSlowdown, n.nvmlClocksThrottleReasonHwThermalSlowdown,
                n.nvmlClocksThrottleReasonSwThermalSlowdown, n.nvmlClocksThrottleReasonSwPowerCap]
        return [str(sm), str(mx), str(power)] + ["Active" if mask & b else "Not Active" for b in bits]

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self.nvml is not None:
                    self.rows.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(float(os.environ.get("SMCB_BENCH_CLOCK_INTERVAL", 0.1 if self.nvml is not None else 0.2)))

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def workload_name(workload, model, n_global, lk, temp, eps, resampling):
    cfg = {"arma": 1, "PRMwCD": 2, "gauss": 3}[workload]
    return (f"{workload}: {model} N={n_global} particles in total, {lk} tempering={temp} eps={eps} resampling={resampling}, "
            f"BASELINE.json configs[{cfg}]")


DUMP_BYTES = 63_000_000    # array data of --dump-outputs: under 64 MB with the .npy headers


def _host(v, rows=None):
    """float64 NumPy copy of a NumPy array, a host or device tensor or a scalar; `rows` selects along the first axis."""
    if hasattr(v, "index_select"):
        import torch
        if rows is not None:
            v = v.index_select(0, torch.as_tensor(rows, device=v.device))
        v = v.cpu().numpy()
    elif rows is not None:
        v = np.asarray(v)[rows]
    return np.asarray(v, dtype=np.float64)


def dump_outputs(out_dir, per_particle, scalars):
    """--dump-outputs: `scalars` (estimates, counters) are written whole; the `per_particle` arrays (one row per particle)
    keep every row if everything fits in DUMP_BYTES, otherwise the same fixed seeded sample of rows each."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    small = {k: _host(v) for k, v in scalars.items()}
    n = len(next(iter(per_particle.values())))
    row_bytes = 8 * sum(int(np.prod(v.shape[1:])) for v in per_particle.values())
    rows = min(n, (DUMP_BYTES - sum(a.nbytes for a in small.values())) // (row_bytes + 8))
    idx = None
    if rows < n:
        idx = np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
        small["sample_rows"] = idx.astype(np.float64)
    for k, v in per_particle.items():
        np.save(out / f"{k}.npy", _host(v, idx))
    for k, a in small.items():
        np.save(out / f"{k}.npy", a)


def run_reference(args):
    """Reference arm: the oracle port of the SMC iteration on the host cores (all threads)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)     # torchrun exports OMP_NUM_THREADS=1 to its workers
    from oracle import smc_oracle as O
    model, kw, eps, lk, temp, log2n, _ = WORKLOADS[args.workload]
    n_full_log2 = args.log2n or log2n
    if args.ref_log2n is not None:
        ref_log2n = args.ref_log2n
    else:
        # the largest power-of-two sample (up to the whole workload) whose W + K iterations fit ~2 minutes on this host:
        # calibrated on two iterations of a small sample
        cal_log2n = 13 if args.workload == "arma" else 9
        cal = O.OracleSMC(2, 1 << cal_log2n, model, eps, lk, temp, seed=10, nthreads=cores, target_kw=kw, save_history=False).init()
        c0 = time.perf_counter()
        cal.step(0); cal.step(1)
        per_particle_step = (time.perf_counter() - c0) / 2 / (1 << cal_log2n)
        ref_log2n = cal_log2n
        while ref_log2n < n_full_log2 and per_particle_step * (1 << (ref_log2n + 1)) * (args.warmup + args.steps) <= 120.0:
            ref_log2n += 1
    n = 1 << ref_log2n
    smc = O.OracleSMC(args.warmup + args.steps, n, model, eps, lk, temp, seed=10, nthreads=cores, target_kw=kw,
                      save_history=False).init()
    for k in range(args.warmup):
        smc.step(k)
    t0 = time.perf_counter()
    for k in range(args.warmup, args.warmup + args.steps):
        smc.step(k)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        k = args.warmup + args.steps - 1
        dump_outputs(args.dump_outputs, {"smc_x": smc.x, "smc_logw": smc.logw},
                     {"smc_mean_estimate": smc.mean_estimate[k], "smc_variance_estimate": smc.variance_estimate[k],
                      "smc_ess": smc.ess[k], "smc_log_likelihood": smc.log_likelihood[k], "smc_phi": smc.phi[k],
                      "smc_leapfrogs": smc.n_leapfrog[k], "smc_resampled": smc.resampled[k]})
    lf = int(smc.n_leapfrog[args.warmup:].sum())
    val = lf / dt
    n_full = 1 << (args.log2n or log2n)
    sample = (f"{n} of the {n_full} particles x {args.steps} SMC iterations, oracle C port of NUTS (OpenMP, {cores} threads) "
              "+ numpy weights/resampling")
    print(json.dumps({
        "impl": "reference", "metric": "leapfrog_grad_evals_per_s", "value": val, "unit": "grad-evals/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "smc_iters_per_s": args.steps / dt,
        "config": {"workload": workload_name(args.workload, model, n_full, lk, temp, eps, "multinomial"),
                   "particles_global": n_full, "particles_timed": n, "dim": smc.D},
        "cpu_baseline": {"value": val, "unit": "grad-evals/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "grad-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference = pure Python + BridgeStan (not installable offline); timed here: its C/numpy oracle port, all host cores",
    }))


def run_micro(args):
    """BASELINE.json configs[4]: weight-update + ESS + systematic resampling microbench, D = 16, 2^25 particles
    per GPU (2^28 over 8 GPUs), sharded with all-to-all-v migration.  HBM-bound: algorithmic bytes per particle are
    SURVEY.md section 8d's: reweight 16D+32, normalise+ESS 24, scan 16, ancestors 12, gather 16D+4."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from smcnuts import _cabi, _device as dev
    from smcnuts.parallel import ShardContext
    from smcnuts.samples.samples import Resampler, normalise
    D = 16
    n = 1 << (args.log2n or 25)
    N = n * world
    sh = ShardContext()
    off = rank * n
    st = dev.stream_ptr()

    def normal(shape_n, d, stream, it):
        out = dev.empty(shape_n, d) if d else dev.empty(shape_n)
        _cabi.call("smcb_normals", 10, it, stream, off, shape_n, d or 1, dev.ptr(out), st)
        return out
    # synthetic inputs (generated outside the timed region): momenta before/after a short move, mild log-weights with a
    # trend across the global index so that rank weight totals differ (ESS ~ 0.3 N; ~1/4 of the rows migrate at P = 8)
    x, r = normal(n, D, 4, 0), normal(n, D, 1, 0)
    r_new = r + 0.05 * normal(n, D, 1, 1)
    lp_x = normal(n, 0, 5, 1)
    lp_xn = lp_x + 0.1 * normal(n, 0, 5, 2)
    gidx = (torch.arange(n, device=x.device, dtype=torch.float64) + off) / N - 0.5
    logw = normal(n, 0, 5, 0) + 1.5 * gidx
    del gidx
    out = dev.empty(n)
    rs = Resampler(N, 10, sh, scheme="systematic")
    rs.keep_idx = False
    rs.use_peer_push = not args.no_peer_push
    names = ["reweight_forward", "lse+normalise", "scan(cdf)", "ancestors+gather+migrate"]
    alg_bytes = [16 * D + 32, 24, 16, 12 + 16 * D + 4]   # SURVEY 8d: 288 + 24 + 16 + (12 + 260) = 600 B at D = 16
    W, K = max(args.warmup, 3), args.steps
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)] for _ in range(K)]

    def step(it, ev=None):
        if ev: ev[0].record()
        _cabi.call("smcb_reweight_forward", dev.ptr(logw), dev.ptr(lp_x), dev.ptr(lp_xn), dev.ptr(r), dev.ptr(r_new), n, D,
                   dev.ptr(out), st)
        if ev: ev[1].record()
        wn, stats, _, scan = normalise(out, sh, scan=True)     # lse + normalise, with the tile sums of the scan fused in
        if ev: ev[2].record()
        cdf = rs._cdf(wn, scan)                                # second pass of the scan
        if ev: ev[3].record()
        rs_x = rs.resample_from_cdf(x, cdf, it)
        if ev: ev[4].record()
        return rs_x, stats

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for it in range(W):
        step(it)
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    l0 = _cabi.lib().smcb_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for it in range(K):
        xs, stats = step(W + it, evs[it])
    e1.record()
    barrier()
    launches = _cabi.lib().smcb_launch_count() - l0
    dt = e0.elapsed_time(e1) * 1e-3
    per = np.array([[ev[i].elapsed_time(ev[i + 1]) * 1e-3 for i in range(len(names))] for ev in evs]).mean(axis=0)
    t = torch.tensor([dt] + list(per), dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt, per = t[0].item(), t[1:].cpu().numpy()
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"micro_resampled_x": xs}, {"micro_log_z": stats[0], "micro_ess": stats[1]})
    peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    if rank == 0:
        ess = float(stats[1].item())
        kern = {nm: {"ms": float(p * 1e3), "alg_bytes_per_particle": b, "achieved_gbs": b * n / p / 1e9, "frac": b * n / p / 1e9 / hbm}
                for nm, p, b in zip(names, per, alg_bytes)}
        total_b = sum(alg_bytes)
        print(json.dumps({
            "metric": "resample_chain_particles_per_s", "value": N * K / dt, "unit": "particles/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"micro: weight-update + ESS + systematic resampling, D={D}, N={n}/GPU (global {N}), "
                                   "BASELINE.json configs[4]", "particles_per_gpu": n, "dim": D, "ess": ess,
                       "l2": f"arrays of {n * D * 8 / 1e9:.1f} GB each, far larger than L2"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": total_b * n / (dt / K) / 1e9, "peak": hbm, "unit": "GB/s",
                         "frac": total_b * n / (dt / K) / 1e9 / hbm, "traffic": None,
                         "alg_bytes_per_particle": total_b,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"},
            "kernels": kern, "clocks": clk,
            "migrated_rows_last_step": rs.last_migrated_rows,
            "migration": "single GPU" if world == 1 else ("NCCL all-to-all-v" if args.no_peer_push else
                                                          "fused: peer stores over NVLink inside the gather kernel"),
        }))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="arma", choices=sorted(WORKLOADS) + ["micro"])
    ap.add_argument("--log2n", type=int, default=None, help="log2 particles PER GPU (default: the workload's)")
    ap.add_argument("--ref-log2n", type=int, default=None, help="particles of the CPU reference arm (default: the largest "
                    "power of two, up to the whole workload, that keeps the run within ~2 minutes on this host)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: the workload's particle count in total over all GPUs (default); weak: per GPU")
    ap.add_argument("--cpu-log2n", type=int, default=18, help="particles of the bounded cpu_baseline sample")
    ap.add_argument("--resampling", default="multinomial", choices=["multinomial", "systematic"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-peer-push", action="store_true", help="micro: migrate with NCCL all-to-all-v instead of the fused peer stores")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.workload == "micro":
        return run_micro(args)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from smcnuts import _cabi, _device as dev
    from smcnuts.distributions import StdNormal
    from smcnuts.model.device_model import make_model
    from smcnuts.proposal.nuts import NUTSProposal
    from smcnuts.smc_sampler import SMCSampler

    model, kw, eps, lk, temp, log2n, flop_per_eval = WORKLOADS[args.workload]
    log2n = args.log2n or log2n
    if args.scaling == "strong":
        N = 1 << log2n
        n_local = N // world
    else:
        n_local = 1 << log2n
        N = n_local * world
    W, K = args.warmup, args.steps
    m = make_model(model, **kw)
    D = m.dim

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- FP64 peak of this GPU (roofline denominator)
    sink = dev.zeros(1)
    pb, pt, pi = 148 * 8, 256, 20000
    peak = 0.0
    for _ in range(3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); _cabi.call("smcb_probe_fp64", pb, pt, pi, dev.ptr(sink), dev.stream_ptr()); b.record()
        torch.cuda.synchronize()
        peak = max(peak, pb * pt * pi * 16 / (a.elapsed_time(b) * 1e-3))

    # ---------------------------------------------------------------- sharded correctness (part of the warm-up)
    sharded_check = None
    if world > 1:
        from smcnuts.parallel import ShardContext

        def small(shard):
            mm = make_model(model, **({"dim": 8} if model == "gauss" else kw))
            s_ = SMCSampler(K=4, N=1 << 14, target=mm, step_size=eps, sample_proposal=StdNormal(mm.dim),
                            momentum_proposal=StdNormal(mm.dim), lkernel=lk, tempering=temp, rng=10,
                            resampling=args.resampling, shard=shard)
            s_.sample(show_progress=False)
            return s_
        sh_run = small(None)
        if rank == 0:
            one = small(ShardContext(enabled=False))
            with np.errstate(all="ignore"):
                rel = max(float(np.max(np.abs(sh_run.mean_estimate - one.mean_estimate) / (np.abs(one.mean_estimate) + 1e-300))),
                          float(np.max(np.abs(sh_run.ess - one.ess) / one.ess)),
                          float(np.max(np.abs(sh_run.log_likelihood - one.log_likelihood) / np.abs(one.log_likelihood))))
            sharded_check = {"case": f"{model} N=16384 K=4 {lk} resampling={args.resampling}, {world} ranks vs 1 GPU (rank 0)",
                             "leapfrogs_equal": bool(np.array_equal(sh_run.leapfrogs, one.leapfrogs)),
                             "resampled_equal": list(sh_run.resampled) == list(one.resampled),
                             "max_rel_err": rel}
            del one
        del sh_run
        barrier()

    # ---------------------------------------------------------------- device-resident run: W warm-up + K timed steps
    smc = SMCSampler(K=W + K, N=N, target=m, step_size=eps, sample_proposal=StdNormal(D), momentum_proposal=StdNormal(D),
                     lkernel=lk, tempering=temp, rng=10, resampling=args.resampling, save_history=(lk == "asymptoticLKernel"))
    smc.begin()
    smc.forward_kernel.record_events = True
    for k in range(W):
        smc.iterate(k)
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = _cabi.lib().smcb_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(W, W + K):
        smc.iterate(k)
    e1.record()
    barrier()
    launches = _cabi.lib().smcb_launch_count() - launches0
    dt = e0.elapsed_time(e1) * 1e-3
    lf_local = smc._lf[W:W + K].clone()
    nuts_dt = sum(a.elapsed_time(b) for a, b in smc.forward_kernel.events[W:W + K]) * 1e-3
    smc.forward_kernel.record_events = False
    t = torch.tensor([dt, nuts_dt], dtype=torch.float64, device="cuda")
    lf_all = lf_local.sum().reshape(1).clone()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lf_all, op=dist.ReduceOp.SUM)
    dt, nuts_dt = t.tolist()
    lf_total = int(lf_all.item())
    value = lf_total / dt
    lf_rank = int(lf_local.sum().item())

    # ---------------------------------------------------------------- e2e: plugin API with pinned host buffers
    fk = NUTSProposal(m, StdNormal(D), eps, rng=10)
    fk.particle0 = rank * n_local
    x_host = smc.samples.x.cpu().pin_memory()
    r_host = torch.empty_like(x_host).pin_memory()
    r_host.copy_(StdNormal(D, seed=11).rvs(n_local, iteration=0, particle0=rank * n_local))
    phi = float(smc.samples.phi_new)
    e2e_lf = 0
    # warm-up of the host path, result read included: the first call allocates the pinned staging buffers and side
    # streams (99 ms), and the first int32 reduction of the step's result loads its kernel lazily (12-21 ms) -- measured
    # per call with SMCB_BENCH_DEBUG=1; W device-resident steps warm neither
    e2e_warmup = max(W, 15)
    for _ in range(e2e_warmup):
        fk.rvs(x_host, r_host, phi)
        int(fk.last["n_leapfrog"].sum().item())   # the result read is part of a step: its reduction kernel is loaded lazily on first use
    barrier()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    t0.record()
    per_call = []
    for _ in range(K):
        c0 = time.perf_counter()
        xn, rn = fk.rvs(x_host, r_host, phi)
        e2e_lf += int(fk.last["n_leapfrog"].sum().item())       # D2H read of the step's result
        per_call.append((time.perf_counter() - c0) * 1e3)
    t1.record()
    if os.environ.get("SMCB_BENCH_DEBUG"):
        print("e2e per-call ms:", [round(t, 2) for t in per_call], file=sys.stderr)
    barrier()
    e2e_dt = max(t0.elapsed_time(t1) * 1e-3, time.perf_counter() - wall0 if world == 1 else 0.0)
    te = torch.tensor([e2e_dt], dtype=torch.float64, device="cuda")
    le = torch.tensor([e2e_lf], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dist.all_reduce(le, op=dist.ReduceOp.SUM)
    e2e_val = le.item() / te.item()
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        k, s = W + K - 1, smc.samples
        dump_outputs(args.dump_outputs,
                     {"smc_x": s.x, "smc_logw": s.logw, "e2e_x_new": xn, "e2e_r_new": rn,
                      "e2e_n_leapfrog": fk.last["n_leapfrog"]},
                     {"smc_mean_estimate": smc._mean_dev[k], "smc_variance_estimate": smc._var_dev[k],
                      "smc_ess": smc.ess[k], "smc_log_likelihood": smc.log_likelihood[k], "smc_phi": smc.phi[k],
                      "smc_leapfrogs": smc._lf[k], "smc_resampled": smc.resampled[k]})

    # ---------------------------------------------------------------- extra key at N > 1: the same iteration, weak scaling
    # (the workload's particle count PER GPU); `value` above stays the strong-scaling number of the stated configuration
    weak = None
    if world > 1 and args.scaling == "strong":
        n_weak = 1 << log2n
        del xn, rn
        smc_w = SMCSampler(K=W + K, N=n_weak * world, target=m, step_size=eps, sample_proposal=StdNormal(D),
                           momentum_proposal=StdNormal(D), lkernel=lk, tempering=temp, rng=10, resampling=args.resampling,
                           save_history=(lk == "asymptoticLKernel"))
        smc_w.begin()
        for k in range(W):
            smc_w.iterate(k)
        barrier()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        for k in range(W, W + K):
            smc_w.iterate(k)
        w1.record()
        barrier()
        tw = torch.tensor([w0.elapsed_time(w1) * 1e-3], dtype=torch.float64, device="cuda")
        lw = smc_w._lf[W:W + K].sum().reshape(1).clone()
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        dist.all_reduce(lw, op=dist.ReduceOp.SUM)
        weak = {"value": lw.item() / tw.item(), "unit": "grad-evals/s", "ms_per_step": tw.item() / K * 1e3,
                "particles_per_gpu": n_weak, "particles_global": n_weak * world,
                "note": "same steps and warm-up, device-timed, max over ranks; divide by n_gpus x the N = 1 value for the "
                        "weak-scaling efficiency"}
        smc_w.samples.resampler.close()
        del smc_w

    # ---------------------------------------------------------------- cpu_baseline (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import smc_oracle as O
        cores = os.cpu_count() or 1
        ns = min(n_local, 1 << args.cpu_log2n)
        t_or = O.COracleTarget(model, **kw)
        xs = x_host[:ns].numpy().copy()
        rs = r_host[:ns].numpy().copy()
        c0 = time.perf_counter()
        ref = t_or.nuts_batch(xs, rs, eps, phi, 10, seed=10, iteration=0, accrej=(lk == "asymptoticLKernel"), nthreads=cores)
        cdt = time.perf_counter() - c0
        cpu = {"value": float(ref["n_leapfrog"].sum()) / cdt, "unit": "grad-evals/s", "cores": cores, "kind": "port",
               "sample": f"one NUTS transition for the first {ns} of the {n_local} particles of the timed state "
                         f"({int(ref['n_leapfrog'].sum())} leapfrogs, {cdt:.2f} s), oracle/smc_oracle.c with OpenMP"}

    if rank == 0:
        evals = lf_rank + K * n_local                      # leapfrogs + the initial evaluation of every transition
        achieved = evals * flop_per_eval / nuts_dt
        extra_roofline = {"frac_vs_nominal_37.2": achieved / 37.2e12}
        if args.workload == "PRMwCD":
            # SURVEY 8d's algorithmic count: 5.2 kFLOP + 100 exp (one special each); the headline `frac` above counts the
            # exp expansion (12 FP64 instructions each) because the FP64 pipe executes it
            extra_roofline.update({"frac_algorithmic": evals * 5200.0 / nuts_dt / peak, "flop_per_eval_algorithmic": 5200.0,
                                   "note": "frac counts 7.6 k FP64-pipe FLOP-slots per evaluation (exp expanded); "
                                           "frac_algorithmic counts 5.2 kFLOP + 100 exp as one each"})
        hist = (K + W + 1) * n_local * (D + 1) * 8 if smc.save_history else 0
        ws_bytes = n_local * 8 * (4 * D + 12)
        line = {
            "metric": "leapfrog_grad_evals_per_s", "value": value, "unit": "grad-evals/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "smc_iters_per_s": K / dt,
            "leapfrogs_per_particle_per_step": lf_total / (K * N),
            "config": {"workload": workload_name(args.workload, model, N, lk, temp, eps, args.resampling),
                       "particles_per_gpu": n_local, "particles_global": N, "dim": D,
                       "l2": f"per-step working set {ws_bytes / 1e6:.0f} MB of particle arrays (> 126 MB L2 from N=2^20, D>=4: "
                             f"x, r, x_new, r_new + 12 per-particle scalars), inputs larger than L2; no explicit flush"},
            "e2e": {"value": e2e_val, "unit": "grad-evals/s", "h2d_bytes_per_step": 2 * n_local * D * 8,
                    "d2h_bytes_per_step": 2 * n_local * D * 8 + 8, "ms_per_step": te.item() / K * 1e3,
                    "api": "smcnuts.proposal.nuts.NUTSProposal.rvs(x_host, r_host, phi) with pinned host tensors",
                    "warmup_calls": e2e_warmup, "median_ms_per_call": float(np.median(per_call)),
                    "max_ms_per_call": float(np.max(per_call))},
            "gpu_launches": int(launches),
            "roofline": {"bound": "fp64", "kernel": "nuts_transition_kernel", "achieved": achieved / 1e12, "peak": peak / 1e12,
                         "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": TRAFFIC.get((args.workload, n_local), (None, None))[0],
                         "traffic_live": False,
                         "traffic_source": TRAFFIC.get((args.workload, n_local), (None, "no ncu capture at this shard size"))[1],
                         "algorithmic_bytes": n_local * 8 * (4 * D + 9) + n_local * 12,
                         "peak_source": "measured live: smcb_probe_fp64 DFMA loop on this GPU (MEASURED_PEAKS.json has no FP64 entry)",
                         "flop_per_eval": flop_per_eval, "evals": evals, "kernel_s": nuts_dt,
                         "kernel_share_of_step": nuts_dt / dt, **extra_roofline},
            "sharded_check": sharded_check,
            "weak": weak,
            "cpu_baseline": cpu,
            "clocks": clk,
            "history_bytes": hist,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
