"""NUTSProposal -- batched iterative NUTS on the GPU behind the reference's proposal plugin API.

Mirrors smcnuts/proposal/nuts.py of the reference: `NUTSProposal(target, momentum_proposal, step_size, rng)`,
`.rvs(x_cond, r_cond, phi) -> (x_prime, r_prime)`, `.logpdf(r)`.  The per-particle Python loop and the
recursive build_tree (nuts.py:50-53,114-150) are one persistent CUDA kernel (csrc/nuts_kernel.cu).
"""

import os

import torch

from .. import _cabi, _device as dev

# Set max tree depth of the NUTS tree (reference: nuts.py:4)
MAX_TREE_DEPTH = 10


def chunk_bounds(n, fractions):
    """Row boundaries [0, ..., n] of consecutive chunks whose sizes are proportional to `fractions` (empty chunks are
    possible for tiny n and are skipped by the caller)."""
    total, acc, bounds = sum(fractions), 0, [0]
    for c, f in enumerate(fractions):
        acc += f
        bounds.append(n if c + 1 == len(fractions) else max(bounds[-1], (acc * n) // total))
    return bounds


class NUTSProposal:
    accept_reject = False

    def __init__(self, target, momentum_proposal, step_size, rng=None, max_tree_depth=MAX_TREE_DEPTH):
        if not hasattr(target, "handle"):
            raise TypeError("the device NUTS proposal needs a device model (smcnuts.model.device_model / "
                            "smcnuts.model.bridgestan.StanModel); Python targets cannot run on the GPU path")
        self.target = target
        self.momentum_proposal = momentum_proposal
        self.step_size = float(step_size)
        self.rng = rng
        self.seed = dev.seed_from_rng(rng)
        self.max_tree_depth = int(max_tree_depth)
        self.iteration = 0        # Philox iteration key; SMCSampler sets it, standalone calls auto-increment
        self.particle0 = 0        # global index of local particle 0 (multi-GPU shards)
        self.last = None          # per-particle by-products of the last transition (device tensors)
        self.record_events = False  # bench.py: CUDA events tightly around the kernel launch
        self.events = []
        self._ws_bytes = {}
        self.want_accept_stat = False   # also emit the per-particle NUTS acceptance statistic (step-size adaptation)

    # Host inputs of at least this many particles go through the pipelined path (copy/compute overlap)
    PIPELINE_MIN_PARTICLES = 1 << 16
    # Chunk sizes as fractions of N: small first and last chunks keep the exposed head (first H2D) and tail (last
    # D2H) short, few large chunks in between keep the per-launch tail cost low (measured: tools/e2e_time.py)
    PIPELINE_FRACTIONS = (1, 2, 3, 2, 1)
    PIPELINE_STREAMS = 4
    # resident CTAs per SM of each chunk's launch (0 = all that fit: the launches then run one after the other).
    # MEASURED (B200, tools/e2e_time.py, N = 2^20 arma): launches side by side on a quarter of every SM each are slower
    # (4.0-4.1 ms against 3.48 ms): the block scheduler does not spread a 148-CTA grid one CTA per SM.
    PIPELINE_BLOCKS_PER_SM = 0

    def rvs(self, x_cond, r_cond, phi: float = 1.0):
        """Propagate particles through one NUTS transition each.  numpy in -> numpy out; CUDA tensors stay put.

        Host inputs (numpy arrays or CPU tensors, the reference's calling convention) are processed in chunks on
        side streams: the H2D copy of chunk c+1 and the D2H copy of chunk c-1 overlap the kernel of chunk c (PCIe is
        full duplex), and the next chunk's CTAs fill the SMs vacated while the previous chunk's last trees finish.
        Philox streams are keyed by the global particle index, so the result does not depend on the chunking."""
        D = self.target.dim
        host_in = dev.is_host(x_cond) or not x_cond.is_cuda
        n = (x_cond.size if dev.is_host(x_cond) else x_cond.numel()) // D if host_in else 0
        scaled = getattr(self.target, "_scale_dev", None) is not None      # diagonal metric: the simple path converts x <-> z
        if host_in and not scaled and n >= self.PIPELINE_MIN_PARTICLES and (dev.is_host(r_cond) or not r_cond.is_cuda):
            out = self._rvs_pipelined(x_cond, r_cond, float(phi), n)
            self.iteration += 1
            return out
        x = dev.to_device(x_cond).reshape(-1, D)
        r = dev.to_device(r_cond).reshape(-1, D)
        out = self.transition(x, r, phi)
        self.iteration += 1
        return dev.to_host_like(out["x_new"], x_cond, "x_new"), dev.to_host_like(out["r_new"], r_cond, "r_new")

    def _rvs_pipelined(self, x_cond, r_cond, phi, N):
        D = self.target.dim
        xh, x_pinned = dev.host_view(x_cond, N, D)
        rh, r_pinned = dev.host_view(r_cond, N, D)
        if not x_pinned:
            x_stage = dev.pinned_buffer("x_in", (N, D), torch.float64)
        if not r_pinned:
            r_stage = dev.pinned_buffer("r_in", (N, D), torch.float64)
        xo_h = dev.pinned_buffer("x_new", (N, D), torch.float64)
        ro_h = dev.pinned_buffer("r_new", (N, D), torch.float64)
        x, r = dev.empty(N, D), dev.empty(N, D)
        o = self._alloc_outputs(N, D, False)
        bounds = chunk_bounds(N, self.PIPELINE_FRACTIONS)
        nchunk = len(bounds) - 1
        nstream = min(self.PIPELINE_STREAMS, nchunk)
        streams = dev.side_streams(nstream)
        need = 0
        for lo, hi in zip(bounds, bounds[1:]):      # the kernel variant (and its scratch) may depend on the chunk size
            if hi > lo:
                nbytes = _cabi._ll()
                _cabi.call("smcb_nuts_workspace_bytes", self.target.handle, hi - lo, self.max_tree_depth, nbytes)
                need = max(need, nbytes.value)
        wss = [dev.workspace(f"nuts_pipe{i}", need) for i in range(nstream)]
        cur = torch.cuda.current_stream()
        ready = torch.cuda.Event()
        ready.record(cur)
        _cabi.call("smcb_nuts_set_blocks_per_sm", int(self.PIPELINE_BLOCKS_PER_SM))
        for c in range(nchunk):
            lo, hi = bounds[c], bounds[c + 1]
            if hi == lo:
                continue
            s = streams[c % nstream]
            if c < nstream:
                s.wait_event(ready)
            if not x_pinned:
                x_stage[lo:hi].copy_(xh[lo:hi])      # pageable -> pinned on the host thread, overlaps earlier chunks
            if not r_pinned:
                r_stage[lo:hi].copy_(rh[lo:hi])
            with torch.cuda.stream(s):
                x[lo:hi].copy_((xh if x_pinned else x_stage)[lo:hi], non_blocking=True)
                r[lo:hi].copy_((rh if r_pinned else r_stage)[lo:hi], non_blocking=True)
                self._launch(x, r, o, lo, hi, phi, self.iteration, None, wss[c % nstream], s.cuda_stream)
                xo_h[lo:hi].copy_(o["x_new"][lo:hi], non_blocking=True)
                ro_h[lo:hi].copy_(o["r_new"][lo:hi], non_blocking=True)
        _cabi.call("smcb_nuts_set_blocks_per_sm", 0)
        for s in streams:
            cur.wait_stream(s)
        cur.synchronize()
        self.last = o
        return dev.host_result(xo_h, x_cond), dev.host_result(ro_h, r_cond)

    def _workspace_bytes(self, N):
        # the kernel variant (and its scratch) also depends on the A/B environment switches of csrc/nuts_kernel.cu
        key = (N, self.max_tree_depth, _cabi.LIB_PATH, os.environ.get("SMCB_PRM_SCALAR"), os.environ.get("SMCB_GAUSS_SCALAR"),
               os.environ.get("SMCB_NUTS_BLOCKS_PER_SM"), getattr(self.target, "_scale_dev", None) is not None)
        b = self._ws_bytes.get(key)
        if b is None:
            nbytes = _cabi._ll()
            _cabi.call("smcb_nuts_workspace_bytes", self.target.handle, N, self.max_tree_depth, nbytes)
            b = self._ws_bytes[key] = nbytes.value
        return b

    def _alloc_outputs(self, N, D, want_grad):
        o = dict(x_new=dev.empty(N, D), r_new=dev.empty(N, D), A_old=dev.empty(N), B_old=dev.empty(N),
                 A_new=dev.empty(N), B_new=dev.empty(N), ke_old=dev.empty(N), ke_new=dev.empty(N),
                 n_leapfrog=dev.empty(N, dtype=torch.int32), accepted=dev.empty(N, dtype=torch.int32),
                 depth=dev.empty(N, dtype=torch.int32))
        if want_grad:
            o["g_new"] = dev.empty(N, D)
        if self.want_accept_stat:
            o["accept_stat"] = dev.empty(N)
        return o

    def _launch(self, x, r, o, lo, hi, phi, it, carry, ws, stream):
        """One kernel launch over particles [lo, hi) of the given arrays (row slices are contiguous)."""
        cA, cB, cg = carry if carry is not None else (None, None, None)
        sl = lambda t: dev.ptr(None if t is None else t[lo:hi])   # noqa: E731
        _cabi.call("smcb_nuts_transition", self.target.handle, sl(x), sl(r), hi - lo, self.step_size, float(phi),
                   self.max_tree_depth, int(self.accept_reject), self.seed, it, self.particle0 + lo,
                   sl(o["x_new"]), sl(o["r_new"]), sl(o["A_old"]), sl(o["B_old"]), sl(o["A_new"]), sl(o["B_new"]),
                   sl(o["ke_old"]), sl(o["ke_new"]), sl(o["n_leapfrog"]), sl(o["accepted"]), sl(o["depth"]),
                   sl(o.get("accept_stat")), sl(cA), sl(cB), sl(cg), sl(o.get("g_new")), dev.ptr(ws), ws.numel(), stream)

    def prepare(self, N, D, want_grad=False):
        """Allocate the next transition's outputs and scratch now.  The sampler calls this before its one host
        synchronisation per iteration (the ESS read): the allocations (a dozen torch.empty calls) then do not sit
        between that synchronisation and the kernel launch, where the GPU would idle through them."""
        want_grad = want_grad and not self.accept_reject
        self._prepared = ((N, D, want_grad, self.want_accept_stat), self._alloc_outputs(N, D, want_grad),
                          dev.workspace("nuts", self._workspace_bytes(N)))

    def transition(self, x, r, phi=1.0, iteration=None, carry=None, want_grad=False):
        """Device entry point: returns dict of device tensors (x_new, r_new, A_old, B_old, A_new, B_new,
        ke_old, ke_new, n_leapfrog, accepted, depth[, g_new]).

        carry = (A, B, g) at `x` (the previous transition's A_new, B_new, g_new at the same phi) skips the initial
        model evaluation of every transition; want_grad=True also returns g_new for the next call."""
        N, D = x.shape
        it = self.iteration if iteration is None else iteration
        if self.accept_reject:
            carry, want_grad = None, False
        scale = getattr(self.target, "_scale_dev", None)
        x_in = x
        if scale is not None:   # diagonal metric: the kernel works on z = x / scale (gradients there are z-space: no carry-over)
            carry, want_grad = None, False
            z = dev.empty(N, D)
            _cabi.call("smcb_scale_rows", dev.ptr(x), N, D, dev.ptr(scale), 1, dev.ptr(z), dev.stream_ptr())
            x = z
        prepared, self._prepared = getattr(self, "_prepared", None), None
        if prepared is not None and prepared[0] == (N, D, want_grad, self.want_accept_stat):
            o, ws = prepared[1], prepared[2]
        else:
            o, ws = self._alloc_outputs(N, D, want_grad), dev.workspace("nuts", self._workspace_bytes(N))
        if self.record_events:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        self._launch(x, r, o, 0, N, phi, it, carry, ws, dev.stream_ptr())
        if self.record_events:
            e1.record()
            self.events.append((e0, e1))
        if scale is not None and self.accept_reject:   # back to x-space, in place; a rejected particle keeps its x row
            _cabi.call("smcb_scale_rows_accepted", dev.ptr(o["x_new"]), dev.ptr(o["accepted"]), dev.ptr(x_in), N, D,
                       dev.ptr(scale), dev.ptr(o["x_new"]), dev.stream_ptr())
        elif scale is not None:                        # back to x-space, in place
            _cabi.call("smcb_scale_rows", dev.ptr(o["x_new"]), N, D, dev.ptr(scale), 0, dev.ptr(o["x_new"]), dev.stream_ptr())
        self.last = o
        return o

    def logpdf(self, r):
        """Log density of the forward kernel, i.e. of the momentum (nuts.py:177-189)."""
        if dev.is_std_normal(self.momentum_proposal, self.target.dim):
            rd = dev.to_device(r).reshape(-1, self.target.dim)
            out = dev.empty(rd.shape[0])
            _cabi.call("smcb_std_normal_logpdf", dev.ptr(rd), rd.shape[0], self.target.dim, dev.ptr(out),
                       dev.stream_ptr())
            return dev.like_input(out, r)
        # foreign momentum plugin (e.g. a scipy frozen distribution): it gets host NumPy, whatever container came in
        return self.momentum_proposal.logpdf(dev.to_numpy(r))
