"""GPU (B200): every code path the particle kernels dispatch on -- dimension, particle count, 16-byte alignment --
against a plain extended-precision reference of the same operation.

The shipped workloads run only a few of these paths (arma, PRMwCD, gauss at D = 8 / 100); this file runs the others.
Tolerances are forward error bounds in u = 2^-53 (e.g. |B - B_ref| <= c (D + 2) u |x|'|P||x| / 2), so that a dropped
or permuted term fails where a flat rtol would not.  Outputs are written into guarded buffers: a band of
signalling-NaN bit patterns after (and, for offset views, before) the elements a kernel may write, checked bit for
bit afterwards, so an overrun fails an assertion inside the test's own allocation instead of corrupting a neighbour.
"""
import math

import numpy as np
import pytest
import torch
from scipy.special import logsumexp

from oracle import philox
from oracle import smc_oracle as O
from smcnuts import _cabi

if torch.cuda.is_available():
    from smcnuts import _device as dev
    from smcnuts.distributions import StdNormal
    from smcnuts.lkernel.gaussian_lkernel import GaussianApproxLKernel
    from smcnuts.model.device_model import make_model
    from smcnuts.parallel import ShardContext
    from smcnuts.proposal.nuts import NUTSProposal
    from smcnuts.samples.samples import normalise

U = 2.0 ** -53
LD = np.longdouble


# ------------------------------------------------------------------------------------------------ helpers
def dense_spd(D, seed):
    """Q diag(lambda) Q' with a random orthogonal Q and lambda log-uniform in [1/4, 4], exactly symmetric: every
    entry nonzero and distinct (the AR(1) precision of the default gauss model is tridiagonal)."""
    rng = np.random.default_rng(seed)
    Q, R = np.linalg.qr(rng.normal(size=(D, D)))
    Q *= np.sign(np.diag(R))
    lam = np.exp(rng.uniform(math.log(0.25), math.log(4.0), D))
    P = (Q * lam) @ Q.T
    return 0.5 * (P + P.T)


_SENTINEL = {torch.float64: (torch.int64, 0x7FF0000000000001),   # signalling NaN
             torch.int64: (torch.int64, 0x7FF0000000000001),
             torch.int32: (torch.int32, 0x7F800001)}
GUARD = 4096


def guarded(n, dtype=torch.float64, off=0):
    """n elements (after `off` guard elements) followed by GUARD more, all set to a signalling-NaN bit pattern.
    Returns (view of the n elements, check) where check() asserts that nothing outside the view changed."""
    ity, pat = _SENTINEL[dtype]
    buf = torch.empty(off + n + GUARD, dtype=dtype, device=dev.device())
    bits = buf.view(ity)
    bits.fill_(pat)

    def check():
        torch.cuda.synchronize()
        b = bits.cpu()
        assert bool((b[:off] == pat).all()), "write before the start of the buffer"
        bad = (b[off + n:] != pat).nonzero().flatten()
        assert bad.numel() == 0, f"{bad.numel()} guard elements overwritten past element {n} (first at +{int(bad[0])})"
    return buf[off:off + n], check


def placed(a, off=0, dtype=torch.float64):
    """A device copy of `a` that starts `off` elements into its allocation: off = 1 gives an 8-byte-misaligned
    pointer, which drives the unaligned fallbacks."""
    a = np.ascontiguousarray(a)
    buf = torch.empty(off + a.size, dtype=dtype, device=dev.device())
    v = buf[off:]
    v.copy_(torch.from_numpy(a.ravel()).to(dtype))
    return v.view(a.shape)


def st():
    return dev.stream_ptr()


def assert_within(got, want, bound, what):
    got = np.asarray(got, dtype=np.float64)
    err = np.abs(got.astype(LD) - want)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} outside the bound; worst err/bound "
                           f"{float(np.max(err[bad] / np.maximum(bound[bad] if np.ndim(bound) else bound, 1e-300)))}")


def dyadic_weights(p, total_log2=30, seed=0):
    """Weights k_i / 2^m with integer k_i summing to 2^m: every partial sum is exact, so the device scan equals
    np.cumsum bit for bit and ancestors are decided by the search alone."""
    rng = np.random.default_rng(seed)
    k = rng.multinomial(1 << total_log2, p / p.sum()).astype(np.float64)
    return k / float(1 << total_log2)


# ------------------------------------------------------------------------------------------------ 1. Gaussian NUTS
NUTS_DIMS = [1, 2, 3, 7, 8, 9, 16, 17, 31, 32, 33, 63, 64, 65, 100, 103, 104, 105, 113, 114, 127, 128]


def _ld_gauss(P, X, phi):
    """-x'Px/2 and -phi P x in long double, with the magnitudes |x|'|P||x|/2 and phi |P||x| of the error bounds."""
    Pl, Xl = P.astype(LD), X.astype(LD)
    Px = Xl @ Pl.T
    aPx = np.abs(Xl) @ np.abs(Pl).T
    return (-0.5 * np.einsum("nd,nd->n", Xl, Px), -LD(phi) * Px, 0.5 * np.einsum("nd,nd->n", np.abs(Xl), aPx),
            LD(phi) * aPx)


def _nuts_inputs(P, N, seed):
    rng = np.random.default_rng(seed)
    D = len(P)
    C = np.linalg.cholesky(np.linalg.inv(P))
    x = rng.normal(size=(N, D)) @ C.T
    r = rng.normal(size=(N, D))
    eps = 0.25 * 0.5   # a quarter of the smallest posterior sd (eigenvalues of P are <= 4)
    return x, r, eps


def _check_model_values(P, X, A, B, g, phi, what):
    D = len(P)
    Bref, gref, qabs, gabs = _ld_gauss(P, X, phi)
    assert np.all(A == 0.0), what
    assert_within(B, Bref, 2 * (D + 2) * U * qabs, f"{what} B")
    if g is not None:
        assert_within(g, gref, (D + 2) * U * gabs, f"{what} grad")


@pytest.mark.gpu
@pytest.mark.parametrize("D", NUTS_DIMS)
def test_gauss_nuts_model_values_and_trees(D, monkeypatch):
    """One NUTS transition with a dense precision on the kernel D selects (GaussModelG<NT8> for NT8 = 1/2/4/8/13 up to
    D = 104, the plain GaussModel above): the model values the kernel emits (A, B at x and x_new, the gradient at x_new)
    against long double, the trees against the recursive C oracle, and the tensor-core kernel against the
    one-lane-per-particle kernel (SMCB_GAUSS_SCALAR=1)."""
    P = dense_spd(D, 1000 + D)
    m, t = make_model("gauss", precision=P), O.COracleTarget("gauss", precision=P)
    N = 2000 if D <= 32 else 1000
    x, r, eps = _nuts_inputs(P, N, D)
    phi, seed, it, p0 = 0.7, 5, 2, 1 << 33
    outs = {}
    for mode in (("0", "1") if D <= 104 else ("0",)):
        monkeypatch.setenv("SMCB_GAUSS_SCALAR", mode)
        k = NUTSProposal(m, StdNormal(D), eps, rng=seed, max_tree_depth=6)
        k.particle0 = p0
        o = k.transition(dev.to_device(x), dev.to_device(r), phi, iteration=it, want_grad=True)
        outs[mode] = o = {kk: v.cpu().numpy() for kk, v in o.items()}
        _check_model_values(P, x, o["A_old"], o["B_old"], None, phi, f"D={D} mode={mode} at x")
        _check_model_values(P, o["x_new"], o["A_new"], o["B_new"], o["g_new"], phi, f"D={D} mode={mode} at x_new")
    o = outs["0"]
    ref = t.nuts_batch(x, r, eps, phi, 6, seed=seed, iteration=it, particle0=p0, nthreads=8)
    same = o["n_leapfrog"] == ref["n_leapfrog"]
    assert same.mean() >= 0.995, same.mean()
    assert np.array_equal(o["depth"][same], ref["depth"][same])
    row_ok = np.all(np.isclose(o["x_new"][same], ref["x_new"][same], rtol=1e-6, atol=1e-8), axis=1) & \
        np.all(np.isclose(o["r_new"][same], ref["r_new"][same], rtol=1e-6, atol=1e-7), axis=1) & \
        np.isclose(o["A_new"][same] + phi * o["B_new"][same], ref["lp_new"][same], rtol=1e-8, atol=1e-6)
    assert row_ok.mean() >= 0.9995, row_ok.mean()
    np.testing.assert_allclose(o["ke_old"], 0.5 * np.sum(r * r, axis=1), rtol=1e-13)
    if "1" in outs:
        a, b = outs["1"], outs["0"]
        same = a["n_leapfrog"] == b["n_leapfrog"]
        assert same.mean() >= 0.995, same.mean()
        assert np.array_equal(a["depth"][same], b["depth"][same])
        row_ok = np.all(np.isclose(a["x_new"][same], b["x_new"][same], rtol=1e-6, atol=1e-8), axis=1)
        assert row_ok.mean() >= 0.9995, row_ok.mean()


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 127, 128])
def test_gauss_plain_model_logpdf_and_grad(D):
    """logpdf / logpdfgrad run the plain GaussModel (smcb_logp_grad) at every D."""
    P = dense_spd(D, 2000 + D)
    m = make_model("gauss", precision=P)
    X = np.random.default_rng(D).normal(size=(3001, D))
    for phi in (1.0, 0.37):
        Bref, gref, qabs, gabs = _ld_gauss(P, X, phi)
        assert_within(m.logpdf(X, phi), LD(phi) * Bref, phi * 2 * (D + 2) * U * qabs + U * np.abs(phi * Bref),
                      f"D={D} logpdf")
        assert_within(m.logpdfgrad(X, phi), gref, (D + 2) * U * gabs, f"D={D} logpdfgrad")


@pytest.mark.gpu
def test_gauss_model_symmetrises_the_precision():
    """A precision that is not exactly symmetric (here straight out of np.linalg.inv) is used as (P + P')/2, the matrix
    of the oracle: both kernels then return the gradient of their own B."""
    D = 20
    Ps = dense_spd(D, 7)
    K = np.random.default_rng(1).normal(size=(D, D)) * 1e-6
    P = Ps + (K - K.T)          # same B = -x'Px/2, but -Px and -P'x are not its gradient
    m = make_model("gauss", precision=P)
    X = np.random.default_rng(0).normal(size=(500, D))
    Bref, gref, qabs, gabs = _ld_gauss(Ps, X, 1.0)
    assert_within(m.logpdfgrad(X, 1.0), gref, (D + 2) * U * gabs, "plain kernel grad")
    x, r, eps = _nuts_inputs(Ps, 256, 1)
    o = NUTSProposal(m, StdNormal(D), eps, rng=1, max_tree_depth=4).transition(dev.to_device(x), dev.to_device(r), 1.0,
                                                                                iteration=0, want_grad=True)
    o = {k: v.cpu().numpy() for k, v in o.items()}
    _check_model_values(Ps, o["x_new"], o["A_new"], o["B_new"], o["g_new"], 1.0, "tensor-core kernel")


# ------------------------------------------------------------------------------------------------ 2. Gaussian L-kernel
LK_DIMS = sorted(set(NUTS_DIMS) | set(range(60, 71)) | set(range(100, 129)))


class _Dim:
    def __init__(self, D):
        self.dim = D


def _lk_data(D, N, seed):
    rng = np.random.default_rng(seed)
    A = np.eye(D) + 0.3 * rng.normal(size=(D, D)) / math.sqrt(D)
    x_new = rng.normal(size=(N, D)) @ A
    r_new = 0.5 * rng.normal(size=(N, D)) - 0.2 * x_new
    return r_new, x_new


def _nt8_kk(D):
    nt8 = next(k for k, hi in ((1, 8), (2, 16), (4, 32), (8, 64), (13, 104)) if D <= hi)
    return nt8, (2 * D + 3) // 4


def test_gaussL_scratch_query_covers_the_packed_fragments():
    """CPU: the tensor-core logpdf packs NT8 * KK * 32 doubles of G' into the caller's scratch (D <= 104); the size
    query the host code allocates from must cover that for every D.  The earlier fixed size, 2 D (D + 8) + 4096
    doubles, was 142 doubles short at D = 65."""
    L = _cabi.lib()
    for D in range(1, 105):
        nt8, kk = _nt8_kk(D)
        assert L.smcb_gaussL_logpdf_scratch_bytes(D) >= 8 * nt8 * kk * 32, D
    for D in range(105, 129):
        assert L.smcb_gaussL_logpdf_scratch_bytes(D) >= 0


@pytest.mark.gpu
@pytest.mark.parametrize("D", LK_DIMS)
def test_gaussian_lkernel_values_at_every_dispatch(D):
    """Gram on FP64 tensor cores for D <= 104 and in 64 x 64 scalar tiles above; logpdf on tensor cores (NT8 = 1 .. 13)
    for D <= 104, scalar with G in shared memory up to D = 113 and in global memory above."""
    N = 4 * D + 37
    r_new, x_new = _lk_data(D, N, D)
    lk = GaussianApproxLKernel(_Dim(D), N)
    L = lk.calculate_L(r_new, x_new)
    assert lk.last_status.cpu().numpy()[1] == 0.0
    np.testing.assert_allclose(L, O.gaussian_lkernel(r_new, x_new), rtol=1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize("D,N", [(105, 60), (106, 61)])
def test_gaussian_lkernel_pinv_path_above_the_tensor_core_range(D, N):
    """N <= D: C_xx is singular and the factorisation takes the one-CTA Jacobi pseudo-inverse; at odd D its
    round-robin pairing has a bye every round."""
    rng = np.random.default_rng(D)
    x_new, r_new = rng.normal(size=(N, D)), rng.normal(size=(N, D))
    lk = GaussianApproxLKernel(_Dim(D), N)
    L = lk.calculate_L(r_new, x_new)
    assert np.all(np.isfinite(L))
    assert lk.last_status.cpu().numpy()[1] == 1.0
    np.testing.assert_allclose(L, O.gaussian_lkernel(r_new, x_new), rtol=1e-6, atol=1e-6)


def _host_frag_doubles(D):
    """The scratch the host code (GaussianApproxLKernel.calculate_L) allocates for smcb_gaussL_logpdf."""
    return _cabi.lib().smcb_gaussL_logpdf_scratch_bytes(D) // 8


@pytest.mark.gpu
def test_gaussian_lkernel_writes_stay_inside_their_buffers():
    """Factor and logpdf at every D in 1..128 with guarded outputs and scratch of exactly the size the host code
    allocates.  Regression: at D = 65 the fragment packing wrote 13 728 doubles into a 13 586-double scratch."""
    bad = []
    for D in range(1, 129):
        N = 2 * D + 37
        r_new, x_new = _lk_data(D, N, 3 * D)
        X = np.hstack([-r_new, x_new])
        mean = X.mean(axis=0)
        Xc = X - mean
        r, x, md, gram = (dev.to_device(a) for a in (r_new, x_new, mean, Xc.T @ Xc))
        G, cG = guarded(D * 2 * D)
        logdet, cL = guarded(2)
        scratch, cS = guarded(6 * D * D)
        out, cO = guarded(N)
        nf = _host_frag_doubles(D)
        frag, cF = guarded(nf) if nf else (None, lambda: None)
        _cabi.call("smcb_gaussL_factor", dev.ptr(gram), N, D, GaussianApproxLKernel.RIDGE, dev.ptr(G), dev.ptr(logdet),
                   dev.ptr(scratch), st())
        _cabi.call("smcb_gaussL_logpdf", dev.ptr(r), dev.ptr(x), N, D, dev.ptr(md), dev.ptr(G), dev.ptr(logdet),
                   dev.ptr(out), dev.ptr(frag), st())
        for name, chk in (("G", cG), ("logdet", cL), ("factor scratch", cS), ("out", cO), ("logpdf scratch", cF)):
            try:
                chk()
            except AssertionError as e:
                bad.append((D, name, str(e)))
        if not any(b[0] == D for b in bad) and \
                not np.allclose(out.cpu().numpy(), O.gaussian_lkernel(r_new, x_new), rtol=1e-9, atol=0):
            bad.append((D, "values", "logpdf differs from the oracle"))
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ 3. weight kernels
W_DIMS = [1, 2, 3, 4, 5, 8, 16, 23, 24, 25, 32, 64, 65, 110, 111, 128, 200]
W_SIZES = [1, 2, 3, 4, 5, 31, 33, 255, 256, 257, 4097, 100_003]
C2PI = 0.5 * np.log(LD(2) * LD(np.pi))


def _mapped(lp):
    return np.where(np.isfinite(lp), lp, -np.inf)


@pytest.mark.gpu
@pytest.mark.parametrize("D", W_DIMS)
def test_weight_kernels_every_shape_and_alignment(D):
    """Row norms, init_logw and the reweight family: coop kernel (aligned D in {4, 8, 16, 32, 64}), shared-memory tile
    (D <= 110; above 48 KB of shared memory from D = 24), one warp per row (D >= 111), unaligned fallback (off = 1)."""
    rng = np.random.default_rng(D)
    for N in W_SIZES:
        r, rn = rng.normal(size=(2, N, D))
        logw, lpx, lpn, L, q = rng.normal(size=(5, N)) * 30.0
        ke0, ke1 = rng.exponential(size=(2, N)) * D
        A0, B0, A1, B1 = rng.normal(size=(4, N)) * 50.0
        # non-finite split densities map to -inf (bridgestan.py:47-49): B = -inf, NaN, +inf, inf - inf
        for arr, val in ((B0, -np.inf), (A1, np.nan), (B1, np.inf), (B0, np.inf)):
            arr[rng.integers(0, N, max(1, N // 50))] = val
        A0[rng.integers(0, N, max(1, N // 50))] = -np.inf
        S0, S1 = np.sum(r.astype(LD) ** 2, axis=1), np.sum(rn.astype(LD) ** 2, axis=1)
        c = LD(D) * C2PI
        sq_b = (D + 2) * U
        for off in (0, 1):
            rd, rnd = placed(r, off), placed(rn, off)
            dl = {k: placed(v, off) for k, v in dict(logw=logw, lpx=lpx, lpn=lpn, L=L, q=q, ke0=ke0, ke1=ke1, A0=A0,
                                                      B0=B0, A1=A1, B1=B1).items()}
            p = {k: dev.ptr(v) for k, v in dl.items()}
            tag = f"D={D} N={N} off={off}"

            def run(name, *args):
                out, chk = guarded(N, off=off)
                _cabi.call(name, *args, dev.ptr(out), st())
                chk()
                return out.cpu().numpy()

            out = run("smcb_row_half_sqnorm", dev.ptr(rd), N, D)
            assert_within(out, S0 / 2, sq_b * S0 / 2 + 1e-300, f"{tag} row_half_sqnorm")
            out = run("smcb_std_normal_logpdf", dev.ptr(rd), N, D)
            ref = -S0 / 2 - c
            assert_within(out, ref, sq_b * S0 / 2 + 4 * U * (c + np.abs(ref)), f"{tag} std_normal_logpdf")
            out = run("smcb_init_logw", p["lpx"], dev.ptr(rd), N, D)
            ref = lpx.astype(LD) + S0 / 2 + c
            assert_within(out, ref, sq_b * S0 / 2 + 4 * U * (c + np.abs(lpx) + np.abs(ref)), f"{tag} init_logw")
            out = run("smcb_reweight_forward", p["logw"], p["lpx"], p["lpn"], dev.ptr(rd), dev.ptr(rnd), N, D)
            ref = logw.astype(LD) + lpn - lpx - S1 / 2 + S0 / 2
            mag = np.abs(logw) + np.abs(lpn) + np.abs(lpx) + S0 / 2 + S1 / 2 + 2 * c
            assert_within(out, ref, sq_b * (S0 + S1) / 2 + 6 * U * mag, f"{tag} reweight_forward")
            out = run("smcb_reweight_forward_ke", p["logw"], p["lpx"], p["lpn"], p["ke0"], p["ke1"], N)
            ref = logw.astype(LD) + lpn - lpx - ke1 + ke0
            assert_within(out, ref, 6 * U * (np.abs(logw) + np.abs(lpn) + np.abs(lpx) + ke0 + ke1), f"{tag} _ke")
            out = run("smcb_reweight_general", p["logw"], p["lpx"], p["lpn"], p["L"], p["q"], N)
            ref = logw.astype(LD) + lpn - lpx + L - q
            assert_within(out, ref, 6 * U * (np.abs(logw) + np.abs(lpn) + np.abs(lpx) + np.abs(L) + np.abs(q)),
                          f"{tag} _general")
            for phi in (1.0, 0.3):
                out = run("smcb_reweight_forward_split", p["logw"], p["A0"], p["B0"], p["A1"], p["B1"], p["ke0"], p["ke1"],
                          phi, N)
                with np.errstate(invalid="ignore"):
                    l0, l1 = _mapped(A0 + phi * B0), _mapped(A1 + phi * B1)
                    ref = logw.astype(LD) + l1 - l0 - ke1 + ke0
                fin = np.isfinite(ref)
                assert np.array_equal(out[~fin], ref[~fin].astype(np.float64), equal_nan=True), f"{tag} _split non-finite"
                mag = (np.abs(logw) + np.abs(A0) + np.abs(phi * B0) + np.abs(A1) + np.abs(phi * B1) + ke0 + ke1)[fin]
                assert_within(out[fin], ref[fin], 8 * U * mag, f"{tag} _split")
                out = run("smcb_reweight_asymptotic", p["logw"], p["A0"], p["B0"], phi, 0.1, N)
                with np.errstate(invalid="ignore"):
                    ref = logw.astype(LD) + _mapped(A0 + phi * B0) - _mapped(A0 + 0.1 * B0)
                fin = np.isfinite(ref)
                assert np.array_equal(out[~fin], ref[~fin].astype(np.float64), equal_nan=True), f"{tag} asymptotic"
                mag = (np.abs(logw) + 2 * np.abs(A0) + 2 * np.abs(B0))[fin]
                assert_within(out[fin], ref[fin], 8 * U * mag, f"{tag} asymptotic")


# ------------------------------------------------------------------------------------------------ 4. reductions
def _sum_bound(n):
    """Relative forward error of the device's blocked sums of n non-negative terms: a per-thread chain of at most
    ceil(n / 256) terms, then tree merges (each rescales by an exp: a few u) -- generous, but far below one term."""
    return (math.ceil(n / 256) + 64) * U


def _lse_ref(logw):
    keep = ~np.isneginf(logw)
    if not keep.any():
        return -np.inf, np.nan, np.zeros_like(logw)
    z = logsumexp(logw[keep])
    w = np.exp((logw[keep].astype(LD) - LD(z)))
    s1, s2 = np.sum(w), np.sum(w * w)
    return LD(z) + np.log(s1), s1 * s1 / s2, None


def _normalise_inputs(N, rng):
    cases = {}
    v = rng.normal(size=N) * 4.0
    if N >= 3:
        a = rng.integers(0, N - N // 3)
        v[a:a + N // 3] = -np.inf                   # a run of -inf
    top = np.nanmax(np.where(np.isneginf(v), np.nan, v)) if np.isfinite(v).any() else 0.0
    v[rng.integers(0, N, max(1, N // 5))] = top + 1.5   # ties at the maximum
    cases["mixed"] = v
    cases["all_neg_inf"] = np.full(N, -np.inf)
    w = rng.normal(size=N)
    w[rng.integers(0, N)] = np.nan
    cases["nan"] = w
    return cases


NORM_SIZES = list(range(1, 10)) + [4095, 4097, 3_000_000]


@pytest.mark.gpu
@pytest.mark.parametrize("N", NORM_SIZES)
def test_normalise_every_size_and_alignment(N):
    """lse_partial (pipelined 16-byte quads when aligned, scalar otherwise, N % 4 tail) + finalize + normalise, and the
    fused normalise + tile sums of the resampling scan, against scipy's logsumexp and 1 / sum wn^2 in long double."""
    sh = ShardContext()
    rng = np.random.default_rng(N)
    for name, logw in _normalise_inputs(N, rng).items():
        for off in (0, 1):
            lw = placed(logw, off)
            tag = f"N={N} {name} off={off}"
            for scan in (False, True):
                res = normalise(lw, sh, scan=scan)
                wn, stats = res[0].cpu().numpy(), res[1].cpu().numpy()
                if name == "nan":
                    assert np.isnan(stats[0]) and np.isnan(stats[1]), tag   # NaN poisons, as scipy's logsumexp
                    continue
                if name == "all_neg_inf":
                    # nothing to sum: logZ = logsumexp([]) = -inf, ESS = 0/0 -- every weight is 0
                    assert stats[0] == -np.inf and np.isnan(stats[1]) and np.all(wn == 0.0), (tag, stats)
                    continue
                z, ess, _ = _lse_ref(logw)
                eb = _sum_bound(N)
                assert_within(stats[0], z, eb + 2 * U * abs(z), f"{tag} logZ")
                assert_within(stats[1], ess, 4 * eb * ess, f"{tag} ESS")
                with np.errstate(invalid="ignore"):
                    ref = np.where(np.isneginf(logw), LD(0), np.exp(logw.astype(LD) - z))
                    bound = np.where(np.isneginf(logw), 0, ref * (2 * U * (1 + np.abs(logw) + abs(float(z))) + eb + 2 * U))
                assert_within(wn, ref, bound, f"{tag} wn (scan={scan})")


@pytest.mark.gpu
def test_lse_partial_empty_and_positive_infinity():
    tri = dev.empty(3)
    _cabi.call("smcb_lse_partial", dev.ptr(dev.empty(1)), 0, dev.ptr(tri), dev.ptr(dev.reduce_ws()), st())
    t = tri.cpu().numpy()
    assert t[0] == -np.inf and t[1] == 0.0 and t[2] == 0.0, t
    sh = ShardContext()
    rng = np.random.default_rng(3)
    for N in (1, 2, 3, 4, 5, 8, 9, 4097):
        base = rng.normal(size=N)
        for pos in (range(N) if N < 10 else (0, 1, 2, 3, N // 2, N - 2, N - 1)):
            v = base.copy()
            v[pos] = np.inf
            for off in (0, 1):
                stats = normalise(placed(v, off), sh)[1].cpu().numpy()
                assert not np.isfinite(stats[0]), (N, pos, off, stats)


@pytest.mark.gpu
def test_ess_multi_phi_every_candidate_count():
    """NV = 1 / 4 / 8 / 16 instantiations; each candidate's triple -> logsumexp and ESS of phi*loglik + logpri - c."""
    rng = np.random.default_rng(5)
    N = 10007
    ll, pri, c = rng.normal(size=N) * 20, rng.normal(size=N), rng.normal(size=N)
    pri[rng.integers(0, N, 300)] = -np.inf
    lld, prid, cd = placed(ll), placed(pri, 1), placed(c)
    for m in range(1, 17):
        phis = np.sort(rng.uniform(0, 1, m))
        out, chk = guarded(3 * m)
        phid = dev.to_device(phis)
        _cabi.call("smcb_ess_multi_phi", dev.ptr(lld), dev.ptr(prid), dev.ptr(cd), N, dev.ptr(phid), m,
                   dev.ptr(out), dev.ptr(dev.reduce_ws()), st())
        chk()
        o = out.cpu().numpy().reshape(m, 3)
        for j, ph in enumerate(phis):
            z, ess, _ = _lse_ref((ph * ll + pri) - c)
            eb = _sum_bound(N)
            assert_within(o[j, 0] + math.log(o[j, 1]), z, eb + 4 * U * abs(z), f"m={m} j={j} logZ")
            assert_within(o[j, 1] ** 2 / o[j, 2], ess, 4 * eb * ess, f"m={m} j={j} ESS")


def _multinomial_wn(N, rng):
    """Normalised weights whose sum is exactly 1 (dyadic), so that sum wn (v - c) and c + sum wn (v - c) mean the
    same thing in every precision."""
    return dyadic_weights(rng.exponential(size=N) ** 2, 40, int(rng.integers(1 << 30)))


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 3, 7, 13, 100, 128, 129, 200, 255, 256])
def test_weighted_moment_every_width(D):
    """threads_used = (256 / D) D columns per sweep; exp on the last coordinate (arma / PRMwCD constraint)."""
    rng = np.random.default_rng(D)
    N = 3001
    x = rng.normal(size=(N, D)) + rng.normal(size=D) * 3
    wn = _multinomial_wn(N, rng)
    cen = rng.normal(size=D)
    xd, wd = placed(x), placed(wn)
    for constrain in (_cabi.CONSTRAIN_NONE, _cabi.CONSTRAIN_EXP_LAST):
        v = x.astype(LD)
        if constrain == _cabi.CONSTRAIN_EXP_LAST:
            v[:, -1] = np.exp(x[:, -1])
        for center in (None, cen):
            for power in (1, 2):
                out, chk = guarded(D)
                cd = dev.to_device(center) if center is not None else None
                _cabi.call("smcb_weighted_moment", dev.ptr(xd), dev.ptr(wd), N, D, constrain, dev.ptr(cd), power,
                           dev.ptr(out), dev.ptr(dev.reduce_ws()), st())
                chk()
                t = (v - (center.astype(LD) if center is not None else 0)) ** power
                ref = np.sum(wn.astype(LD)[:, None] * t, axis=0)
                mag = np.sum(wn.astype(LD)[:, None] * np.abs(t), axis=0)
                assert_within(out.cpu().numpy(), ref, _sum_bound(N) * mag + 4 * U * mag,
                              f"D={D} constrain={constrain} center={center is not None} power={power}")


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 2, 3, 7, 13, 64, 100, 127, 128])
def test_weighted_moments12_and_finalize_against_two_pass(D):
    """The one-pass moments SMCSampler uses (centre = the previous mean): mean = c + m1 and var = m2 - m1^2 against
    a two-pass long double reference.  Within 10 sd of the mean the centre costs nothing (~1e-12); further out the
    subtraction cancels (offset / sd)^2 u of the variance, which is pinned here."""
    rng = np.random.default_rng(D)
    N = 4099
    sd = np.exp(rng.uniform(-3, 3, D))
    x = rng.normal(size=(N, D)) * sd + rng.normal(size=D) * 5
    x[:, -1] = rng.normal(size=N) * 0.5     # exp() of the last coordinate stays O(1)
    wn = _multinomial_wn(N, rng)
    xd, wd = placed(x), placed(wn, 1)
    for constrain in (_cabi.CONSTRAIN_NONE, _cabi.CONSTRAIN_EXP_LAST):
        v = x.astype(LD)
        if constrain == _cabi.CONSTRAIN_EXP_LAST:
            v[:, -1] = np.exp(x[:, -1])
        w = wn.astype(LD)[:, None]
        mean = np.sum(w * v, axis=0)
        var = np.sum(w * (v - mean) ** 2, axis=0)
        s = np.sqrt(var)
        for k_sd in (None, 0.0, 10.0, 1e4):
            center = None if k_sd is None else (mean + LD(k_sd) * s * np.where(np.arange(D) % 2, 1, -1)).astype(np.float64)
            sums, chk = guarded(2 * D)
            cd = dev.to_device(center) if center is not None else None
            _cabi.call("smcb_weighted_moments12", dev.ptr(xd), dev.ptr(wd), N, D, constrain, dev.ptr(cd), dev.ptr(sums),
                       dev.ptr(dev.reduce_ws()), st())
            chk()
            mu, va = guarded(D), guarded(D)
            _cabi.call("smcb_moments12_finalize", dev.ptr(sums), dev.ptr(cd), D, dev.ptr(mu[0]), dev.ptr(va[0]), st())
            mu[1](), va[1]()
            off = np.abs((center.astype(LD) if center is not None else LD(0)) - mean)
            tag = f"D={D} constrain={constrain} centre={k_sd}"
            close = off <= 10.0 * s * (1 + 1e-12)
            tol_m = 1e-12 * (s + np.abs(mean)) + 8 * U * off
            tol_v = np.where(close, 1e-12 * var, 1e-12 * var + 64 * U * (off ** 2 + var))   # ~ 64 (off / sd)^2 u
            assert_within(mu[0].cpu().numpy(), mean, tol_m, f"{tag} mean")
            assert_within(va[0].cpu().numpy(), var, tol_v, f"{tag} var")


@pytest.mark.gpu
def test_counters_sum_int32_sum_f64_count_moved():
    ws = dev.reduce_ws()
    rng = np.random.default_rng(0)
    v = (2 ** 31 - 1) - rng.integers(0, 1000, 1 << 20).astype(np.int32)   # the total needs 52 bits
    vd = placed(v, 1, torch.int32)
    out, chk = guarded(1, torch.int64)
    _cabi.call("smcb_sum_int32", dev.ptr(vd), len(v), dev.ptr(out), dev.ptr(ws), st())
    chk()
    assert int(out.item()) == int(v.astype(np.int64).sum())
    for N in (1, 257, 1_000_000):
        a = rng.normal(size=N) * np.exp(rng.uniform(-5, 5, N))
        out, chk, ad = *guarded(1), placed(a, N % 2)
        _cabi.call("smcb_sum_f64", dev.ptr(ad), N, dev.ptr(out), dev.ptr(ws), st())
        chk()
        assert_within(out.cpu().numpy(), LD(math.fsum(a)), _sum_bound(N) * np.sum(np.abs(a)), f"sum_f64 N={N}")
        D = 3
        x = rng.normal(size=(N, D))
        xn = x.copy()
        change = rng.random((N, D)) < 0.8
        xn[change] += 1.0
        out, chk, xd, xnd = *guarded(1), placed(x), placed(xn, 1)
        _cabi.call("smcb_count_moved", dev.ptr(xd), dev.ptr(xnd), N, D, dev.ptr(out), dev.ptr(ws), st())
        chk()
        assert out.item() == float(np.sum(np.all(change, axis=1))), N


# ------------------------------------------------------------------------------------------------ 5. resampling
def _sys_positions(j0, M, M_total, u0):
    return (np.arange(j0, j0 + M, dtype=np.float64) + u0) / float(M_total)


def _sys_want(cdf, j0, M, M_total, u0):
    return np.minimum(np.searchsorted(cdf, _sys_positions(j0, M, M_total, u0), side="right"), len(cdf) - 1)


def _resample_weights(N, rng):
    p = rng.exponential(size=N) ** 2
    a = int(rng.integers(0, N - 3000))
    p[a:a + 3000] = 0.0            # a zero-weight run longer than 2048 entries: tiles that span it binary-search
    wn = dyadic_weights(p, 30, int(rng.integers(1 << 30)))
    return wn, O.cdf_of(wn)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 2, 3, 4, 8, 13, 16, 32, 64, 100])
def test_resample_systematic_every_path(D):
    """Fused kernel (aligned D in {2, 4, ..., 64}: ballot rank for tiles spanning <= 2048 cdf entries, binary search
    above) and the unfused search + gather; shard offsets j0 > 0 with M_total != N; idx = None."""
    rng = np.random.default_rng(D)
    N = 20_000
    wn, cdf = _resample_weights(N, rng)
    cdf_t, _ = _dev_cdf(wn)
    assert np.array_equal(cdf_t.cpu().numpy(), cdf)     # dyadic weights: the device scan is np.cumsum bit for bit
    x = rng.normal(size=(N, D))
    fused = D in (2, 4, 8, 16, 32, 64)
    for M in (1, 31, 32, 33, 1000, (1 << 17) + 5):
        for j0, M_total in ((0, M), (7, M + 7 + 11)):
            u0 = float(rng.random())
            want = _sys_want(cdf, j0, M, M_total, u0)
            for off in (0, 1):
                xd = placed(x, off)
                out, chk = guarded(M * D, off=off)
                idx, chk_i = guarded(M, torch.int64)
                ws = dev.empty((_cabi.lib().smcb_resample_workspace_bytes(M, D) + 7) // 8)
                _cabi.call("smcb_resample_systematic", dev.ptr(cdf_t), N, u0, None, j0, M_total, M, dev.ptr(xd), D,
                           dev.ptr(out), dev.ptr(idx), dev.ptr(ws), st())
                chk(), chk_i()
                tag = f"D={D} M={M} j0={j0} off={off}"
                got = idx.cpu().numpy()
                assert np.array_equal(got, want), (tag, np.flatnonzero(got != want)[:10])
                assert np.array_equal(out.cpu().numpy().reshape(M, D), x[want]), tag
                if fused and off == 0:
                    out2, chk2 = guarded(M * D)
                    _cabi.call("smcb_resample_systematic", dev.ptr(cdf_t), N, u0, None, j0, M_total, M, dev.ptr(xd), D,
                               dev.ptr(out2), None, dev.ptr(ws), st())
                    chk2()
                    assert np.array_equal(out2.cpu().numpy().reshape(M, D), x[want]), tag
                elif not fused:
                    with pytest.raises(_cabi.SmcbError):
                        _cabi.call("smcb_resample_systematic", dev.ptr(cdf_t), N, u0, None, j0, M_total, M, dev.ptr(xd),
                                   D, dev.ptr(out), None, dev.ptr(ws), st())


def _dev_cdf(wn):
    n = len(wn)
    w = dev.to_device(wn)
    cdf, tot = dev.empty(n), dev.empty(1)
    ws = dev.workspace("scan", _cabi.lib().smcb_scan_workspace_bytes(n))
    _cabi.call("smcb_cdf", dev.ptr(w), n, 0, 0, dev.ptr(cdf), dev.ptr(tot), dev.ptr(ws), st())
    return cdf, tot


@pytest.mark.gpu
@pytest.mark.parametrize("D", [2, 4, 16])
def test_resample_systematic_ties_follow_searchsorted_right(D):
    """u0 = 1/2 and M a power of two: positions (j + 1/2) / M land exactly on cdf values; the ancestor of a position
    equal to cdf[i] is i + 1 (np.searchsorted side='right'), in the ballot rank and in the binary search alike."""
    for M, N in ((1024, 2048), (1024, 2048 * 8), (64, 2048 * 64)):
        wn = np.full(N, 1.0 / N)
        cdf = O.cdf_of(wn)
        pos = _sys_positions(0, M, M, 0.5)
        assert np.isin(pos, cdf).all()
        want = _sys_want(cdf, 0, M, M, 0.5)
        x = np.random.default_rng(M).normal(size=(N, D))
        idx, chk = guarded(M, torch.int64)
        out, cdf_d, xd = dev.empty(M, D), dev.to_device(cdf), dev.to_device(x)
        ws = dev.empty((_cabi.lib().smcb_resample_workspace_bytes(M, D) + 7) // 8)
        _cabi.call("smcb_resample_systematic", dev.ptr(cdf_d), N, 0.5, None, 0, M, M, dev.ptr(xd), D, dev.ptr(out),
                   dev.ptr(idx), dev.ptr(ws), st())
        chk()
        assert np.array_equal(idx.cpu().numpy(), want), (M, N)
        assert np.array_equal(out.cpu().numpy(), x[want])


def _peer_table(base, P, rows_per_rank, gap, D):
    """P destination pointers into one buffer, each rank's slots followed by `gap` untouched rows."""
    stride = (rows_per_rank + gap) * D * 8
    return dev.to_device(np.array([base.data_ptr() + q * stride for q in range(P)], dtype=np.int64), torch.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [2, 4, 16])
def test_resample_systematic_push_on_one_gpu(D):
    """The push variant with the peer table pointing at slices of one local buffer: every slot of [j0, j0 + M) is
    written with its ancestor's row, in the scattered tile order (nruns > 1), and nothing else changes."""
    rng = np.random.default_rng(D)
    N = 20_000
    wn, cdf = _resample_weights(N, rng)
    cdf_t = dev.to_device(cdf)
    x = rng.normal(size=(N, D))
    xd = dev.to_device(x)
    M, j0 = (1 << 14) + 3, 5
    M_total = j0 + M + 2
    assert ((M + 31) // 32) >> 4 > 1
    for rpr in (1, 7, -(-M // 3)):
        gap = 1
        P = -(-(j0 + M) // rpr)
        nrows = P * (rpr + gap)
        buf, chk = guarded(nrows * D)
        table = _peer_table(buf, P, rpr, gap, D)
        idx, chk_i = guarded(M, torch.int64)
        ws = dev.empty((_cabi.lib().smcb_resample_workspace_bytes(M, D) + 7) // 8)
        u0 = float(rng.random())
        _cabi.call("smcb_resample_systematic_push", dev.ptr(cdf_t), N, u0, j0, M_total, M, dev.ptr(xd), D,
                   dev.ptr(table), rpr, dev.ptr(idx), dev.ptr(ws), st())
        chk(), chk_i()
        want = _sys_want(cdf, j0, M, M_total, u0)
        assert np.array_equal(idx.cpu().numpy(), want), rpr
        gj = np.arange(j0, j0 + M)
        row = (gj // rpr) * (rpr + gap) + gj % rpr
        got = buf.cpu().numpy().reshape(nrows, D)
        assert np.array_equal(got[row], x[want]), rpr
        untouched = np.ones(nrows, bool)
        untouched[row] = False
        bits = buf.view(torch.int64).cpu().numpy().reshape(nrows, D)
        assert np.all(bits[untouched] == _SENTINEL[torch.float64][1]), rpr


@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 3])
def test_resample_multinomial_push_emulated_ranks(P):
    """Owner-push multinomial resampling with P ranks emulated on one GPU: each call gets its segment of the global
    cdf, the segment ends and its particle0; the union of the writes is the single-GPU multinomial resampling."""
    rng = np.random.default_rng(P)
    N, D, seed, it = 30_001, 4, 10, 4
    wn = dyadic_weights(rng.exponential(size=N) ** 3, 30, P)
    cdf = O.cdf_of(wn)
    x = rng.normal(size=(N, D))
    u = O.uniforms(seed, it, philox.STREAM_RESAMPLE, 0, N)
    want = np.searchsorted(cdf, u, side="right")
    cuts = np.sort(rng.choice(np.arange(1, N), P - 1, replace=False))
    seg = np.split(np.arange(N), cuts)
    ends = dev.to_device(np.array([cdf[s[-1]] for s in seg]))
    rpr = -(-N // P)
    out, chk = guarded(P * rpr * D)
    oidx, chk_i = guarded(P * rpr, torch.int64)
    table = _peer_table(out, P, rpr, 0, D)
    itable = dev.to_device(np.array([oidx.data_ptr() + q * rpr * 8 for q in range(P)], dtype=np.int64), torch.int64)
    keep = []
    for q, s in enumerate(seg):
        c_q, x_q = dev.to_device(cdf[s]), placed(x[s], q % 2)
        keep += [c_q, x_q]
        _cabi.call("smcb_resample_multinomial_push", dev.ptr(c_q), len(s), dev.ptr(ends), q, P, seed, it,
                   philox.STREAM_RESAMPLE, N, int(s[0]), dev.ptr(x_q), D, dev.ptr(table), dev.ptr(itable), rpr, st())
    chk(), chk_i()
    assert np.array_equal(oidx.cpu().numpy()[:N], want)
    assert np.array_equal(out.cpu().numpy()[:N * D].reshape(N, D), x[want])
    tail = oidx.view(torch.int64).cpu().numpy()[N:]
    assert np.all(tail == _SENTINEL[torch.int64][1])
