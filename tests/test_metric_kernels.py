"""The diagonal-metric NUTS kernels (ScaledModel<M>, csrc/models.cuh) at every model and dispatch they are built for.

A diagonal mass matrix diag(1 / s^2) is identity-metric NUTS on z = x / s: the kernels evaluate the model at x = z * s and
return the gradient g * s, the host converts x -> z before the launch and z_new -> x_new after it (proposal/nuts.py).  The
recursive C oracle does the same operations in the same order (COracleTarget.nuts_batch(..., scale=s)), so wherever the
unscaled lanes equal the oracle bit for bit, the scaled ones must too; elsewhere they are held to the tolerances of the
unscaled comparisons.

CPU: the lanes through tests/hostsim (one-lane kernels, and the 4-lanes-per-particle kernels on the warp emulator), and the
wrapper alone on a probe model.  GPU: the parity build bit for bit, the product build at every dispatch, generated
plug-ins, smcb_scale_rows / smcb_scale_rows_accepted in guarded buffers, and the validation of set_metric_scale.

Scales span e^-2 .. e^2 in a non-monotone order, so that a permuted or lane-swapped scale changes the result."""
import math

import numpy as np
import pytest
import torch

from oracle import smc_oracle as O
from tests.hostsim import sim

PRM_CENTRE = np.array([0.8925, 0.0946, 1.3969, 0.1151, -1.4883, -0.0898, 0.6766, -1.7521, -0.3014, 1.6721, -0.1868,
                       -0.1491, math.log(0.3326)])


def metric_scale(D, lo=-2.0, hi=2.0):
    """exp of D points spread over [lo, hi], in a fixed non-monotone order (a stride permutation plus a swap of the
    first two, so no coordinate keeps its rank and no lane of a group sees a sorted run)."""
    if D == 1:
        return np.array([math.exp(0.37 * hi)])
    v = np.exp(np.linspace(lo, hi, D))
    step = next(k for k in (7, 5, 3, 2, 1) if math.gcd(k, D) == 1 and k < D)
    perm = (np.arange(D) * step + D // 2) % D
    out = v[perm]
    out[[0, 1]] = out[[1, 0]]
    return out


def _inputs(tname, D, N, seed):
    """Start points with wild rows (divergent trajectories; -inf densities where the model has them)."""
    rng = np.random.default_rng(seed)
    if tname == "arma":
        x = rng.normal(size=(N, D)) * 0.3 + np.array([0.0, 0.9, 0.0, -1.7])
        x[:20] = rng.normal(size=(20, 4)) * 2.0
        x[0, 3] = 800.0                                    # sigma = inf -> A = -inf
    elif tname == "PRMwCD":
        x = PRM_CENTRE + rng.normal(size=(N, D)) * 0.05
        x[:6] = rng.normal(size=(6, D)) * 3.0
        x[6:9, 0] = -800.0                                 # lambda underflows to 0 with y > 0 -> B = -inf
    else:
        x = rng.normal(size=(N, D)) * 0.3
        x[:4] *= 40.0                                      # far out in the tails: divergent trajectories
    return x, rng.normal(size=(N, D))


def _lp(o, phi):
    with np.errstate(invalid="ignore"):
        lp_old, lp_new = o["A_old"] + phi * o["B_old"], o["A_new"] + phi * o["B_new"]
    return np.where(np.isfinite(lp_old), lp_old, -np.inf), np.where(np.isfinite(lp_new), lp_new, -np.inf)


def _assert_bitwise(o, ref, r, phi, what):
    for k in ("n_leapfrog", "depth", "accepted"):
        assert np.array_equal(o[k], ref[k]), (what, k, float((o[k] != ref[k]).mean()))
    assert np.array_equal(o["x_new"], ref["x_new"], equal_nan=True), (what, "x_new")
    assert np.array_equal(o["r_new"], ref["r_new"], equal_nan=True), (what, "r_new")
    lp_old, lp_new = _lp(o, phi)
    assert np.array_equal(lp_old, ref["lp_old"]) and np.array_equal(lp_new, ref["lp_new"]), (what, "lp")
    np.testing.assert_allclose(o["ke_old"], 0.5 * np.sum(r * r, axis=1), rtol=1e-14)


# ================================================================================================== CPU
@pytest.mark.parametrize("tname,D,eps,N", [("arma", 4, 0.03, 400), ("PRMwCD", 13, 0.01, 40), ("gauss", 1, 0.5, 300),
                                           ("gauss", 3, 0.05, 300), ("gauss", 13, 0.03, 150), ("gauss", 100, 0.02, 40),
                                           ("gauss", 128, 0.02, 30)])
@pytest.mark.parametrize("devmath", [False, True])
def test_scaled_lane_matches_c_oracle_bitwise(tname, D, eps, N, devmath):
    """One-lane kernels (ArmaModel, PrmModel, the plain GaussModel) under a metric: the same statements as the oracle's
    ctx_eval (x = z * s, g * s), so every output is the oracle's bit for bit, in both exp / log flavours."""
    t = O.COracleTarget(tname, **({"dim": D} if tname == "gauss" else {}))
    x, r = _inputs(tname, D, N, 5)
    s = metric_scale(D)
    for accrej, phi in ((False, 1.0), (True, 0.2)):
        with O.devmath(devmath):
            ref = t.nuts_batch(x, r, eps, phi, 10, seed=77, iteration=3, particle0=1000, accrej=accrej, scale=s)
        o = sim.nuts(tname, t.np_target, x, r, eps, phi, 10, accrej, 77, 3, 1000, lanes=32, devmath=devmath, scale=s)
        _assert_bitwise(o, ref, r, phi, f"{tname} D={D} accrej={accrej}")
        if accrej:
            assert 0 < (ref["accepted"] == 0).sum() < N, "the MH epilogue rejects some particles and keeps others"
    # scale = ones: x * 1 and g * 1 are exact, so the wrapper is invisible
    ones = sim.nuts(tname, t.np_target, x, r, eps, 0.2, 10, True, 77, 3, 1000, lanes=7, devmath=devmath, scale=np.ones(D))
    plain = sim.nuts(tname, t.np_target, x, r, eps, 0.2, 10, True, 77, 3, 1000, lanes=7, devmath=devmath)
    for k in plain:
        assert np.array_equal(ones[k], plain[k], equal_nan=True), k


@pytest.mark.parametrize("D", [5, 8, 9, 16, 17, 32, 33, 64, 65, 100, 104])
def test_scaled_group_kernel_gauss_matches_c_oracle_bitwise(D):
    """GaussModelG<NT8> under a metric on the emulated warp, NT8 = 1, 2, 4, 8, 13 with a full and a padded last block of
    8 coordinates: lane `sub` of a group holds coordinates sub, sub + 4, ..., and must scale exactly those.  The emulated
    mma sums -Px in the oracle's order, so trees, MH outcomes and returned rows are the oracle's bit for bit (ragged work
    queue: N is not a multiple of the 8 particles a warp holds)."""
    t = O.COracleTarget("gauss", dim=D)
    N = 45 if D <= 17 else 19 if D <= 33 else 11     # ragged: 5.6, 2.4 and 1.4 warps' worth of particles
    x, r = _inputs("gauss", D, N, D)
    s = metric_scale(D)
    eps = 0.03
    for accrej, phi in ((False, 1.0), (True, 0.7)):
        ref = t.nuts_batch(x, r, eps, phi, 10, seed=77, iteration=3, particle0=1000, accrej=accrej, scale=s)
        o = sim.nuts_simt("gauss", t.np_target, x, r, eps, phi, 10, accrej, 77, 3, 1000, scale=s)
        for k in ("n_leapfrog", "depth", "accepted", "x_new", "r_new"):
            assert np.array_equal(o[k], ref[k]), (accrej, k)
        np.testing.assert_allclose(o["ke_old"], 0.5 * np.sum(r * r, axis=1), rtol=1e-14)
        # the quadratic form is folded over the 4 lanes of a group by shuffles (a tree), the oracle sums it in order
        np.testing.assert_allclose(o["A_new"] + phi * o["B_new"], ref["lp_new"], rtol=1e-13)
    ones = sim.nuts_simt("gauss", t.np_target, x, r, eps, 0.7, 10, True, 77, 3, 1000, scale=np.ones(D))
    plain = sim.nuts_simt("gauss", t.np_target, x, r, eps, 0.7, 10, True, 77, 3, 1000)
    for k in plain:
        assert np.array_equal(ones[k], plain[k]), k


def test_scaled_group_kernel_prmwcd_matches_c_oracle():
    """PrmModelG under a metric on the emulated warp (13 coordinates in 16 slots: lanes 1-3 pad their last slot), with
    the tolerances of the unscaled comparison: its tensor-core sums are associated differently from the oracle's."""
    t = O.COracleTarget("PRMwCD")
    N = 44
    x, r = _inputs("PRMwCD", 13, N, 21)
    s = metric_scale(13, -0.7, 0.7)     # e^+-2 on this target leaves almost every tree at the depth cap
    phi = 0.6
    ref = t.nuts_batch(x, r, 0.01, phi, 10, seed=3, iteration=1, accrej=True, scale=s)
    o = sim.nuts_simt("PRMwCD", t.np_target, x, r, 0.01, phi, 10, True, 3, 1, 0, scale=s)
    Ao, Bo, _, _ = t.split(x / s * s, grads=False)          # the start point the lanes evaluate: (x / s) * s
    assert np.all(np.isneginf(o["B_old"][6:9])) and np.array_equal(np.isfinite(o["B_old"]), np.isfinite(Bo))
    fin = np.isfinite(Bo)
    np.testing.assert_allclose(o["A_old"][fin], Ao[fin], rtol=1e-13)
    np.testing.assert_allclose(o["B_old"][fin], Bo[fin], rtol=1e-12)
    same = o["n_leapfrog"] == ref["n_leapfrog"]
    assert same.mean() >= 0.9, same.mean()
    assert np.array_equal(o["depth"][same], ref["depth"][same])
    ok = same & (o["accepted"] == ref["accepted"]) & np.isfinite(ref["x_new"]).all(axis=1)
    close = np.isclose(o["x_new"][ok], ref["x_new"][ok], rtol=1e-4, atol=1e-6).all(axis=1)
    assert close.mean() >= 0.85, close.mean()
    rej = o["accepted"] == 0
    assert rej.any() and np.array_equal(o["x_new"][rej], x[rej]) and np.array_equal(o["r_new"][rej], r[rej])
    ones = sim.nuts_simt("PRMwCD", t.np_target, x, r, 0.01, phi, 10, True, 3, 1, 0, scale=np.ones(13))
    plain = sim.nuts_simt("PRMwCD", t.np_target, x, r, 0.01, phi, 10, True, 3, 1, 0)
    for k in plain:
        assert np.array_equal(ones[k], plain[k], equal_nan=True), k


@pytest.mark.parametrize("group,nloc,dims", [(1, 4, [1, 3, 4]), (4, 4, [13, 16]), (4, 2, [1, 5, 8]),
                                             (4, 8, [9, 16]), (4, 16, [33, 63, 64]), (4, 26, [65, 100, 104])])
def test_scaled_model_maps_slots_to_coordinates(group, nloc, dims):
    """The wrapper alone, on a probe model whose gradient is the x it is evaluated at: slot i of lane `sub` must be scaled
    by scale[sub + GROUP i] on the way in and on the way out (g = s * s * z), padded slots (coordinate >= D) by exactly
    1.  Through NUTS the padding is invisible (its z and gradient are 0), so it is pinned here."""
    rng = np.random.default_rng(group * 100 + nloc)
    for D in dims:
        s = metric_scale(D)
        z = rng.normal(size=(32, nloc))
        g = sim.scaled_probe(group, nloc, D, s, z)
        lane = np.arange(32)[:, None]
        coord = (lane % group) + group * np.arange(nloc)[None, :] if group > 1 else np.broadcast_to(np.arange(nloc), (32, nloc))
        sc = np.where(coord < D, s[np.minimum(coord, D - 1)], 1.0)
        assert np.array_equal(g, (z * sc) * sc), (group, nloc, D)


# ================================================================================================== GPU
if torch.cuda.is_available():
    from smcnuts import _cabi, _device as dev
    from smcnuts.distributions import StdNormal
    from smcnuts.model.device_model import make_model
    from smcnuts.proposal.nuts import NUTSProposal
    from smcnuts.proposal.nuts_acc_rej import NUTSProposalWithAccRej
    from tests.test_gpu_dispatch import W_DIMS, W_SIZES, dense_spd, guarded, placed


def _host(o):
    return {k: v.cpu().numpy() for k, v in o.items()}


def _transition(m, x, r, eps, phi, accrej, seed, it, max_depth=10, particle0=0):
    """One transition whose outputs start as NaN / -1: a row the kernel does not write fails the comparisons instead of
    keeping what an earlier transition left in the same (recycled) allocation."""
    cls = NUTSProposalWithAccRej if accrej else NUTSProposal
    k = cls(m, StdNormal(m.dim), eps, rng=seed, max_tree_depth=max_depth)
    k.particle0 = particle0
    k.prepare(len(x), m.dim)
    pre = k._prepared[1]
    for v in pre.values():
        v.fill_(float("nan") if v.is_floating_point() else -1)
    o = k.transition(dev.to_device(x), dev.to_device(r), phi, iteration=it)
    assert all(o[key].data_ptr() == v.data_ptr() for key, v in pre.items())   # the pre-filled buffers were used
    return _host(o)


@pytest.fixture
def scalar_kernels(monkeypatch):
    """One lane per particle (the kernels whose summation order is the oracle's)."""
    monkeypatch.setenv("SMCB_PRM_SCALAR", "1")
    monkeypatch.setenv("SMCB_GAUSS_SCALAR", "1")


@pytest.fixture
def blocks_per_sm():
    """smcb_nuts_set_blocks_per_sm is a process-wide setting: always put it back."""
    yield lambda n: _cabi.call("smcb_nuts_set_blocks_per_sm", n)
    _cabi.call("smcb_nuts_set_blocks_per_sm", 0)


@pytest.mark.gpu
@pytest.mark.parametrize("tname,D,eps,N", [("arma", 4, 0.01, 3001), ("PRMwCD", 13, 0.01, 1501), ("gauss", 8, 0.03, 1001),
                                           ("gauss", 16, 0.03, 601), ("gauss", 33, 0.03, 301), ("gauss", 64, 0.02, 201),
                                           ("gauss", 100, 0.02, 201), ("gauss", 128, 0.02, 201)])
def test_scaled_parity_build_equals_oracle_bit_for_bit(tname, D, eps, N, scalar_kernels):
    """libsmcnuts_b200_parity.so (-DSMCB_PARITY=1 -fmad=false) with a metric set through smcb_model_set_scale, against the
    oracle in device-arithmetic mode: every output identical, with and without the MH epilogue, tempered and not.  The
    one-lane kernels (SMCB_GAUSS_SCALAR=1 takes every D to the plain Gaussian kernel)."""
    t = O.COracleTarget(tname, **({"dim": D} if tname == "gauss" else {}))
    x, r = _inputs(tname, D, N, 5)
    s = metric_scale(D, -1.0, 1.0) if tname == "PRMwCD" else metric_scale(D)
    for accrej, phi in ((False, 1.0), (True, 0.2)):
        with O.devmath():
            ref = t.nuts_batch(x, r, eps, phi, 10, seed=77, iteration=3, particle0=1000, accrej=accrej, nthreads=8,
                               scale=s)
        with _cabi.use_library(_cabi.PARITY_LIB_PATH) as L:
            assert L.smcb_build_flavour() == 1
            m = make_model(tname, **({"dim": D} if tname == "gauss" else {}))
            m.set_metric_scale(s)
            o = _transition(m, x, r, eps, phi, accrej, 77, 3, particle0=1000)
            del m
        _assert_bitwise(o, ref, r, phi, f"{tname} D={D} accrej={accrej}")
        if accrej:
            assert (o["accepted"] == 0).any()
    if tname == "PRMwCD":
        assert ref["n_leapfrog"].max() >= 511       # the long, chaotic trees are part of the comparison


# the product build: D -> kernel (GaussModelG<NT8> for NT8 = 1 / 2 / 4 / 8 / 13 up to D = 104, the plain kernel above)
PRODUCT_CASES = [("gauss", D, "0") for D in (1, 8, 9, 16, 17, 32, 33, 64, 65, 104, 105, 128)] + \
    [("gauss", 33, "1"), ("PRMwCD", 13, "0"), ("PRMwCD", 13, "1"), ("arma", 4, "0")]


@pytest.mark.gpu
@pytest.mark.parametrize("tname,D,scalar", PRODUCT_CASES)
def test_scaled_product_kernels_match_oracle_at_every_dispatch(tname, D, scalar, monkeypatch, blocks_per_sm):
    """The product build under a metric against the oracle, with the tolerances of the unscaled metric test: >= 97 % equal
    trees, rows to 1e-6, A / B by-products equal to the x-space split at x_new.  Ragged N (not a multiple of a CTA or of a
    warp's 8 particles); a cap of one CTA per SM must not change a bit; scale = ones must equal no metric bit for bit."""
    monkeypatch.setenv("SMCB_GAUSS_SCALAR", scalar)
    monkeypatch.setenv("SMCB_PRM_SCALAR", scalar)
    N = 2048 + 13
    rng = np.random.default_rng(D)
    if tname == "gauss":
        P = dense_spd(D, 1000 + D)
        m, t = make_model("gauss", precision=P), O.COracleTarget("gauss", precision=P)
        s = metric_scale(D)
        x = rng.normal(size=(N, D)) @ np.linalg.cholesky(np.linalg.inv(P)).T
        eps = 0.25 * 0.5 / s.max()          # a quarter of the smallest z-space sd (eigenvalues of P are <= 4)
    else:
        m, t = make_model(tname), O.COracleTarget(tname)
        s = metric_scale(D, -0.7, 0.7)     # the range the unscaled-metric comparison of these models runs at
        x = rng.normal(size=(N, D)) * 0.1 + (np.array([0.0, 0.9, 0.0, -1.7]) if tname == "arma" else 0.0)
        eps = 0.02 if tname == "arma" else 0.01
    r = rng.normal(size=(N, D))
    phi, seed, it = 0.8, 7, 2
    plain = _transition(m, x, r, eps, phi, False, seed, it, max_depth=6)
    m.set_metric_scale(np.ones(D))
    try:
        ones = _transition(m, x, r, eps, phi, False, seed, it, max_depth=6)
        m.set_metric_scale(s)
        o = _transition(m, x, r, eps, phi, False, seed, it, max_depth=6)
        blocks_per_sm(1)
        capped = _transition(m, x, r, eps, phi, False, seed, it, max_depth=6)
        blocks_per_sm(0)
        A, B = (v.cpu().numpy() for v in m.split(o["x_new"]))
    finally:
        m.set_metric_scale(None)
    for k in plain:
        assert np.array_equal(ones[k], plain[k], equal_nan=True), ("scale = ones", k)
        assert np.array_equal(capped[k], o[k], equal_nan=True), ("one CTA per SM", k)
    ref = t.nuts_batch(x, r, eps, phi, 6, seed=seed, iteration=it, nthreads=8, scale=s)
    same = o["n_leapfrog"] == ref["n_leapfrog"]
    assert same.mean() > 0.97, same.mean()
    assert not np.array_equal(o["x_new"], plain["x_new"])                  # the metric is in effect
    np.testing.assert_allclose(o["x_new"][same], ref["x_new"][same], rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(o["r_new"][same], ref["r_new"][same], rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(o["A_new"], A, rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(o["B_new"], B, rtol=1e-9, atol=1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("tname,D", [("arma", 4), ("gauss", 33), ("gauss", 105)])
def test_rejected_particles_keep_their_rows_under_a_metric(tname, D):
    """With the MH epilogue, a rejected particle returns its x row unchanged.  The kernel hands back z = x / s for it,
    and z * s need not round to x: the way back to x-space takes the rejected rows from x (smcb_scale_rows_accepted)."""
    N = 4096 + 5
    s = metric_scale(D)
    if tname == "gauss":
        rng = np.random.default_rng(D)
        m = make_model(tname, precision=dense_spd(D, D))
        x, r, eps = rng.normal(size=(N, D)) * 0.3, rng.normal(size=(N, D)), 0.5 / s.max()
    else:
        m = make_model(tname)
        (x, r), eps = _inputs(tname, D, N, 4), 0.03
    m.set_metric_scale(s)
    try:
        o = _transition(m, x, r, eps, 0.4, True, 3, 1, max_depth=5)
    finally:
        m.set_metric_scale(None)
    rej = o["accepted"] == 0
    assert 0 < rej.sum() < N
    assert np.array_equal(o["x_new"][rej], x[rej]) and np.array_equal(o["r_new"][rej], r[rej])
    assert (x[rej] / s * s != x[rej]).any()                   # a round trip through z would have moved some of them


# ------------------------------------------------------------------------------------------------ plug-ins
def _arma_data():
    from tests.test_stan_codegen import _arma_data as data
    return data()


@pytest.mark.gpu
def test_generated_arma_series_under_a_metric_runs_like_the_builtin():
    """ScaledModel<generated struct>: the plug-in of tests/stan/arma_series.stan and the built-in arma under the same
    metric: the same trees up to the rounding of two formulations of one density."""
    from pathlib import Path
    from smcnuts.model.generated import GeneratedModel
    stan = Path(__file__).resolve().parent / "stan"
    gen = GeneratedModel((stan / "arma_series.stan").read_text(), _arma_data(), "arma_series")
    ref = make_model("arma")
    rng = np.random.default_rng(3)
    N = 4096 + 3
    x = rng.normal(size=(N, 4)) * 0.05 + np.array([0.0, 0.9, 0.0, -1.7])
    r = rng.normal(size=(N, 4))
    sc = metric_scale(4, -0.7, 0.7)
    kg, kr = NUTSProposal(gen, StdNormal(4), 0.01, rng=10), NUTSProposal(ref, StdNormal(4), 0.01, rng=10)
    xr0, _ = kr.rvs(x, r, 1.0)
    gen.set_metric_scale(sc)
    ref.set_metric_scale(sc)
    try:
        kg.iteration = kr.iteration = 0
        xg, _ = kg.rvs(x, r, 1.0)
        xr, _ = kr.rvs(x, r, 1.0)
    finally:
        gen.set_metric_scale(None)
        ref.set_metric_scale(None)
    same = (kg.last["n_leapfrog"] == kr.last["n_leapfrog"]).cpu().numpy()
    assert same.mean() > 0.99, same.mean()
    assert not np.array_equal(xr, xr0)
    np.testing.assert_allclose(xg[same], xr[same], rtol=1e-6, atol=1e-8)


NORMAL_SD = "data { int<lower=1> D; vector<lower=0>[D] sd; } parameters { vector[D] x; } model { x ~ normal(0, sd); }"


@pytest.mark.gpu
def test_generated_model_metric_is_a_change_of_variables():
    """x ~ normal(0, sd) with the metric s is identity-metric NUTS on z = x / s, i.e. the program with sd / s and no
    metric started at z: the same trees up to two roundings of one trajectory.  D = 13: every kernel block of the plug-in
    is one lane per particle, and the metric must cover all 13 coordinates."""
    from smcnuts.model.generated import GeneratedModel
    D, N = 13, 4096 + 7
    rng = np.random.default_rng(13)
    sd = np.exp(rng.uniform(-1.0, 1.0, D))
    s = metric_scale(D)
    a = GeneratedModel(NORMAL_SD, {"D": D, "sd": sd.tolist()}, "normal_sd")
    b = GeneratedModel(NORMAL_SD, {"D": D, "sd": (sd / s).tolist()}, "normal_sd_z")
    x = rng.normal(size=(N, D)) * sd
    r = rng.normal(size=(N, D))
    eps = 0.2 * np.min(sd / s)
    a.set_metric_scale(s)
    try:
        oa = _transition(a, x, r, eps, 1.0, False, 5, 0, max_depth=8)
    finally:
        a.set_metric_scale(None)
    ob = _transition(b, x / s, r, eps, 1.0, False, 5, 0, max_depth=8)
    same = oa["n_leapfrog"] == ob["n_leapfrog"]
    assert same.mean() >= 0.99, same.mean()
    np.testing.assert_allclose(oa["x_new"][same], ob["x_new"][same] * s, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(oa["r_new"][same], ob["r_new"][same], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose((oa["A_new"] + oa["B_new"])[same], (ob["A_new"] + ob["B_new"])[same] -
                               np.sum(np.log(s)), rtol=1e-9, atol=1e-9)    # densities differ by the Jacobian log|S|


def _dirichlet_multinomial():
    from smcnuts.model.generated import GeneratedModel
    from tests.test_stan_codegen import STAN
    alpha = np.array([1.0, 2.0, 0.5, 3.0, 1.5])
    counts = np.array([12, 3, 0, 25, 8])
    m = GeneratedModel((STAN / "dirichlet_multinomial.stan").read_text(),
                       {"K": 5, "alpha": alpha.tolist(), "counts": counts.tolist()}, "dm")
    a = alpha + counts
    a0 = a.sum()
    return m, a / a0, a * (a0 - a) / (a0 ** 2 * (a0 + 1))


@pytest.mark.gpu
def test_dirichlet_multinomial_metric_adaptation_recovers_the_posterior():
    """simplex[K] has dim = K - 1 unconstrained coordinates and constrained_dim = K values: set_metric_scale takes dim
    entries and refuses constrained_dim of them, metric adaptation produces dim entries, and tempered SMC with step-size
    and metric adaptation recovers the exact posterior moments with the tolerances of the unadapted run
    (tests/test_stan_constrained_types.py: means within 4 standard errors, variances within 25 %).

    target_accept = 0.95: the forwards L-kernel weights NUTS moves by the Hamiltonian ratio of the selected point, which
    is exact only for small energy errors.  MEASURED on B200 (seeds 4 / 5 / 6): at the default 0.8 the adapted runs end
    7.2 / 1.9 / 5.5 standard errors from the exact means, and step-size adaptation WITHOUT a metric 3.9 / 4.7 / 4.7 with
    the variances 16-31 % low -- the larger adapted step, not the metric; at 0.95: 3.2 / 1.2 / 2.2, variances >= 95 %."""
    m, exact_mean, exact_var = _dirichlet_multinomial()
    K = m.constrained_dim
    assert m.dim == K - 1 and K == 5
    with pytest.raises(ValueError):
        m.set_metric_scale(np.ones(K))
    assert m.metric_scale is None
    m.set_metric_scale(np.full(K - 1, 0.5))
    m.set_metric_scale(None)
    from smcnuts.smc_sampler import SMCSampler
    s = SMCSampler(K=30, N=1 << 16, target=m, step_size=0.2, sample_proposal=StdNormal(m.dim),
                   momentum_proposal=StdNormal(m.dim), lkernel="forwardsLKernel", tempering=True, rng=4,
                   adapt_step_size=12, adapt_mass_matrix=True, target_accept=0.95)
    s.sample(show_progress=False)
    assert s.metric_scale.shape == (K - 1,) and np.all(s.metric_scale > 0)
    assert m.metric_scale is None and s.phi[-1] == 1.0
    # the adapted step settles once the first metric is in: it grew to 8000x the initial step at acceptance 0 while the
    # dual averaging was restarted at every metric change
    assert np.all(s.step_sizes[2:] < 50 * s.step_sizes[0]), s.step_sizes
    mean, var = s.mean_estimate[-1], s.variance_estimate[-1]
    assert mean.shape == (K,) and abs(mean.sum() - 1.0) <= 1e-12
    se = np.sqrt(var / s.ess[-1])
    assert np.all(np.abs(mean - exact_mean) <= 4 * se), (mean, exact_mean, se)
    np.testing.assert_allclose(var, exact_var, rtol=0.25)


def test_dual_averaging_carries_across_a_metric_change():
    """DualAveragingStepSize.rescale(f) moves the whole averaging state into the new units: every later step size, and
    the averaged one, is f times the one without the change.  At acceptance 0 the step only shrinks."""
    from tests.test_step_size import _adapter_cls
    cls = _adapter_cls()
    acc = np.random.default_rng(3).uniform(0.0, 1.0, 12)
    a, b = cls(0.2, 0.8), cls(0.2, 0.8)
    for i, v in enumerate(acc):
        ea, eb = a.update(v), b.update(v)
        if i == 4:
            eb = b.rescale(3.7)
        f = 3.7 if i >= 4 else 1.0
        assert math.isclose(eb, f * ea, rel_tol=1e-13), i
    assert math.isclose(b.averaged(), 3.7 * a.averaged(), rel_tol=1e-13)
    c = cls(0.2, 0.8)
    steps = [c.update(1.0)] + [c.rescale(1.0) for _ in range(1)]
    for _ in range(8):
        steps.append(c.update(0.0))
        steps.append(c.rescale(1.0))
    assert all(y <= x for x, y in zip(steps[1::2], steps[3::2])), steps     # never grows while every tree diverges


# ------------------------------------------------------------------------------------------------ x <-> z conversion
@pytest.mark.gpu
@pytest.mark.parametrize("D", W_DIMS if torch.cuda.is_available() else [])
def test_scale_rows_every_shape_and_alignment(D):
    """smcb_scale_rows (x * s, x / s; out of place and in place) and smcb_scale_rows_accepted into guarded buffers, views
    misaligned by one double: numpy's correctly rounded products and quotients bit for bit, nothing written outside."""
    rng = np.random.default_rng(D)
    s = metric_scale(D)
    sd = dev.to_device(s)
    for N in W_SIZES:
        x = rng.normal(size=(N, D)) * np.exp(rng.uniform(-20, 20, size=(N, D)))
        acc = (rng.random(N) < 0.6).astype(np.int32)
        keep = rng.normal(size=(N, D))
        for off in (0, 1):
            xd = placed(x, off)
            tag = f"D={D} N={N} off={off}"
            for inverse, want in ((0, x * s), (1, x / s)):
                out, chk = guarded(N * D, off=off)
                _cabi.call("smcb_scale_rows", dev.ptr(xd), N, D, dev.ptr(sd), inverse, dev.ptr(out), dev.stream_ptr())
                chk()
                assert np.array_equal(out.cpu().numpy().reshape(N, D), want), (tag, inverse)
                inplace, chk = guarded(N * D, off=off)
                inplace.copy_(xd.reshape(-1))
                _cabi.call("smcb_scale_rows", dev.ptr(inplace), N, D, dev.ptr(sd), inverse, dev.ptr(inplace),
                           dev.stream_ptr())
                chk()
                assert np.array_equal(inplace.cpu().numpy().reshape(N, D), want), (tag, inverse, "in place")
            z, chk = guarded(N * D, off=off)
            z.copy_(xd.reshape(-1))
            accd, keepd = placed(acc, off, torch.int32), placed(keep, off)
            _cabi.call("smcb_scale_rows_accepted", dev.ptr(z), dev.ptr(accd), dev.ptr(keepd), N, D, dev.ptr(sd),
                       dev.ptr(z), dev.stream_ptr())
            chk()
            want = np.where(acc[:, None] != 0, x * s, keep)
            assert np.array_equal(z.cpu().numpy().reshape(N, D), want), (tag, "accepted")


# ------------------------------------------------------------------------------------------------ validation
@pytest.mark.gpu
@pytest.mark.parametrize("tname", ["arma", "gauss"])
def test_set_metric_scale_refuses_bad_scales_and_keeps_the_metric(tname):
    """0, -0, negative, NaN, +-inf, >= 1e300 entries and a vector of the wrong length are refused, and the metric set
    before stays in force: the next transition is the one that metric gives."""
    from smcnuts._cabi import SmcbError
    m = make_model(tname, **({"dim": 9} if tname == "gauss" else {}))
    D = m.dim
    s = metric_scale(D, -0.7, 0.7)
    rng = np.random.default_rng(1)
    N = 999
    x = rng.normal(size=(N, D)) * 0.1 + (np.array([0.0, 0.9, 0.0, -1.7]) if tname == "arma" else 0.0)
    r = rng.normal(size=(N, D))
    m.set_metric_scale(s)
    try:
        want = _transition(m, x, r, 0.01, 0.8, True, 9, 4, max_depth=6)
        for bad in (0.0, -0.0, -1.0, np.nan, np.inf, -np.inf, 1e300, 1e308):
            for pos in (0, D - 1):
                v = s.copy()
                v[pos] = bad
                with pytest.raises(SmcbError):
                    m.set_metric_scale(v)
                assert np.array_equal(m.metric_scale, s)
        for n in (D - 1, D + 1):
            with pytest.raises(ValueError):
                m.set_metric_scale(np.ones(n))
        got = _transition(m, x, r, 0.01, 0.8, True, 9, 4, max_depth=6)
    finally:
        m.set_metric_scale(None)
    for k in want:
        assert np.array_equal(got[k], want[k], equal_nan=True), k
    m.set_metric_scale(np.full(D, np.nextafter(1e300, 0)))      # the extremes that are accepted
    m.set_metric_scale(np.full(D, 5e-324))
    m.set_metric_scale(None)
