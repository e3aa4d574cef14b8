"""ctypes wrapper for tests/hostsim/hostsim.cpp (CPU simulation of the device lanes; test tool only)."""
import ctypes
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)
_LIBS = {}


def lib(devmath=False):
    """devmath=True: the build with -DSMCB_DEVMATH, in which exp / log are the table-driven device algorithms restated
    for the host (csrc/common.cuh) -- the CPU twin of the parity device build (libsmcnuts_b200_parity.so)."""
    if devmath not in _LIBS:
        so = HERE / ("_hostsim_devmath.so" if devmath else "_hostsim.so")
        src = HERE / "hostsim.cpp"
        hdrs = list((HERE.parents[1] / "smc-nuts_b200" / "csrc").glob("*.cuh"))
        if not so.exists() or so.stat().st_mtime < max(p.stat().st_mtime for p in [src] + hdrs):
            subprocess.run(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas",
                            *(["-DSMCB_DEVMATH=1"] if devmath else []), "-o", str(so), str(src)], check=True)
        _LIBS[devmath] = ctypes.CDLL(str(so))
    return _LIBS[devmath]


_LIB_SIMT = None


def lib_simt():
    """The warp-emulated build (hostsim_simt.cpp + simt_emu.h): group kernels with shuffles / votes / mma on fibers."""
    global _LIB_SIMT
    if _LIB_SIMT is None:
        so = HERE / "_hostsim_simt.so"
        srcs = [HERE / "hostsim_simt.cpp", HERE / "simt_emu.h"]
        hdrs = list((HERE.parents[1] / "smc-nuts_b200" / "csrc").glob("*.cuh"))
        if not so.exists() or so.stat().st_mtime < max(p.stat().st_mtime for p in srcs + hdrs):
            subprocess.run(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas",
                            "-o", str(so), str(srcs[0])], check=True)
        _LIB_SIMT = ctypes.CDLL(str(so))
    return _LIB_SIMT


def pack_model(name, np_target):
    """Host blob -> (kind, packed data, dim, T, q) in the device layout of csrc/models.cuh."""
    if name == "arma":
        return 0, np.ascontiguousarray(np_target.y), 4, len(np_target.y), 0.0
    if name == "PRMwCD":
        t = np_target
        rows = np.zeros((t.Nobs, 12))
        rows[:, :11] = t.X
        rows[:, 11] = t.y
        hdr = np.zeros(16)
        for i in range(t.Nobs):          # same accumulation order as smcb_model_create
            hdr[0] += t.y[i]
            hdr[1:12] += t.y[i] * t.X[i]
            hdr[12] += t.lgam[i]
        return 1, np.ascontiguousarray(np.concatenate([hdr, rows.ravel()])), 13, t.Nobs, t.q
    return 2, np.ascontiguousarray(np_target.P.ravel()), np_target.dim, 0, 0.0


def _to_z(x, scale):
    """Diagonal metric: the lanes run on z = x / scale (proposal/nuts.py converts with smcb_scale_rows)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    if scale is None:
        return x, None
    scale = np.ascontiguousarray(scale, dtype=np.float64)
    return np.ascontiguousarray(x / scale), scale


def _to_x(o, x, scale):
    """Back to x-space as proposal/nuts.py does: x_new = z_new * scale, except that a particle the MH epilogue rejected
    keeps its x row (smcb_scale_rows_accepted)."""
    if scale is not None:
        o["x_new"] = np.where(o["accepted"][:, None] != 0, o["x_new"] * scale, x)
    return o


def nuts(name, np_target, x, r, eps, phi, max_depth=10, accrej=False, seed=0, iteration=0, particle0=0, lanes=32,
         carry=None, want_grad=False, devmath=False, scale=None):
    """One NUTS transition per particle on the one-lane kernels.  scale: diagonal metric (ScaledModel); x and x_new are
    then x-space rows, converted as proposal/nuts.py converts them."""
    kind, data, dim, T, q = pack_model(name, np_target)
    x_in = np.ascontiguousarray(x, dtype=np.float64)
    x, scale = _to_z(x_in, scale)
    r = np.ascontiguousarray(r, dtype=np.float64)
    N = len(x)
    o = dict(x_new=np.empty_like(x), r_new=np.empty_like(r), A_old=np.empty(N), B_old=np.empty(N), A_new=np.empty(N),
             B_new=np.empty(N), ke_old=np.empty(N), ke_new=np.empty(N), n_leapfrog=np.empty(N, dtype=np.int32),
             accepted=np.empty(N, dtype=np.int32), depth=np.empty(N, dtype=np.int32))
    if want_grad:
        o["g_new"] = np.empty_like(x)
    cA, cB, cg = (np.ascontiguousarray(c, dtype=np.float64) for c in carry) if carry is not None else (None, None, None)
    P = lambda a: a.ctypes.data_as(_dp) if a is not None else None  # noqa: E731
    I = lambda a: a.ctypes.data_as(_ip)  # noqa: E731
    lib(devmath).hostsim_nuts(ctypes.c_int(kind), P(data), ctypes.c_int(data.size), ctypes.c_int(dim), ctypes.c_int(T),
                       ctypes.c_double(q), P(x), P(r), ctypes.c_longlong(N), ctypes.c_double(eps), ctypes.c_double(phi),
                       ctypes.c_int(max_depth), ctypes.c_int(int(accrej)), ctypes.c_ulonglong(seed),
                       ctypes.c_uint(iteration), ctypes.c_ulonglong(particle0), P(o["x_new"]), P(o["r_new"]),
                       P(o["A_old"]), P(o["B_old"]), P(o["A_new"]), P(o["B_new"]), P(o["ke_old"]), P(o["ke_new"]),
                       I(o["n_leapfrog"]), I(o["accepted"]), I(o["depth"]), P(cA), P(cB), P(cg), P(o.get("g_new")),
                       ctypes.c_int(lanes), P(scale))
    return _to_x(o, x_in, scale)


def nuts_simt(name, np_target, x, r, eps, phi, max_depth=10, accrej=False, seed=0, iteration=0, particle0=0, scale=None):
    """One NUTS transition per particle on the EMULATED 4-lanes-per-particle kernels (PRMwCD: PrmModelG<13>; gauss:
    GaussModelG<ceil(D/8)>), one persistent warp pulling particles from the work queue.  scale: as in nuts()."""
    kind, data, dim, T, q = pack_model(name, np_target)
    assert kind in (1, 2)
    x_in = np.ascontiguousarray(x, dtype=np.float64)
    x, scale = _to_z(x_in, scale)
    r = np.ascontiguousarray(r, dtype=np.float64)
    N = len(x)
    o = dict(x_new=np.empty_like(x), r_new=np.empty_like(r), A_old=np.empty(N), B_old=np.empty(N), A_new=np.empty(N),
             B_new=np.empty(N), ke_old=np.empty(N), ke_new=np.empty(N), n_leapfrog=np.empty(N, dtype=np.int32),
             accepted=np.empty(N, dtype=np.int32), depth=np.empty(N, dtype=np.int32))
    P = lambda a: a.ctypes.data_as(_dp) if a is not None else None  # noqa: E731
    I = lambda a: a.ctypes.data_as(_ip)  # noqa: E731
    rc = lib_simt().hostsim_nuts_simt(
        ctypes.c_int(kind), P(data), ctypes.c_int(data.size), ctypes.c_int(dim), ctypes.c_int(T), ctypes.c_double(q), P(x),
        P(r), ctypes.c_longlong(N), ctypes.c_double(eps), ctypes.c_double(phi), ctypes.c_int(max_depth),
        ctypes.c_int(int(accrej)), ctypes.c_ulonglong(seed), ctypes.c_uint(iteration), ctypes.c_ulonglong(particle0),
        P(o["x_new"]), P(o["r_new"]), P(o["A_old"]), P(o["B_old"]), P(o["A_new"]), P(o["B_new"]), P(o["ke_old"]),
        P(o["ke_new"]), I(o["n_leapfrog"]), I(o["accepted"]), I(o["depth"]), P(scale))
    assert rc == 0
    return _to_x(o, x_in, scale)


def scaled_probe(group, nloc, dim, scale, z):
    """ScaledModel<probe>::eval on one emulated warp: z[32, nloc] slot values -> g[32, nloc] = s * (s * z) per slot, where
    the probe model returns the x it sees as its gradient (hostsim_simt.cpp)."""
    scale = np.ascontiguousarray(scale, dtype=np.float64)
    z = np.ascontiguousarray(z, dtype=np.float64).reshape(32, nloc)
    g = np.empty_like(z)
    rc = lib_simt().hostsim_scaled_probe(ctypes.c_int(group), ctypes.c_int(nloc), ctypes.c_int(dim),
                                         scale.ctypes.data_as(_dp), z.ctypes.data_as(_dp), g.ctypes.data_as(_dp))
    assert rc == 0
    return g


_LIB_BISECT = None


def bisect(f, xa, xb):
    """The device bisection walk (csrc/bisect.cuh compiled with g++) on a Python objective f(array) -> array.
    Returns (root, status, iterations, nan_at, passes)."""
    global _LIB_BISECT
    if _LIB_BISECT is None:
        so, src = HERE / "_hostsim_bisect.so", HERE / "hostsim_bisect.cpp"
        hdrs = list((HERE.parents[1] / "smc-nuts_b200" / "csrc").glob("*.cuh"))
        if not so.exists() or so.stat().st_mtime < max(p.stat().st_mtime for p in [src] + hdrs):
            subprocess.run(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas",
                            "-o", str(so), str(src)], check=True)
        _LIB_BISECT = ctypes.CDLL(str(so))
    cb_t = ctypes.CFUNCTYPE(None, _dp, ctypes.c_int, _dp)

    def cb(xp, m, fp):
        vals = np.asarray(f(np.array([xp[i] for i in range(m)])), dtype=np.float64)
        for i in range(m):
            fp[i] = vals[i]
    out = (ctypes.c_double * 4)()
    passes = _LIB_BISECT.hostsim_bisect(ctypes.c_double(xa), ctypes.c_double(xb), cb_t(cb), out, None)
    return out[0], int(out[1]), int(out[2]), out[3], passes
