"""GeneratedModel -- any Stan program of the supported subset as a device model (SURVEY.md section 8 f3).

The reference compiles arbitrary Stan programs through BridgeStan (smcnuts/model/bridgestan.py:13-26).  Here
`stan_codegen.generate` translates the program into a model struct, this module wraps it into a plug-in translation
unit (csrc/nuts_plugin.cuh), compiles it with nvcc for sm_100a into smcnuts/_lib/gen/<digest>/model.so and hands it to
the library with smcb_model_create_plugin.  The result has the reference's target API (`dim`, `constrained_dim`,
`param_names`, `logpdf`, `logpdfgrad`, `constrain`) and runs through the same NUTS / SMC kernels as the built-in models.
No CPU fallback: without nvcc or a GPU the constructor raises.
"""
import ctypes
import os
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from .. import _cabi, _device as dev
from . import stan_codegen
from .device_model import DeviceModel

PKG = Path(__file__).resolve().parents[1]
CSRC = PKG.parent / "csrc"
GEN_DIR = PKG / "_lib" / "gen"
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-shared"]


def _csrc_digest():
    """Hash of the kernel headers a plug-in is compiled against: a cached plug-in built against other headers (another
    NutsArgs layout, say) must never be loaded."""
    import hashlib
    h = hashlib.sha256()
    for name in sorted(p.name for p in CSRC.glob("*.cuh")):
        h.update((CSRC / name).read_bytes())
    return h.hexdigest()[:8]


def build_plugin(src: stan_codegen.GeneratedSource, force=False, parity=False):
    """Write and compile the plug-in of a generated model; returns the path of the shared object (cached by the digests of
    the generated text + data and of the kernel headers)."""
    out_dir = GEN_DIR / (f"{src.digest}_{_csrc_digest()}" + ("_parity" if parity else ""))
    so = out_dir / "model.so"
    if so.exists() and not force:
        return so
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).exists():
        raise _cabi.SmcbError("nvcc not found: generated models are compiled at run time (no CPU fallback exists)")
    # built in a private directory and moved into place in one step: several ranks of a sharded run (or several
    # processes) may generate the same model at the same time
    GEN_DIR.mkdir(parents=True, exist_ok=True)
    work = Path(tempfile.mkdtemp(prefix=out_dir.name + ".", dir=GEN_DIR))
    try:
        (work / "model_gen.cuh").write_text(src.text)
        (work / "plugin.cu").write_text(
            "// GENERATED: plug-in translation unit of a Stan-subset model (smcnuts/model/generated.py)\n"
            "#define SMCB_PLUGIN_TU 1\n#include \"nuts_plugin.cuh\"\n#include \"model_gen.cuh\"\n"
            f"SMCB_DEFINE_PLUGIN({src.struct_name})\n")
        flags = NVCC_FLAGS + (["-DSMCB_PARITY=1", "-fmad=false"] if parity else [])
        cmd = [nvcc, *flags, f"-I{CSRC}", f"-I{work}", str(work / "plugin.cu"), "-o", str(work / "model.so")]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise _cabi.SmcbError(f"nvcc failed for the generated model:\n{r.stdout}\n{r.stderr}")
        out_dir.mkdir(parents=True, exist_ok=True)
        for name in ("model_gen.cuh", "plugin.cu"):
            os.replace(work / name, out_dir / name)
        os.replace(work / "model.so", so)          # last: its presence marks the directory as complete
    finally:
        shutil.rmtree(work, ignore_errors=True)
    return so


class GeneratedModel(DeviceModel):
    """Device model generated from a Stan program.  `GeneratedModel(stan_text, data)` or `.from_files(model_path, data_path)`."""

    def __init__(self, stan_text, data=None, name="generated"):
        self.source = stan_codegen.generate(stan_text, data or {})
        self.name = name
        self.dim = self.source.dim
        self.so_path = build_plugin(self.source, parity=_cabi.LIB_PATH.name.endswith("_parity.so"))
        blob = np.ascontiguousarray(self.source.blob, dtype=np.float64)
        h = ctypes.c_void_p()
        dev.device()
        _cabi.call("smcb_model_create_plugin", str(self.so_path).encode(), blob.ctypes.data if blob.size else None, blob.size,
                   ctypes.byref(h))
        self._h = h
        # constrained names in BridgeStan's form (a simplex[K] theta gives theta.1 ... theta.K) and the dim unconstrained ones
        self.param_names = list(self.source.param_names)
        self.param_unc_names = list(self.source.param_unc_names)
        # BridgeStan's constrain() appends transformed parameters and generated quantities (bridgestan.py:24,93-120 of the
        # reference: param_num(include_tp=True, include_gq=True)); here they enter the density (transformed parameters) or
        # are skipped (generated quantities) but are NOT appended: estimates cover the declared parameters only
        self.constrained_dim = _cabi.lib().smcb_model_constrained_dim(self._h)
        assert self.constrained_dim == self.source.cdim, (self.constrained_dim, self.source.cdim)
        kinds = [t[0] for t in self.source.transforms]
        if all(k == "none" for k in kinds):
            self.constrain_kind = _cabi.CONSTRAIN_NONE
        elif kinds[-1] == "lower" and self.source.transforms[-1][1] == 0.0 and all(k == "none" for k in kinds[:-1]):
            self.constrain_kind = _cabi.CONSTRAIN_EXP_LAST       # the fused exp-on-last moments of the built-in models
        else:
            self.constrain_kind = _cabi.CONSTRAIN_MODEL

    @classmethod
    def from_files(cls, model_path, data_path=None, name=None):
        return cls(Path(model_path).read_text(), stan_codegen.load_data(data_path), name or Path(model_path).stem)

    def constrain(self, x, include_tparams=True, include_gqs=True):
        """Stan's constraining transforms of the declared parameters (bridgestan.py:93-120): [..., dim] -> [...,
        constrained_dim], one kernel of the model's plug-in for the whole particle array; `include_tparams` /
        `include_gqs` are accepted and ignored (see __init__)."""
        xd = dev.to_device(x).reshape(-1, self.dim).contiguous()
        out = dev.empty(xd.shape[0], self.constrained_dim)
        _cabi.call("smcb_model_constrain", self._h, dev.ptr(xd), xd.shape[0], dev.ptr(out), dev.stream_ptr())
        shape = tuple(np.shape(x)[:-1]) + (self.constrained_dim,)
        if dev.is_host(x):
            return dev.to_numpy(out).reshape(shape)
        return out.reshape(shape)
