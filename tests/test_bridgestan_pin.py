"""Pins the model arithmetic against Stan itself WHEN BridgeStan is importable (SURVEY.md section 8 f3); skipped in the
offline build image, where the package cannot be installed -- DESIGN.md section 6 then reads "parity unpinned against
BridgeStan" and the three independent restatements stand in.  CPU only: oracle densities and the g++ build of the generated
model structs against `bridgestan.StanModel.log_density[_gradient]`, evaluated the way the reference does
(smcnuts/model/bridgestan.py:46,78 of the reference)."""
import json
from pathlib import Path

import numpy as np
import pytest

from oracle import bridgestan_target as BT
from oracle import smc_oracle as O

ROOT = Path(__file__).resolve().parents[1]
STAN = ROOT / "tests" / "stan"
REF_STAN = ROOT / "tests" / "golden" / "reference_stan"
DATA = ROOT / "smc-nuts_b200" / "smcnuts" / "data"

pytestmark = pytest.mark.skipif(not BT.available(), reason="bridgestan is not installed (offline image)")


def _data(name):
    raw = (DATA / name / f"{name}.json").read_text()
    try:
        d = json.loads(raw)
    except json.JSONDecodeError:
        d = json.loads(raw + " 1.0}")
    return d


def _programs(name):
    out = [STAN / {"arma": "arma_series.stan", "PRMwCD": "prm_kernel.stan"}[name]]
    if (REF_STAN / f"{name}.stan").exists():
        out.append(REF_STAN / f"{name}.stan")       # the original project's own text, where it is stored
    return out


@pytest.mark.parametrize("name", ["arma", "PRMwCD"])
def test_oracle_densities_equal_bridgestan(name):
    t = O.COracleTarget(name)
    x = np.random.default_rng(1).normal(size=(64, t.dim)) * 0.5
    for prog in _programs(name):
        b = BT.BridgeStanTarget(prog, _data(name))
        assert b.dim == t.dim
        A, B = b.split(x)
        Ao, Bo, _, _ = t.split(x, grads=False)
        np.testing.assert_allclose(A, Ao, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(B, Bo, rtol=1e-12, atol=1e-10)
        for phi in (0.0, 0.37, 1.0):
            np.testing.assert_allclose(b.logpdfgrad(x, phi), t.logpdfgrad(x, phi), rtol=1e-9, atol=1e-8)


@pytest.mark.parametrize("fixture", ["regression", "containers", "logistic", "mixed"])
def test_generated_models_equal_bridgestan(tmp_path, fixture):
    """The Stan-subset generator against Stan itself on the fixtures of tests/stan (values and gradients)."""
    import sys
    sys.path.insert(0, str(Path(__file__).resolve().parent))
    import test_stan_codegen as T
    rng = np.random.default_rng(11)
    data = {"regression": lambda: T._regression_data(rng), "containers": lambda: T._containers_data(rng, 1),
            "logistic": lambda: T._logistic_data(rng),
            "mixed": lambda: {"N": 12, "t": rng.normal(size=12).tolist(), "y": rng.lognormal(size=12).tolist(),
                              "k": rng.integers(0, 6, 12).tolist()}}[fixture]()
    src = T.SC.generate((STAN / f"{fixture}.stan").read_text(), data)
    h = T.HostModel(src, tmp_path)
    b = BT.BridgeStanTarget(STAN / f"{fixture}.stan", data)
    assert b.dim == src.dim
    x = rng.normal(size=(32, src.dim)) * 0.5
    for phi in (0.0, 0.45, 1.0):
        A, B, g = h.split(x, phi)
        # `~` statements: the generator drops parameter-free terms term by term, which is what Stan's propto does and what
        # BridgeStan's log_density defaults to; the comparison still allows one additive constant per phi in case a
        # BridgeStan version defaults the other way -- a constant does not move a sampler
        lp = b.logpdf(x, phi)
        d = (A + phi * B) - lp
        np.testing.assert_allclose(d, d[0], rtol=0, atol=1e-9)
        np.testing.assert_allclose(g, b.logpdfgrad(x, phi), rtol=1e-9, atol=1e-8)
