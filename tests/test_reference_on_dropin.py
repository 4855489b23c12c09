"""The reference's own call sequence on the drop-in shims, on the GPU -- the check behind INTEGRATION.md section 1.
parameters.py:108-114 loads `os.getcwd() + "/C/nlplant_xcg25.so"`; the test gives a child process a working directory whose C/
is f16_mpc_oop_py_b200/dropin/C and has the oracle's restatement of env.py (the same restatement that reproduces the
reference's own results bit for bit on the CPU, tests/test_oracle.py::test_golden_env_py) call the shim found there for
every Nlplant / atmos: trim with Nelder-Mead, _calc_xdot, linearise, 2000 F16.step calls, _calc_xdot_na and
_calc_LQR_gain().  The results are compared with tests/golden: the same calls made by the unmodified reference on its
shipped CPU .so (tools/gen_golden.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import REPO, load_golden

pytestmark = pytest.mark.gpu

DROPIN = os.path.join(REPO, "f16_mpc_oop_py_b200", "dropin", "C")


@pytest.mark.parametrize("tag", ["xcg25", "xcg35", "lofi_xcg25"])
def test_reference_call_sequence_on_the_dropin(tmp_path, tag):
    os.symlink(DROPIN, tmp_path / "C")
    out = tmp_path / "out.npz"
    env = dict(os.environ, F16_MATH="strict")
    r = subprocess.run([sys.executable, os.path.join(REPO, "tests", "_run_reference_calls_on_dropin.py"), REPO, str(tmp_path), tag,
                        str(out)], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    o, g = np.load(out), load_golden(tag)
    # it really was our library: the shim under <cwd>/C and libf16_b200.so are mapped, no other Nlplant
    loaded = [str(s) for s in o["loaded"]]
    assert any("libf16_b200.so" in s for s in loaded) and any("dropin/C/nlplant_xcg" in s for s in loaded), loaded
    assert all("libf16_b200.so" in s or "dropin/C/nlplant_xcg" in s for s in loaded), loaded

    def rel(a, b, floor):
        return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))

    # derivative calls at the golden points: the 1e-12 bar (scaled: a derivative that cancels to ~0 is measured against 1e-3)
    assert rel(o["xdot_trim"], g["xdot_trim"], 1e-3) < 1e-12
    assert rel(o["xdots"], g["xdots"], 1e-3) < 1e-12
    assert rel(o["na_xdots"], g["na_xdots"], 1e-3) < 1e-12
    # F16.linearise at the golden trim point (forward differences, eps 1e-5): the 1e-8 bar
    assert np.abs(o["Ac"] - g["Ac"]).max() < 1e-8 and np.abs(o["Bc"] - g["Bc"]).max() < 1e-8
    # 2000 calls of F16.step from the golden trim: the 1e-9 bar
    assert rel(o["traj_x"], g["traj_x"], 1e-3) < 1e-9
    # trim(10000, 700) by Nelder-Mead over our Nlplant: the search is chaotic in the last bits of the objective, so the
    # optimiser's point is pinned to the reference's by position (the tolerance the reference's own xatol gives: 1e-10 on the
    # unknowns is not reachable across libm builds) -- 1e-5 of each state's natural size
    scale = np.array([1, 1, 1e4, 1, 1, 1, 700, 0.1, 0.1, 1, 1, 1, 3e3, 1, 1, 1, 1, 1.0])
    assert np.max(np.abs(o["x_trim"] - g["x_trim"]) / scale) < 1e-5
    # _calc_LQR_gain(): reduced model + cont2discrete + DARE over our derivatives
    assert rel(o["K_lqr"], g["K_lqr"], 1e-2 * np.abs(g["K_lqr"]).max()) < 1e-6
