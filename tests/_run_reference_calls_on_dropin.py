"""Child process of tests/test_reference_on_dropin.py: the calls the reference's F16 makes (trim, _calc_xdot, linearise,
2000 step calls, _calc_xdot_na, _calc_LQR_gain) replayed by the oracle's restatement of env.py, with every Nlplant / atmos
call going to the drop-in shim that parameters.py would load from `<cwd>/C/` (f16_mpc_oop_py_b200/dropin/C), i.e. to the
B200.  Writes what it computed to an .npz for the parent to compare with tests/golden (the same calls of the reference).

    python _run_reference_calls_on_dropin.py <repo> <workdir> <tag> <out.npz>
"""
import os
import sys

import numpy as np

repo, workdir, tag, out = sys.argv[1:5]
sys.dont_write_bytecode = True
sys.path.insert(0, repo)
from oracle import NA_COLS, NA_ROWS, NA_UCOLS, REF, Oracle, discretise, dlqr, reduce_jacobian  # noqa: E402

golden = np.load(os.path.join(repo, "tests", "golden", f"env_{tag}.npz"))
fi, xcg = int(golden["fi"]), float(golden["xcg"])
os.chdir(workdir)                                  # parameters.py resolves os.getcwd() + "/C/nlplant_xcg25.so"
o = Oracle()
so = os.path.join("C", "nlplant_xcg35.so" if xcg == 0.35 else "nlplant_xcg25.so")
rc = o.lib.orc_ref_open(so.encode(), workdir.encode(), xcg)   # the shim in place of the reference's own .so
if rc != 0:
    sys.exit(f"orc_ref_open({so}) failed: {rc}")
loaded = [l.split()[-1] for l in open("/proc/self/maps") if "nlplant_xcg" in l or "libf16_b200" in l]


def col(v):
    return np.ascontiguousarray(np.asarray(v, dtype=np.float64).reshape(-1, 1))


x_trim, info, st = o.trim(10000, 700, fi, xcg, backend=REF)    # F16.trim(10000, 700): Nelder-Mead over the shim's Nlplant
assert st == 0 and info["converged"], (st, info)
# from here on at the GOLDEN trim point, so that every comparison is of the same function at the same argument
gx, gu = golden["x_trim"], golden["u_trim"]
xdot_trim, st = o.calc_xdot_batch(col(gx), col(gu), fi, xcg, REF)
assert not st.any()
A, B, st = o.linearise_batch(col(gx), col(gu), 1e-5, 0, fi, xcg, REF)
assert not st.any()
xdots, st = o.calc_xdot_batch(golden["xs"].T.copy(), golden["us"].T.copy(), fi, xcg, REF)
assert not st.any()
traj, x = [gx.copy()], col(gx)
for k in range(4):                                 # 4 x 500 F16.step calls, open loop
    x, st = o.step_batch(x, col(gu), 500, 0.001, fi, xcg, None, REF)
    assert not st.any()
    traj.append(x[:, 0].copy())
# _calc_xdot_na: the mpc states and inputs written into the trim state (inputs into the actuator states too), rows NA_ROWS
n = len(golden["na_x"])
xn, un = np.repeat(gx[:, None], n, 1), np.repeat(gu[:, None], n, 1)
xn[NA_COLS], xn[NA_UCOLS], un[1:] = golden["na_x"].T, golden["na_u"].T, golden["na_u"].T
na_xdots, st = o.calc_xdot_batch(xn, un, fi, xcg, REF)
assert not st.any()
# _calc_LQR_gain(): reduced model + cont2discrete + DARE over the shim's Jacobian
Ana, Bna = reduce_jacobian(A[0])
K, _ = dlqr(*discretise(Ana, Bna, 0.001), np.eye(9), np.eye(3))
np.savez(out, x_trim=x_trim, xdot_trim=xdot_trim[:, 0], Ac=A[0], Bc=B[0], xdots=xdots.T, traj_x=np.array(traj), K_lqr=-K,
         na_xdots=na_xdots[NA_ROWS].T, loaded=np.array(loaded))
