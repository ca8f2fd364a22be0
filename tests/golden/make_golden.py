#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the REAL reference modules.

Run in the build container only (needs /root/reference; the GPU box has no copy):
    python tests/golden/make_golden.py

The reference cannot be imported as-is here (SURVEY §8c): ``osqp``/``cvxopt`` are
absent and two lines are incompatible with Python 3.12 / NumPy 2.x.  This script
  * installs in-memory stubs: ``cvxopt.solvers.qp(Q,b)`` -> ``numpy.linalg.solve(Q,-b)``
    (what an unconstrained cvxopt qp computes) and ``osqp.OSQP`` -> oracle/osqp_port
    driven to 1e-9 (so the closed loop follows the exact QP optimum);
  * patches two source lines IN MEMORY (nothing is written to /root/reference):
      PredictiveControllers.py:33   ndarray dataclass default  -> None
      PredictiveControllers.py:502  ``self.xPred == []``       -> list-emptiness test
  * drives the reference classes exactly like src/main.py:39-120 (N=12 instead of 14,
    BASELINE.json's horizon) with ``np.random.seed(0)``, running the oracle restatement
    in lock-step on the same inputs and asserting agreement at every step;
  * stores full-state snapshots at selected steps so that the tests can replay single
    steps without the reference.
"""
import os
import sys
import types
import importlib.util
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "support"))
REF = "/root/reference/src"
OUT = os.path.dirname(os.path.abspath(__file__))

from oracle import osqp_port, ftocp, vehicle, ltv_model   # noqa: E402
from oracle.track import TrackTable                       # noqa: E402
import golden_file                                        # noqa: E402


# ------------------------------------------------------------------ stubs
def install_stubs():
    cv = types.ModuleType("cvxopt")
    sol = types.ModuleType("cvxopt.solvers")
    sol.options = {}

    def qp(Q, b):
        return {"x": np.linalg.solve(np.asarray(Q), -np.asarray(b)).reshape(-1, 1)}
    sol.qp = qp
    cv.solvers = sol
    cv.matrix = lambda a: np.asarray(a, dtype=float)
    cv.spmatrix = None
    sys.modules["cvxopt"] = cv
    sys.modules["cvxopt.solvers"] = sol

    om = types.ModuleType("osqp")

    class OSQP:
        def setup(self, P=None, q=None, A=None, l=None, u=None, **kw):
            self.args = (P, q, A, l, u)

        def warm_start(self, x=None):
            pass

        def solve(self):
            P, q, A, l, u = self.args
            x, info, y = osqp_port.solve(P, q, A, l, u, eps_abs=1e-9, eps_rel=1e-9, max_iter=400000, polish_strict=1)
            res = types.SimpleNamespace()
            res.x = x
            res.y = y
            res.info = types.SimpleNamespace(status_val=1 if info["status"] == 1 else 2, iter=info["iters"])
            return res
    om.OSQP = OSQP
    sys.modules["osqp"] = om


def load_patched(name, path, patches):
    src = open(path).read()
    for old, new in patches:
        assert old in src, (name, old)
        src = src.replace(old, new)
    mod = types.ModuleType(name)
    mod.__file__ = path
    sys.modules[name] = mod
    exec(compile(src, path, "exec"), mod.__dict__)
    return mod


def load_reference():
    install_stubs()
    for sub in ("fnc/simulator", "fnc/controller", "fnc", ""):
        sys.path.append(os.path.join(REF, sub))
    PC = load_patched("PredictiveControllers", os.path.join(REF, "fnc/controller/PredictiveControllers.py"), [
        ("Q: np.array = field(default=np.array((n, n)))", "Q: np.array = field(default=None)"),
        ("if self.xPred == []:", "if isinstance(self.xPred, list) and len(self.xPred) == 0:"),
    ])
    import PredictiveModel as PM
    import Utilities as UT
    import SysModel as SM
    import Track as TR
    import initControllerParameters as IP
    return PC, PM, UT, SM, TR, IP


def qp_of(ctrl, x0):
    """The OSQP-form data the reference hands to the solver (PC.py:124,270-273)."""
    P = np.asarray(ctrl.H_FTOCP.todense())
    F = np.asarray(ctrl.F_FTOCP.todense())
    G = np.asarray(ctrl.G_FTOCP.todense())
    beq = np.add(np.dot(ctrl.E_FTOCP, x0), ctrl.L_FTOCP)
    return ftocp.osqp_form(P, np.asarray(ctrl.q_FTOCP).ravel(), F, ctrl.b_FTOCP, G, beq)


def close(a, b, tol, what):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    fin = np.isfinite(a)
    assert np.array_equal(fin, np.isfinite(b)), what
    err = np.max(np.abs(a[fin] - b[fin])) if fin.any() else 0.0
    assert err <= tol, (what, err)
    return err


def lmpc_state(c, pm):
    """Everything needed to replay one LMPC.solve() on a fresh oracle object."""
    d = dict(it=c.it, timeStep=c.timeStep, zt=np.array(c.zt), xLin=np.array(c.xLin), uLin=np.array(c.uLin),
             OldInput=np.array(c.OldInput), LapTime=np.array(c.LapTime), nlap=len(c.SS),
             has_pred=0 if isinstance(c.xPred, list) else 1,
             xPred_prev=np.zeros((c.N + 1, c.n)) if isinstance(c.xPred, list) else np.array(c.xPred),
             pm_nlap=len(pm.xStored))
    for j in range(len(c.SS)):
        d["SS%d" % j], d["uSS%d" % j], d["Qfun%d" % j] = np.array(c.SS[j]), np.array(c.uSS[j]), np.array(c.Qfun[j])
    for j in range(len(pm.xStored)):
        d["pmx%d" % j], d["pmu%d" % j] = np.array(pm.xStored[j]), np.array(pm.uStored[j])
    return d


def main():
    N = 12
    PC, PM, UT, SM, TR, IP = load_reference()
    gold = {}

    # ---- track ------------------------------------------------------------------
    rmap = TR.Map(0.4)
    omap = TrackTable(0.4)
    assert np.array_equal(rmap.PointAndTangent, omap.PointAndTangent)
    assert rmap.TrackLength == omap.TrackLength
    s_probe = np.concatenate([np.linspace(0, 3 * rmap.TrackLength, 400)[:-1], rmap.PointAndTangent[:, 3],
                              rmap.PointAndTangent[:, 3] + 1e-12])
    s_probe = s_probe[(s_probe % rmap.TrackLength) != 0.0] if False else s_probe
    curv = []
    for s in s_probe:
        try:
            curv.append(rmap.curvature(s))
        except Exception:
            curv.append(np.nan)
    curv = np.array(curv)
    ocurv = []
    for s in s_probe:
        try:
            ocurv.append(omap.curvature(s))
        except Exception:
            ocurv.append(np.nan)
    assert np.array_equal(np.isnan(curv), np.isnan(np.array(ocurv)))
    assert np.array_equal(curv[~np.isnan(curv)], np.array(ocurv)[~np.isnan(curv)])
    gold["track_table"], gold["track_length"] = rmap.PointAndTangent, np.array(rmap.TrackLength)
    gold["curv_s"], gold["curv_val"] = s_probe, curv

    # ---- PID lap (main.py:45-66) ------------------------------------------------
    x0 = np.array([0.5, 0, 0, 0, 0, 0])
    xS = [x0, x0]
    np.random.seed(0)
    xP, uP, gP, _ = SM.Simulator(rmap).sim(xS, UT.PID(0.8))
    np.random.seed(0)
    oxP, ouP, ogP, _ = vehicle.closed_loop(omap, xS, vehicle.PIDFollower(0.8))
    assert np.array_equal(xP, oxP) and np.array_equal(uP, ouP) and np.array_equal(gP, ogP)
    gold["pid_x"], gold["pid_u"], gold["pid_glob"] = xP, uP, gP
    rng_after_pid = np.random.get_state()

    # ---- LTI sys-id + LTI MPC (main.py:72-80) -----------------------------------
    A, B, _ = UT.Regression(xP, uP, 1e-7)
    oA, oB, _ = vehicle.ridge_sysid(xP, uP, 1e-7)
    assert np.array_equal(A, oA) and np.array_equal(B, oB)
    gold["lti_A"], gold["lti_B"] = A, B
    mpcParam, ltvParam = IP.initMPCParams(6, 2, N, 0.8)
    omp, oltv = ftocp.mpc_params(6, 2, N, 0.8)
    mpcParam.A, mpcParam.B = A, B
    omp.A, omp.B = A, B
    rmpc = PC.MPC(mpcParam)
    ompc = ftocp.OracleMPC(omp, qp=osqp_port.tight_qp)
    xs = [x0]
    gs = [x0]
    worst = 0.0
    for t in range(30):
        rmpc.solve(xs[-1])
        ompc.solve(xs[-1])
        rq, oq = qp_of(rmpc, xs[-1]), ompc.last_qp
        for a, b, nm in zip(rq, oq, "PqAlu"):
            worst = max(worst, close(a, b, 1e-13, "lti " + nm))
        worst = max(worst, close(rmpc.uPred, ompc.uPred, 1e-9, "lti uPred"))
        if t in (0, 7):
            for a, nm in zip(rq, "PqAlu"):
                gold["lti_t%d_qp_%s" % (t, nm)] = a
            gold["lti_t%d_x0" % t], gold["lti_t%d_old" % t] = xs[-1], np.zeros(2) if t == 0 else prev_u
            gold["lti_t%d_xPred" % t], gold["lti_t%d_uPred" % t] = rmpc.xPred, rmpc.uPred
        prev_u = rmpc.uPred[0].copy()
        xt, gt = vehicle.dyn_model(omap, xs[-1], gs[-1], rmpc.uPred[0])
        xs.append(xt)
        gs.append(gt)
    print("LTI-MPC lock-step 30 steps: max |diff| =", worst)

    # ---- LTV MPC (main.py:86-94) ------------------------------------------------
    rpm = PM.PredictiveModel(6, 2, rmap, 1)
    rpm.addTrajectory(xP, uP)
    opm = ltv_model.LocalLTVModel(6, 2, omap, 1)
    opm.addTrajectory(xP, uP)
    ltvParam.timeVarying = True
    oltv.timeVarying = True
    rltv = PC.MPC(ltvParam, rpm)
    oltvc = ftocp.OracleMPC(oltv, opm, qp=osqp_port.tight_qp)
    xs, gs = [x0], [x0]
    worst = 0.0
    for t in range(40):
        pre = dict(xLin=np.array(rltv.xLin), uLin=np.array(rltv.uLin), old=np.array(rltv.OldInput).ravel())
        rltv.solve(xs[-1])
        oltvc.solve(xs[-1])
        for a, b, nm in zip(qp_of(rltv, xs[-1]), oltvc.last_qp, "PqAlu"):
            worst = max(worst, close(a, b, 1e-12, "ltv " + nm))
        worst = max(worst, close(np.array(rltv.A), np.array(oltvc.A), 1e-12, "ltv A"))
        worst = max(worst, close(rltv.uPred, oltvc.uPred, 1e-8, "ltv uPred"))
        if t in (0, 1, 20):
            k = "ltv_t%d_" % t
            gold[k + "xLin"], gold[k + "uLin"], gold[k + "old"], gold[k + "x0"] = pre["xLin"], pre["uLin"], pre["old"], xs[-1]
            gold[k + "A"], gold[k + "B"], gold[k + "C"] = np.array(rltv.A), np.array(rltv.B), np.array(rltv.C)
            for a, nm in zip(qp_of(rltv, xs[-1]), "PqAlu"):
                gold[k + "qp_" + nm] = a
            gold[k + "xPred"], gold[k + "uPred"] = rltv.xPred, rltv.uPred
        xt, gt = vehicle.dyn_model(omap, xs[-1], gs[-1], rltv.uPred[0])
        xs.append(xt)
        gs.append(gt)
    print("LTV-MPC lock-step 40 steps: max |diff| =", worst)

    # k-NN indices for a few probe queries on the PID lap (PM.py:180-197)
    rng = np.random.default_rng(5)
    probes = np.hstack((xP[rng.integers(0, 990, 24)][:, [0, 1, 2]], uP[rng.integers(0, 990, 24)])) + rng.normal(0, 0.02, (24, 5))
    idx = np.array([rpm.computeIndices(p, 0)[0] for p in probes])
    Kw = np.array([rpm.computeIndices(p, 0)[1] for p in probes])
    oidx = np.array([opm.knn(p, 0)[0] for p in probes])
    assert np.array_equal(idx, oidx)
    gold["knn_probe"], gold["knn_idx"], gold["knn_K"] = probes, idx, Kw

    # ---- LMPC (main.py:99-120) --------------------------------------------------
    # The reference stores the SAME xPID array object in all four safe-set slots and in the
    # regression model; its first solve mutates that array through the xLin view (PC.py:394,432).
    # Work on copies so the PID golden above stays pristine, but keep the aliasing.
    numSS_it, numSS_Points, Laps, _, Qts, lmpcPar = IP.initLMPCParams(rmap, N)
    _, _, _, _, oQts, olmpcPar = ftocp.lmpc_params(omap, N)
    lmpcPar.timeVarying = True
    olmpcPar.timeVarying = True
    rx, ru, rg = xP.copy(), uP.copy(), gP.copy()
    ox, ou, og = xP.copy(), uP.copy(), gP.copy()
    rpm4 = PM.PredictiveModel(6, 2, rmap, 4)
    opm4 = ltv_model.LocalLTVModel(6, 2, omap, 4)
    for _ in range(4):
        rpm4.addTrajectory(rx, ru)
        opm4.addTrajectory(ox, ou)
    rl = PC.LMPC(numSS_Points, numSS_it, Qts, lmpcPar, rpm4)
    ol = ftocp.OracleLMPC(numSS_Points, numSS_it, oQts, olmpcPar, opm4, qp=osqp_port.tight_qp)
    for _ in range(4):
        rl.addTrajectory(rx, ru, rg)
        ol.addTrajectory(ox, ou, og)
    close(np.array(rl.Qfun[0]), np.array(ol.Qfun[0]), 0, "Qfun")
    gold["pid_Qfun"] = np.array(rl.Qfun[0])

    np.random.set_state(rng_after_pid)
    xS_lap = [x0, x0]
    snaps = {(4, 0), (4, 1), (4, 60), (4, 200), (5, 0), (5, 90), (6, 0), (6, 40)}
    lap_lengths = []
    worst = 0.0
    for lap in range(4, 7):
        xs, gs, us = [xS_lap[0]], [xS_lap[1]], []
        t = 0
        while True:
            key = (lap, t)
            if key in snaps:
                st = lmpc_state(rl, rpm4)
                for k, v in st.items():
                    gold["lmpc_%d_%d_%s" % (lap, t, k)] = v
                gold["lmpc_%d_%d_x0" % key] = np.array(xs[-1])
            rl.solve(xs[-1])
            ol.solve(xs[-1])
            rq, oq = qp_of(rl, xs[-1]), ol.last_qp
            for a, b, nm in zip(rq, oq, "PqAlu"):
                worst = max(worst, close(a, b, 1e-11, "lmpc %s lap %d t %d" % (nm, lap, t)))
            worst = max(worst, close(np.array(rl.A), np.array(ol.A), 1e-11, "lmpc A"))
            worst = max(worst, close(rl.uPred, ol.uPred, 1e-7, "lmpc uPred lap %d t %d" % (lap, t)))
            worst = max(worst, close(rl.zt, ol.zt, 1e-6, "lmpc zt"))
            # keep the oracle on the reference's exact iterate so that both stay in lock-step
            ol.xPred, ol.uPred, ol.zt, ol.zt_u = rl.xPred.copy(), rl.uPred.copy(), rl.zt.copy(), rl.zt_u.copy()
            ol.xLin, ol.uLin, ol.OldInput = rl.xLin.copy(), rl.uLin.copy(), rl.OldInput.copy()
            if key in snaps:
                k = "lmpc_%d_%d_" % key
                for a, nm in zip(rq, "PqAlu"):
                    gold[k + "qp_" + nm] = a
                gold[k + "A"], gold[k + "B"], gold[k + "C"] = np.array(rl.A), np.array(rl.B), np.array(rl.C)
                gold[k + "SS_sel"], gold[k + "Qfun_sel"] = rl.SS_PointSelectedTot, rl.Qfun_SelectedTot
                gold[k + "Succ_SS"], gold[k + "Succ_uSS"] = rl.Succ_SS_PointSelectedTot, rl.Succ_uSS_PointSelectedTot
                gold[k + "xPred"], gold[k + "uPred"], gold[k + "lambd"] = rl.xPred, rl.uPred, rl.lambd
                gold[k + "zt_out"], gold[k + "ztu_out"] = rl.zt, rl.zt_u
            us.append(rl.uPred[0, :].copy())
            rl.addPoint(xs[-1], us[-1])
            ol.addPoint(xs[-1], us[-1])
            xt, gt = vehicle.dyn_model(omap, xs[-1], gs[-1], us[-1])
            xs.append(xt)
            gs.append(gt)
            t += 1
            if xs[-1][4] > rmap.TrackLength or t >= 400:
                break
        xF = [np.array(xs[-1]) - np.array([0, 0, 0, 0, rmap.TrackLength, 0]), np.array(gs[-1])]
        xs.pop()
        gs.pop()
        xl, ul, gl = np.array(xs), np.array(us), np.array(gs)
        rl.addTrajectory(xl, ul, gl)
        ol.addTrajectory(xl.copy(), ul.copy(), gl.copy())
        rpm4.addTrajectory(xl, ul)
        opm4.addTrajectory(xl.copy(), ul.copy())
        lap_lengths.append(xl.shape[0])
        print("lap", lap, "steps", xl.shape[0], "Qfun[0]", rl.Qfun[lap][0], "worst", worst)
        xS_lap = xF
    gold["lmpc_lap_lengths"] = np.array(lap_lengths)
    print("LMPC lock-step laps 4-6: max |diff| =", worst)

    golden_file.save(os.path.join(OUT, "reference_golden.npz"), gold)
    print("wrote", os.path.join(OUT, "reference_golden.npz"), len(gold), "arrays")


if __name__ == "__main__":
    main()
