"""Generates the committed golden fixtures from a checkout of the reference, forgi86/pyMPC.

For every case the QP is assembled by the UNMODIFIED reference (pyMPC.mpc.MPCController with a
stub ``osqp`` module, tests/refharness.py), solved by ``oracle.kkt.solve_exact`` and certified by
the solver-independent KKT residuals (< 1e-9) on the reference-assembled (P, q, A, l, u).
Closed loops use the linear plant x+ = Ad x + Bd u (README.md:59-77 pattern).
ref_assembly.npz and pend_osqp_calls.npz hold what the reference itself computed and handed to
its solver, so that the tests compare against the reference without needing it.

    python tests/golden/make_golden.py PATH_TO_PYMPC_CHECKOUT [fixture ...]
"""
import json
import os
import sys

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from refharness import load_reference_controller  # noqa: E402
from oracle.kkt import solve_exact, kkt_residuals  # noqa: E402
from pympc_b200.workloads import point_mass, pendulum, mimo, pendulum_random  # noqa: E402
from test_oracle import LIVE_VARIANTS, live_variant  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
MPC = None


def exact(K, warm=None):
    P, A = K.P.toarray(), K.A.toarray()
    z, y, r = solve_exact(P, K.q, A, K.l, K.u, warm=warm)
    assert max(r.values()) < 1e-9, r
    return z, y, r


def first_solve(name, cfg):
    K = MPC(**cfg); K.setup(solve=False)
    z, y, r = exact(K)
    NX = (K.Np + 1) * K.nx; NU = K.Nc * K.nu
    obj = 0.5 * z @ (K.P @ z) + K.q @ z
    np.savez_compressed(os.path.join(OUT, f"{name}_first.npz"), z=z, y=y, q=K.q, l=K.l, u=K.u,
                        P_data=K.P.toarray()[np.nonzero(K.P.toarray())], A_sum=np.array([K.A.toarray().sum(), np.abs(K.A.toarray()).sum()]),
                        u_seq=z[NX:NX + NU], x_seq=z[:NX], eps_seq=z[NX + NU:], obj=obj, J_CNST=K.J_CNST,
                        kkt=np.array([r['stat'], r['prim'], r['comp']]))
    print(name, "first u0", z[NX:NX + K.nu], r)


def closed_loop(name, cfg, nsteps, xref_fn=None):
    K = MPC(**cfg); K.setup(solve=False)
    Ad, Bd = np.asarray(cfg['Ad']), np.asarray(cfg['Bd'])
    NX = (K.Np + 1) * K.nx
    x = np.array(cfg['x0'], float); um1 = np.array(cfg['uminus1'], float)
    xs, us, warm = [], [], None
    for t in range(nsteps):
        K.update(x, um1, xref=(xref_fn(t) if xref_fn else None), solve=False)
        z, y, r = exact(K, warm)
        warm = (z, y)
        u0 = z[NX:NX + K.nu].copy()
        xs.append(x.copy()); us.append(u0)
        x = Ad @ x + Bd @ u0; um1 = u0
    np.savez_compressed(os.path.join(OUT, f"{name}_loop.npz"), x=np.array(xs), u=np.array(us))
    print(name, "loop u[:8]", np.array(us)[:8].ravel())


def random_batch(B=24, nsteps=4):
    cfg = pendulum()
    X0, Xref = pendulum_random(B, seed=0)
    Ad, Bd = cfg['Ad'], cfg['Bd']
    U = np.zeros((nsteps, B, 1)); X = np.zeros((nsteps, B, 4))
    for b in range(B):
        c = dict(cfg); c['x0'] = X0[b]; c['xref'] = Xref[b]
        K = MPC(**c); K.setup(solve=False)
        x = X0[b].copy(); um1 = np.zeros(1); warm = None
        for t in range(nsteps):
            K.update(x, um1, solve=False)
            z, y, r = exact(K, warm); warm = (z, y)
            u0 = z[84:85].copy(); U[t, b] = u0; X[t, b] = x
            x = Ad @ x + Bd @ u0; um1 = u0
    np.savez_compressed(os.path.join(OUT, "pend_rand.npz"), X0=X0, Xref=Xref, U=U, X=X)
    print("pend_rand", U[0, :4].ravel())


def variants():
    out = {}
    # (a) Nc < Np, time-varying xref, nonzero uref, Qu > 0  (mpc.py:618-692 demo shape)
    c = point_mass(); c['Np'] = 25; c['Nc'] = 10; c['uref'] = np.array([0.1])
    c['xmin'] = np.array([-10.0, -10.0]); c['xmax'] = np.array([7.0, 10.0])
    Xref = np.kron(np.ones((26, 1)), c['xref']); Xref[:, 0] = np.linspace(5.0, 7.0, 26)
    c['xref'] = Xref
    K = MPC(**c); K.setup(solve=False); z, y, r = exact(K)
    out['a_z'] = z; out['a_xref'] = Xref
    # (b) small MIMO with Nc < Np (channel-mixing delta-u quirk live)
    c = mimo(); c['Np'] = 12; c['Nc'] = 5; c['x0'] = np.array([0.3, -0.2, 0.1, 0.0, -0.4, 0.2, 0.0, 0.1])
    c['umin'] = -0.5 * np.ones(4); c['umax'] = 0.5 * np.ones(4); c['Qu'] = 0.1 * np.eye(4)
    K = MPC(**c); K.setup(solve=False); z, y, r = exact(K)
    out['b_z'] = z
    # (c) pendulum starting outside the soft position bound (slacks strongly active)
    c = pendulum(); c['x0'] = np.array([0.45, 0.3, -0.05, 0.1])
    K = MPC(**c); K.setup(solve=False); z, y, r = exact(K)
    out['c_z'] = z
    np.savez_compressed(os.path.join(OUT, "variants.npz"), **out)
    print("variants ok")


def put_csc(out, name, M):
    M = sp.csc_matrix(M)
    out[name + "_data"], out[name + "_indices"], out[name + "_indptr"], out[name + "_shape"] = M.data, M.indices, M.indptr, np.array(M.shape)


def reference_assembly():
    """the reference's (P, A, q, l, u) at setup and (q, l, u, J_CNST) after three updates with seeded random x, u_-1, xref, for
    every case of tests/test_oracle.py::test_assembly_matches_reference_live"""
    out = {}
    for v in LIVE_VARIANTS:
        cfg = live_variant(v)
        K = MPC(**cfg); K.setup(solve=False)
        put_csc(out, f"{v}__P", K.P); put_csc(out, f"{v}__A", K.A)
        out[f"{v}__q"], out[f"{v}__l"], out[f"{v}__u"] = K.q.copy(), K.l.copy(), K.u.copy()
        rng = np.random.default_rng(3); rec = {k: [] for k in ("x", "um1", "xref", "q", "l", "u", "J_CNST")}
        for t in range(3):
            x = rng.normal(size=K.nx); um1 = rng.normal(size=K.nu)
            xr = np.array(cfg["xref"]) if t == 0 else rng.normal(size=np.shape(cfg["xref"]))
            K.update(x, um1, xref=xr, solve=False)
            for k, val in (("x", x), ("um1", um1), ("xref", xr), ("q", K.q), ("l", K.l), ("u", K.u), ("J_CNST", K.J_CNST)):
                rec[k].append(np.copy(val))
        for k, vals in rec.items():
            out[f"{v}__upd_{k}"] = np.array(vals)
    np.savez_compressed(os.path.join(OUT, "ref_assembly.npz"), **out)
    print("ref_assembly", len(out), "arrays")


def pend_osqp_calls(nsteps=5):
    """what the reference hands its `osqp` object in the pendulum closed loop at eps 1e-9: the setup() call (matrices, vectors,
    keyword arguments), then the update(l=, u=, q=) of each step, the states and previous inputs taken from pend_loop.npz"""
    cfg = pendulum(); g = np.load(os.path.join(OUT, "pend_loop.npz"))
    K = MPC(**cfg, eps_abs=1e-9, eps_rel=1e-9); K.setup(solve=False)
    (P, q, A, l, u), kw = K.prob.setup_args
    out = {"q": np.copy(q), "l": np.copy(l), "u": np.copy(u), "setup_kwargs": np.array(json.dumps(kw, sort_keys=True))}
    put_csc(out, "P", P); put_csc(out, "A", A)
    rec = {"q": [], "l": [], "u": []}
    for t in range(nsteps):
        um1 = np.array(cfg["uminus1"], float) if t == 0 else g["u"][t - 1]
        K.update(g["x"][t], um1, solve=False)
        for k in rec:
            rec[k].append(np.copy(K.prob.update_args[k]))
    for k, vals in rec.items():
        out["upd_" + k] = np.array(vals)
    np.savez_compressed(os.path.join(OUT, "pend_osqp_calls.npz"), **out)
    print("pend_osqp_calls", kw)


FIXTURES = {
    "pm_first": lambda: first_solve("pm", point_mass()), "pend_first": lambda: first_solve("pend", pendulum()),
    "mimo_first": lambda: first_solve("mimo", mimo()),
    "pm_loop": lambda: closed_loop("pm", point_mass(), 30), "pend_loop": lambda: closed_loop("pend", pendulum(), 40),
    "mimo_loop": lambda: closed_loop("mimo", mimo(), 12),
    "pend_rand": random_batch, "variants": variants, "ref_assembly": reference_assembly, "pend_osqp_calls": pend_osqp_calls,
}


if __name__ == "__main__":
    if len(sys.argv) < 2:
        raise SystemExit(__doc__)
    MPC = load_reference_controller(os.path.abspath(sys.argv[1]))
    for name in sys.argv[2:] or FIXTURES:
        FIXTURES[name]()
