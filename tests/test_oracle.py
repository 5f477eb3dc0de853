"""CPU tests of the oracle: assembly vs the reference / golden fixtures, exact solver and the C
restatement of OSQP vs the KKT-certified goldens."""
import json

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import golden
from oracle.qp_assembly import QPData
from oracle.kkt import solve_exact, kkt_residuals
from pympc_b200.workloads import point_mass, pendulum, mimo, WORKLOADS

CASES = {"pm": point_mass, "pend": pendulum, "mimo": mimo}
LIVE_VARIANTS = ["pm", "pend", "mimo", "pm_Nc_tv", "mimo_Nc_uref", "pend_inf"]


def live_variant(variant):
    """configuration of one case of test_assembly_matches_reference_live (also read by tests/golden/make_golden.py)"""
    if variant in CASES:
        return CASES[variant]()
    if variant == "pm_Nc_tv":
        cfg = point_mass(); cfg["Np"] = 25; cfg["Nc"] = 10; cfg["xref"] = np.kron(np.ones((26, 1)), cfg["xref"])
    elif variant == "mimo_Nc_uref":
        cfg = mimo(); cfg["Np"] = 12; cfg["Nc"] = 5; cfg["uref"] = np.array([0.1, -0.2, 0.3, 0.0]); cfg["Qu"] = np.diag([1., 2, 3, 4])
    else:
        cfg = pendulum(); cfg["Qx"] = sp.diags([0.3, 0, 1.0, 0]); cfg["xmax"] = np.array([np.inf, 1, 2, 3]); cfg["Dumin"] = np.array([-np.inf])
    return cfg


def golden_csc(g, name):
    """a sparse matrix stored by tests/golden/make_golden.py as its CSC arrays"""
    return sp.csc_matrix((g[name + "_data"], g[name + "_indices"], g[name + "_indptr"]), shape=tuple(g[name + "_shape"]))


@pytest.mark.parametrize("name", list(CASES))
def test_assembly_matches_golden_vectors(name):
    """q, l, u and fingerprints of P, A stored from the reference's own assembly."""
    g = golden(f"{name}_first.npz")
    Q = QPData(**CASES[name]())
    assert np.array_equal(Q.q, g["q"])
    for a, b in ((Q.l, g["l"]), (Q.u, g["u"])):
        assert np.array_equal(np.isinf(a), np.isinf(b))
        assert np.array_equal(np.where(np.isinf(a), 0, a), np.where(np.isinf(b), 0, b))
    assert np.array_equal(Q.P[np.nonzero(Q.P)], g["P_data"])
    assert np.allclose([Q.A.sum(), np.abs(Q.A).sum()], g["A_sum"], rtol=0, atol=1e-12)


@pytest.mark.parametrize("variant", LIVE_VARIANTS)
def test_assembly_matches_reference_live(variant):
    """(P, A, q, l, u) and J_CNST exactly as the unmodified reference's MPCController assembled them, at setup and after three
    update() calls with random x, u_-1 and xref (stored by tests/golden/make_golden.py in ref_assembly.npz)"""
    g = golden("ref_assembly.npz")
    k = lambda name: g[f"{variant}__{name}"]
    cfg = live_variant(variant)
    Q = QPData(**cfg)
    fin = lambda v: np.where(np.isinf(v), 0, v)
    assert np.array_equal(golden_csc(g, f"{variant}__P").toarray(), Q.P) and np.array_equal(golden_csc(g, f"{variant}__A").toarray(), Q.A)
    assert np.array_equal(k("q"), Q.q) and np.array_equal(fin(k("l")), fin(Q.l)) and np.array_equal(fin(k("u")), fin(Q.u))
    for t in range(3):
        Q.update(k("upd_x")[t], k("upd_um1")[t], k("upd_xref")[t])
        assert np.array_equal(k("upd_q")[t], Q.q) and np.array_equal(fin(k("upd_l")[t]), fin(Q.l)) and np.array_equal(fin(k("upd_u")[t]), fin(Q.u))
        assert abs(k("upd_J_CNST")[t] - Q.constant_term()) < 1e-12


@pytest.mark.parametrize("name", ["pm", "pend"])
def test_exact_solver_reproduces_golden(name):
    g = golden(f"{name}_first.npz")
    Q = QPData(**CASES[name]())
    z, y, r = solve_exact(Q.P, Q.q, Q.A, Q.l, Q.u)
    assert max(r.values()) < 1e-9
    assert np.max(np.abs(z[Q.NX:Q.NX + Q.NU] - g["u_seq"])) < 1e-8
    rg = kkt_residuals(Q.P, Q.q, Q.A, Q.l, Q.u, g["z"], g["y"])
    assert max(rg.values()) < 1e-9          # the stored golden is itself a KKT point of the oracle-assembled QP


def test_point_mass_analytic_known_answer():
    """rate- then magnitude-limited ramp 0.2, 0.4, ..., 1.2, 1.2 (SURVEY.md §4)."""
    g = golden("pm_loop.npz")
    expect = np.minimum(0.2 * (np.arange(8) + 1), 1.2)
    assert np.max(np.abs(g["u"][:8, 0] - expect)) < 1e-9


@pytest.mark.parametrize("name", ["pm", "pend", "mimo"])
def test_osqp_port_default_and_tight(name, osqp_port_lib):
    """The C restatement: at the reference's eps=1e-3 it stops within a few 1e-2 of the optimum (as OSQP does);
    at eps=1e-9 it agrees with the certified optimum to 1e-6."""
    g = golden(f"{name}_first.npz")
    Q = QPData(**CASES[name]()); Pu, Ac = Q.to_csc()
    s = osqp_port_lib.OSQP().setup(Pu, Q.q, Ac, Q.l, Q.u)
    r = s.solve()
    assert r.info.status == "solved" and r.info.iter % 25 == 0
    assert np.max(np.abs(r.x[Q.u0_slice()] - g["u_seq"][:Q.nu])) < 5e-2
    s2 = osqp_port_lib.OSQP().setup(Pu, Q.q, Ac, Q.l, Q.u, eps_abs=1e-9, eps_rel=1e-9, max_iter=200000)
    r2 = s2.solve()
    assert r2.info.status == "solved"
    assert np.max(np.abs(r2.x[Q.u0_slice()] - g["u_seq"][:Q.nu])) < 1e-6
    assert abs(r2.info.obj_val - float(g["obj"])) < 1e-6 * (1 + abs(float(g["obj"])))


def test_unmodified_reference_runs_on_the_port(osqp_port_lib):
    """The calls the unmodified reference MPCController makes on its `osqp` object in the pendulum closed loop (eps 1e-9),
    recorded along the golden loop's states by tests/golden/make_golden.py in pend_osqp_calls.npz, replayed on osqp_port:
    setup() with the reference's own keyword arguments, then per step update(l=, u=, q=) and solve(), read back the way
    output() does (status, res.x slice), against the golden loop."""
    c = golden("pend_osqp_calls.npz"); g = golden("pend_loop.npz")
    P, A = golden_csc(c, "P"), golden_csc(c, "A")
    kw = json.loads(str(c["setup_kwargs"]))
    osqp_port_lib.OSQP().setup(P, c["q"], A, c["l"], c["u"], **kw)
    # the reference does not forward max_iter; tight tolerance needs more than OSQP's 4000 default
    prob = osqp_port_lib.OSQP()
    prob.setup(P, c["q"], A, c["l"], c["u"], **dict(kw, max_iter=200000))
    prob.solve()
    cfg = pendulum(); (nx, nu), Np = cfg["Bd"].shape, cfg["Np"]
    for t in range(5):
        prob.update(l=c["upd_l"][t], u=c["upd_u"][t], q=c["upd_q"][t])
        res = prob.solve()
        assert res.info.status == "solved"
        u = res.x[(Np + 1) * nx:(Np + 1) * nx + nu]
        assert np.max(np.abs(u - g["u"][t])) < 1e-6


def test_batch_cpu_driver_matches_single(osqp_port_lib):
    Q = QPData(**pendulum())
    B = 6
    bc = osqp_port_lib.BatchCPU(Q, B, eps_abs=1e-9, eps_rel=1e-9, max_iter=200000)
    g = golden("pend_loop.npz")
    X0 = np.tile(g["x"][0], (B, 1)); Um1 = np.zeros((B, 1)); Xref = np.tile(pendulum()["xref"], (B, 1))
    U, st, it = bc.step(X0, Um1, Xref, nthreads=2)
    assert np.all(st == 1) and np.max(np.abs(U - g["u"][0])) < 1e-6
    bc.close()


@pytest.mark.parametrize("name", ["pm", "pend", "mimo"])
def test_goldens_vs_independent_ldp_solver(name):
    """the goldens (oracle/kkt.py: ADMM -> active set on the reference-form QP) against an algorithmically independent exact
    solver: condensed QP with explicit slack as a least-distance problem solved by ONE Lawson-Hanson NNLS (oracle/ldp.py)"""
    from oracle.ldp import solve_mpc
    cfg = {"pm": point_mass, "pend": pendulum, "mimo": mimo}[name](); g = golden(f"{name}_first.npz")
    assert np.max(np.abs(solve_mpc(QPData(**cfg)) - g["u_seq"])) < 1e-9
    if name == "mimo":
        return
    gl = golden(f"{name}_loop.npz"); x = np.array(cfg["x0"], float); u = np.array(cfg["uminus1"], float)
    for t in range(10):
        c = dict(cfg); c["x0"] = x; c["uminus1"] = u
        assert abs(solve_mpc(QPData(**c))[0] - gl["u"][t][0]) < 1e-9, t
        u = gl["u"][t]; x = cfg["Ad"] @ x + cfg["Bd"] @ u
