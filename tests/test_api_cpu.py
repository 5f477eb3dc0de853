"""CPU tests of the boundary: the C-ABI library loads and exports every symbol of include/bmpc.h, fails loudly
without a device, and the Python mirror validates its arguments like the reference."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from pympc_b200 import _lib
from pympc_b200.workloads import point_mass, pendulum


def test_library_exports_every_declared_symbol(bmpc_lib):
    header = open(os.path.join(ROOT, "include", "bmpc.h")).read()
    declared = set(re.findall(r"\b(bmpc_[a-z_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(bmpc_lib, name)


def test_config_struct_layout_matches_defaults(bmpc_lib):
    c = _lib.BmpcConfig(); bmpc_lib.bmpc_default_config(c)
    assert (c.Np, c.max_iter, c.first_iters, c.pdas_steps, c.polish, c.soft_on) == (20, 4000, 0, 10, 1, 1)
    assert (c.eps_feas, c.sigma, c.alpha, c.eps_abs, c.eps_rel) == (1e6, 1e-6, 1.6, 1e-3, 1e-3)


def test_create_argument_errors(bmpc_lib):
    c = _lib.BmpcConfig(); bmpc_lib.bmpc_default_config(c)
    h = ctypes.c_void_p()
    c.nx, c.nu, c.Np = 0, 1, 20
    assert bmpc_lib.bmpc_create(c, ctypes.byref(h)) == -1
    c.nx, c.Np, c.Nc = 2, 5, 9
    assert bmpc_lib.bmpc_create(c, ctypes.byref(h)) == -1
    assert b"invalid dimensions" in bmpc_lib.bmpc_last_error(None)


def test_no_cpu_fallback_without_device(bmpc_lib):
    """in a process that sees no device (CUDA_VISIBLE_DEVICES empty, so this runs on GPU machines too), setup() raises"""
    import subprocess, sys
    code = ("import sys; sys.path.insert(0, sys.argv[1])\n"
            "from pympc_b200 import MPCController, BmpcError, _lib\n"
            "from pympc_b200.workloads import point_mass\n"
            "assert _lib.load().bmpc_device_count() == 0\n"
            "K = MPCController(**point_mass())\n"
            "try:\n    K.setup()\nexcept BmpcError as exc:\n    print(exc)\nelse:\n    raise SystemExit('setup() succeeded without a device')\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout + r.stderr
    assert re.search("no CUDA device", r.stdout), r.stdout


@pytest.mark.parametrize("kw,msg", [
    (dict(Ad=np.zeros((2, 3))), "Ad should be a square matrix"),
    (dict(Bd=np.zeros((3, 1))), "Bd should be a matrix of dimension"),
    (dict(Np=1), "Np should be > 1"),
    (dict(Nc=21), "Nc should be <= Np"),
    (dict(x0=np.zeros(3)), "x0 should be an array of dimension"),
    (dict(xref=np.zeros((3, 2))), "xref should be either a vector"),
    (dict(uref=np.zeros(2)), "uref should be a vector"),
    (dict(uminus1=np.zeros(2)), "uminus1 should be a vector"),
    (dict(Qx=np.zeros((3, 3))), "Qx should be a matrix"),
    (dict(QxN=np.zeros((3, 3))), "QxN should be a square matrix"),
    (dict(Qu=np.zeros((2, 2))), "Qu should be a square matrix"),
    (dict(QDu=np.zeros((2, 2))), "QDu should be a square matrix"),
    (dict(xmin=np.zeros(3)), "xmin should be a vector"),
    (dict(xmax=np.zeros(3)), "xmax should be a vector"),
    (dict(umin=np.zeros(2)), "umin should be a vector"),
    (dict(umax=np.zeros(2)), "umax should be a vector"),
    (dict(Dumin=np.zeros(2)), "Dumin should be a vector"),
    (dict(Dumax=np.zeros(2)), "Dumax should be a vector"),
])
def test_constructor_validation_like_reference(kw, msg, bmpc_lib):
    from pympc_b200 import MPCController
    cfg = point_mass(); cfg.update(kw)
    with pytest.raises(ValueError, match=msg):
        MPCController(**cfg)


def test_defaults_like_reference(bmpc_lib):
    from pympc_b200 import MPCController
    cfg = pendulum()
    K = MPCController(cfg["Ad"], cfg["Bd"])
    assert K.Np == 20 and K.Nc == 20 and np.all(K.Qx == 0) and K.QxN is K.Qx          # quirk Q3: zeros, not eye
    assert np.all(np.isinf(K.xmin)) and np.all(K.uminus1 == K.uref) and K.eps_feas == 1e6
    assert (K.raise_error, K.JX_ON, K.JU_ON, K.JDU_ON, K.SOFT_ON, K.COMPUTE_J_CNST) == (False, True, True, True, True, False)
    Kb = MPCController(cfg["Ad"], cfg["Bd"], batch=5, x0=np.zeros((5, 4)), xref=np.ones((5, 4)))
    assert Kb.x0.shape == (5, 4) and Kb._xref_device_layout(Kb.xref)[1] == 1


def test_fast_path_shape_table_is_well_formed():
    """csrc/tpi_shapes.inc: every compiled fast-path shape obeys the limits the kernels static_assert (nu == 1, Nc <= Np,
    Np*nx <= 128 bits of working set, Np < 32) and the shipped shapes of DESIGN.md are there."""
    import os, re
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "pympc_b200", "csrc", "tpi_shapes.inc")
    shapes = [tuple(int(v) for v in m.groups()) for m in re.finditer(r"^BMPC_TPI_SHAPE\((\d+),\s*(\d+),\s*(\d+),\s*(\d+)\)", open(path).read(), re.M)]
    assert len(shapes) == len(set(shapes)) >= 4
    for nx, nu, Np, Nc in shapes:
        assert nu == 1 and 1 <= Nc <= Np < 32 and Np * nx <= 128, (nx, nu, Np, Nc)
    for s in ((4, 1, 20, 20), (2, 1, 20, 20), (4, 1, 10, 10), (4, 1, 20, 10)):
        assert s in shapes


def test_fast_path_table_query_and_on_demand_shape_build(bmpc_lib):
    """bmpc_has_fast_path reports the compiled table; build.jit_shape validates the shape limits of the thread-per-instance kernels
    (nu == 1, Np * nx <= 128, Np < 32, Nc <= Np) before invoking nvcc"""
    from pympc_b200 import build
    assert bmpc_lib.bmpc_has_fast_path(4, 1, 20, 20) == 1 and bmpc_lib.bmpc_has_fast_path(4, 1, 20, 0) == 1
    assert bmpc_lib.bmpc_has_fast_path(4, 1, 20, 10) == 1 and bmpc_lib.bmpc_has_fast_path(5, 1, 17, 17) == 0
    for bad in ((4, 2, 20, None), (8, 1, 20, None), (2, 1, 40, None), (3, 1, 10, 11)):
        with pytest.raises(ValueError):
            build.jit_shape(*bad)
    # multi-input table (thread-per-instance Riccati polish over the scalar delta-u chain): MIMO reference-governor shape compiled in
    assert bmpc_lib.bmpc_has_multi_input_fast_path(8, 4, 40, 40) == 1 and bmpc_lib.bmpc_has_multi_input_fast_path(8, 4, 40, 0) == 1
    assert bmpc_lib.bmpc_has_multi_input_fast_path(8, 4, 12, 5) == 1 and bmpc_lib.bmpc_has_multi_input_fast_path(3, 2, 10, 10) == 0
    for bad in ((12, 5, 10, None), (3, 2, 10, 11), (30, 1, 10, None)):      # working-set word: 2 nx + 10 nu <= 64 bits
        with pytest.raises(ValueError):
            build.jit_multi_input_shape(*bad)


def test_output_arrays_are_reused_only_when_the_caller_dropped_them():
    """output() returns an array the caller owns (like the reference's fresh array per call); arrays handed out earlier are
    recycled only once nobody references them — never while the caller (or uminus1_rh) still holds them"""
    from pympc_b200.mpc import MPCController
    class Fake:
        pass
    f = Fake(); f._out_pool = []; f.uminus1_rh = None; f._u0 = np.arange(16384.0).reshape(-1, 1)
    fresh = MPCController._fresh_output
    a = fresh(f); f.uminus1_rh = a
    b = fresh(f); f.uminus1_rh = b
    assert a is not b and np.array_equal(a, f._u0)
    ida = id(a); del a
    c = fresh(f); f.uminus1_rh = c
    assert id(c) == ida                                   # the dropped one came back
    keep = [c]
    d = fresh(f); f.uminus1_rh = d
    e = fresh(f); f.uminus1_rh = e
    assert d is not c and e is not c and e is not d
    for t in range(10):                                   # a plain closed loop cycles through two arrays
        U = fresh(f); f.uminus1_rh = U
    assert len(f._out_pool) <= 7                          # b, c, d, e are still held by this test; the loop itself needs two


def test_batched_xref_shapes_are_unambiguous():
    """a 2-D xref keeps the reference's meaning (one (Np+1, nx) trajectory, mpc.py:120,414-421) even when batch == Np+1 — with a
    warning —; per-instance constant references have the explicit form (batch, 1, nx)"""
    import warnings
    from pympc_b200.mpc import MPCController
    Ad = np.array([[1.0, 0.2], [0.0, 1.0]]); Bd = np.array([[0.0], [0.2]])
    K = MPCController(Ad, Bd, Np=3, batch=4, x0=np.zeros((4, 2)), Qx=np.eye(2), QDu=np.eye(1))
    R = np.arange(8.0).reshape(4, 2)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        arr, rows = K._xref_device_layout(R)
    assert rows == 4 and arr.shape == (4, 8) and (arr == R.ravel()).all() and any("batch, 1, nx" in str(m.message) for m in w)
    arr, rows = K._xref_device_layout(R[:, None, :])
    assert rows == 1 and arr.shape == (4, 2) and (arr == R).all()
    assert K._xref_arg(R[:, None, :]).shape == (4, 1, 2)
    K5 = MPCController(Ad, Bd, Np=3, batch=5, x0=np.zeros((5, 2)), Qx=np.eye(2), QDu=np.eye(1))
    arr, rows = K5._xref_device_layout(np.ones((5, 2)))          # batch != Np+1: (B, nx) is per-instance, as before
    assert rows == 1 and arr.shape == (5, 2)


def test_result_arrays_handed_out_without_a_copy_are_not_overwritten_while_held(monkeypatch):
    """zero-copy results: the solver writes u* into one of a few pinned arrays and output() returns that array itself; an array is
    bound again only when nobody outside holds it (the caller, uminus1_rh and the current result are references)"""
    import pympc_b200.mpc as M

    class FakePin:
        def __init__(self, shape, dtype=np.float64):
            self.array = np.zeros(shape, dtype)
    monkeypatch.setattr(M, "PinnedArray", FakePin)

    class Fake:
        pass
    f = Fake(); f._out_pins = []; f._B = 8; f.nu = 1
    nxt = M.MPCController._next_result_array
    held = []
    p0 = nxt(f); held.append(p0.array)                        # the caller keeps the first result
    p1 = nxt(f); assert p1 is not p0
    a1 = p1.array; del p1
    p2 = nxt(f); assert p2.array is not a1 and p2.array is not held[0]      # a1 still referenced here
    del a1, p2
    p3 = nxt(f); assert p3.array is not held[0]               # one of the dropped ones comes back, never the held one
    assert len(f._out_pins) <= 3
    del p3
    for _ in range(10):                                       # a caller that keeps everything: the pool stops growing, then no array is offered
        p = nxt(f)
        if p is None:
            break
        held.append(p.array); del p
    assert len(f._out_pins) == 6 and nxt(f) is None


def test_multi_input_shape_table_is_well_formed():
    """csrc/tpm_shapes.inc: every entry fits the 64-bit working-set word (2 nx + 10 nu), pattern entries come before the dense entry of
    their shape (bmpc_setup takes the first entry whose masks contain the system's pattern) and the masks of the MIMO reference
    governor's entry are exactly the non-zeros of that system (pympc_b200.workloads.mimo)"""
    import os, re
    from pympc_b200.workloads import mimo
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "pympc_b200", "csrc", "tpm_shapes.inc")
    entries = []
    for line in open(path):
        m = re.match(r"^BMPC_TPM_SPARSE_SHAPE\((\d+),\s*(\d+),\s*(\d+),\s*(\d+),\s*(0x[0-9a-fA-F]+)ull,\s*(0x[0-9a-fA-F]+)u\)", line)
        if m:
            entries.append(tuple(int(v) for v in m.groups()[:4]) + (int(m.group(5), 16), int(m.group(6), 16)))
            continue
        m = re.match(r"^BMPC_TPM_SHAPE\((\d+),\s*(\d+),\s*(\d+),\s*(\d+)\)", line)
        if m:
            entries.append(tuple(int(v) for v in m.groups()) + (None, None))
    assert len(entries) >= 3
    for nx, nu, Np, Nc, am, bm in entries:
        assert 2 * nx + 10 * nu <= 64 and 1 <= Nc <= Np, (nx, nu, Np, Nc)
        if am is not None:
            assert nx * nx <= 64 and nx * nu <= 32 and am < (1 << (nx * nx)) and bm < (1 << (nx * nu))
            later_dense = [e for e in entries[entries.index((nx, nu, Np, Nc, am, bm)) + 1:] if e[:4] == (nx, nu, Np, Nc) and e[4] is None]
            assert later_dense, "a pattern entry needs the dense entry of its shape behind it"
    c = mimo()
    am = sum(1 << i for i, v in enumerate(np.asarray(c["Ad"]).ravel()) if v != 0.0)
    bm = sum(1 << i for i, v in enumerate(np.asarray(c["Bd"]).ravel()) if v != 0.0)
    assert (8, 4, 40, 40, am, bm) in entries
