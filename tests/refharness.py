"""Loads the UNMODIFIED reference (``pyMPC/mpc.py`` of a forgi86/pyMPC checkout) with a stub ``osqp`` module.

Used only by ``tests/golden/make_golden.py`` to generate the committed fixtures; the tests themselves read the fixtures and
never need the reference.  The stub records what pyMPC hands to the solver (SURVEY.md Appendix C)."""
import os
import sys
import types


def load_reference_controller(reference_root):
    if not os.path.isfile(os.path.join(reference_root, "pyMPC", "mpc.py")):
        raise FileNotFoundError(f"{reference_root} is not a pyMPC checkout (no pyMPC/mpc.py)")
    if "osqp" not in sys.modules:
        stub = types.ModuleType("osqp")

        class _OSQP:
            def setup(self, *a, **k):
                self.setup_args = (a, k)

            def update(self, **k):
                self.update_args = k

            def solve(self):
                raise RuntimeError("osqp is not installed; the reference cannot solve here")

        stub.OSQP = _OSQP
        stub.__stub__ = True
        sys.modules["osqp"] = stub
    if reference_root not in sys.path:
        sys.path.insert(0, reference_root)
    from pyMPC.mpc import MPCController
    return MPCController
