"""ORACLE pinning (test infrastructure): run the reference's OWN lietorch test functions
(dpvo/lietorch/run_tests.py:16-226, unmodified) with the CPU restatement oracle/lie.py standing in for
the native `lietorch_backends` module.

The files are imported from the reference tree where it is mounted, else from the copy of the reference's
Python package that oracle/build_ref.py:stage_python packs into oracle/_ref/dpvo_ref_py.zip
(`available()` says whether either is there).  Covers SO3, RxSO3, SE3 and Sim3
(`groups` selects; the product kernels implement SO3 and SE3): the
forward identities at atol 1e-8 in fp64 and the analytic-vs-numeric Jacobian checks of the backward
operators.  Usage: python oracle/pin_lie.py   (exit code 0 = pinned)
"""
import importlib
import os
import sys

REF = "/root/reference/dpvo"
HERE = os.path.dirname(os.path.abspath(__file__))
REF_ZIP = os.path.join(HERE, "_ref", "dpvo_ref_py.zip")


def _ref_dir():
    """the reference's dpvo/ package: the mounted tree, else its staged copy (a zip on sys.path is importable)"""
    if os.path.isdir(REF):
        return REF
    if os.path.exists(REF_ZIP):
        return REF_ZIP + "/dpvo"
    return None


def available():
    return _ref_dir() is not None


def run(verbose=True, groups=("SO3", "SE3")):
    ref = _ref_dir()
    if ref is None:
        raise RuntimeError("reference package found neither at %s nor staged at %s" % (REF, REF_ZIP))
    saved = list(sys.path)
    sys.path[:0] = [os.path.join(HERE, "shims"), ref + "/lietorch", ref]
    for m in ("lietorch", "lietorch_backends", "gradcheck", "run_tests"):
        sys.modules.pop(m, None)
    try:
        import torch
        torch.manual_seed(1234)
        rt = importlib.import_module("run_tests")          # the reference's file, unmodified
        import lietorch as ref_lt                          # the reference's Python classes
        done = []
        for Group in [getattr(ref_lt, g) for g in groups]:
            for fn in (rt.test_exp_log, rt.test_inv, rt.test_adj, rt.test_act):
                fn(Group, device="cpu"); done.append((Group.group_name, fn.__name__))
            tol = 1e-3 if Group.group_name == "Sim3" else 1e-8         # run_tests.py:262-265: Sim3's Jacobians are truncated series
            rt.test_exp_log_grad(Group, device="cpu", tol=tol); done.append((Group.group_name, "test_exp_log_grad"))
            rt.test_inv_log_grad(Group, device="cpu", tol=tol); done.append((Group.group_name, "test_inv_log_grad"))
            for fn in (rt.test_adj_grad, rt.test_adjT_grad, rt.test_act_grad, rt.test_matrix_grad,
                       rt.extract_translation_grad, rt.test_vec_grad, rt.test_fromvec_grad):
                fn(Group, device="cpu"); done.append((Group.group_name, fn.__name__))
        return done
    finally:
        sys.path[:] = saved
        for m in ("lietorch", "lietorch_backends", "gradcheck", "run_tests"):
            sys.modules.pop(m, None)


if __name__ == "__main__":
    d = run()
    print("pinned: %d reference checks passed against oracle/lie.py" % len(d))
