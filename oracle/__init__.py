"""ORACLE -- test infrastructure only.

CPU restatements of the reference algorithms on the DPVO update hot path, used by tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs as the checker.
Nothing under dpvo_b200/ imports this package.
"""


def lietorch_backend():
    """oracle/shims/lietorch_backends.py (the CPU stand-in for the `lietorch_backends` extension), loaded under a
    private name so that it neither shadows nor is shadowed by the product's extension module of that name"""
    import importlib.util
    import os
    import sys
    name = "oracle_lietorch_backends"
    if name not in sys.modules:
        spec = importlib.util.spec_from_file_location(name, os.path.join(os.path.dirname(os.path.abspath(__file__)), "shims", "lietorch_backends.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        sys.modules[name] = mod
    return sys.modules[name]
