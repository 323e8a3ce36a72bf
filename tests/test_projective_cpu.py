"""Host logic of dpvo_b200.projective_ops without a GPU: the same checks as tests/test_projective_gpu.py with the
oracle's lietorch_backends stand-in (oracle/shims) monkeypatched under dpvo_b200.lietorch."""
import importlib.util
import os

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture()
def gpu_tests(monkeypatch):
    from oracle import lietorch_backend
    LB = lietorch_backend()
    import dpvo_b200.lietorch.groups as Gm
    import dpvo_b200.projective_ops as pops
    monkeypatch.setattr(Gm, "_B", LB)
    monkeypatch.setattr(pops, "transform_fused", lambda poses, *a: pops.transform(poses, *a).permute(0, 1, 4, 2, 3))
    spec = importlib.util.spec_from_file_location("_proj_gpu", os.path.join(HERE, "test_projective_gpu.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    m.DEV = "cpu"
    yield m


@pytest.mark.parametrize("name", ["test_transform_and_jacobians_match_oracle", "test_transform_autograd_matches_oracle_autograd",
                                  "test_sim3_jacobian_column_by_finite_differences", "test_flow_mag_and_point_cloud"])
def test_projective_ops_host_logic_on_oracle_backend(gpu_tests, name):
    getattr(gpu_tests, name)(None)
