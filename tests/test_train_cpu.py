"""Training-path host code without a GPU: the differentiable bundle adjustment of dpvo_b200/ba.py against the
REFERENCE's own dpvo/ba.py:BA (imported unmodified from the reference sources where they are at hand, else its
stored outputs; lietorch served by the CPU oracle on both sides), outputs and gradients in fp64; and the sequence loss on a hand-checkable case."""
import pytest
import torch

import refdata
from oracle import refimport
from dpvo_b200 import synthetic


class _UniqueGroups:
    """stand-in for the device grouping kernel (EdgeGroups) on the CPU: group ids ascend with the key"""

    def __init__(self, key):
        keys, inv = torch.unique(key, sorted=True, return_inverse=True)
        self.key_a, self.group_of, self.max_groups = keys, inv.int(), keys.numel()


@pytest.fixture()
def cpu_ops(monkeypatch):
    from oracle import lietorch_backend
    LB = lietorch_backend()
    import dpvo_b200.lietorch.groups as Gm
    import dpvo_b200.ba as ba
    monkeypatch.setattr(Gm, "_B", LB)
    monkeypatch.setattr(ba, "EdgeGroups", _UniqueGroups)
    yield ba


def _problem(seed, structure_only=False):
    st = synthetic.make_state(dict(M=4, lifetime=4, removal=6, opt_window=4, ht=240, wd=320, intrinsics=(160.0, 160.0, 160.0, 120.0)),
                              7, device="cpu", features=False, seed=seed, noise=0.02, buffer=8)
    g = torch.Generator().manual_seed(seed)
    poses = st.poses.double()[None, :st.n]
    patches = st.patches.double()[None, :st.n * 4]
    intr = st.intrinsics.double()[None, :st.n]
    from oracle import ba as OB
    coords = OB.transform(poses, patches, intr, st.ii, st.jj, st.kk)
    target = coords[..., 1, 1, :] + torch.randn(1, st.E, 2, generator=g).double()
    weight = torch.rand(1, st.E, 2, generator=g).double()
    return st, poses, patches, intr, target, weight


@pytest.mark.parametrize("structure_only", [False, True])
def test_differentiable_ba_matches_the_reference_ba_forward_and_backward(cpu_ops, structure_only):
    from dpvo_b200.lietorch import SE3
    st, poses, patches, intr, target, weight = _problem(3)
    bounds = [-64, -64, 80 + 64, 60 + 64]
    names = ("poses", "patches", "d/dtarget", "d/dweight", "d/dpatches")

    def run(BA, SE3cls, lm):
        t = target.clone().requires_grad_(True)
        wt = weight.clone().requires_grad_(True)
        q = patches.clone().requires_grad_(True)
        G, Q = SE3cls(poses.clone()), q
        for _ in range(2):
            G, Q = BA(G, Q, intr, t, wt, lm, st.ii, st.jj, st.kk, bounds, ep=10.0, fixedp=1, structure_only=structure_only)
        g = torch.Generator().manual_seed(9)
        cp = torch.randn(G.data.shape, generator=g).double()
        cq = torch.randn(Q.shape, generator=g).double()
        loss = (G.data * cp).sum() + (Q * cq).sum()
        gt, gw, gq = torch.autograd.grad(loss, (t, wt, q))
        return G.data.detach(), Q.detach(), gt, gw, gq

    mine = run(cpu_ops.BA, SE3, 1e-4)

    def compute(_):
        with refimport.reference_modules():
            import dpvo.ba as RB
            from dpvo.lietorch import SE3 as RSE3
            return dict(zip(names, run(RB.BA, RSE3, 1e-4)))

    R = refdata.reference("train_ba_%s" % ("structure" if structure_only else "full"), refimport if refimport.available() else None, compute)
    for a, nm in zip(mine, names):
        scale = max(1.0, R.absmax(nm))
        assert (R.pick(nm, a) - R[nm]).abs().max().item() <= 1e-8 * scale, (nm, (R.pick(nm, a) - R[nm]).abs().max().item())
    if not structure_only:
        assert (mine[0] - poses).abs().max().item() > 1e-4          # the step moved the poses


def test_spd_solve_failure_gives_a_zero_step_and_no_gradient(cpu_ops):
    H = -torch.eye(3, dtype=torch.float64)[None].requires_grad_(True)            # not positive definite
    b = torch.ones(1, 3, 1, dtype=torch.float64, requires_grad=True)
    x = cpu_ops._SPDSolve.apply(H, b)
    assert torch.equal(x, torch.zeros_like(x))
    gH, gb = torch.autograd.grad(x.sum(), (H, b), allow_unused=True)
    assert gH is None and gb is None


def test_sequence_loss_known_answer(cpu_ops):
    """two identical trajectories and a constant 1-px flow error: pose terms vanish, flow term = 0.1 * 1.0 per iteration"""
    from dpvo_b200.lietorch import SE3
    from dpvo_b200.train import sequence_loss, scale_alignment
    torch.manual_seed(0)
    G = SE3.exp(0.3 * torch.randn(1, 5, 6).double())
    y = torch.randn(1, 12, 3, 3, 2).double()
    x = y.clone()
    x[..., 0] += 1.0
    v = torch.ones(1, 12).double()
    traj = [(v, x, y, G, G, torch.as_tensor(0)) for _ in range(4)]
    loss, m = sequence_loss(traj, 3, flow_weight=0.1, pose_weight=10.0)
    assert abs(loss.item() - 0.4) < 1e-9 and m["tr"].item() < 1e-9 and m["ro"].item() < 1e-9
    A = torch.randn(20, 3).double()
    assert abs(scale_alignment(2.5 * A, A).item() - 2.5) < 1e-9
