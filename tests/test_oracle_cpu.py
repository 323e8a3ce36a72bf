"""The CPU oracle checked against everything the reference offers for this path, without a GPU:
the reference's own lietorch tests (run from the reference's Python package, mounted or staged in oracle/_ref),
its own Python BA / projective ops (imported from the reference sources where they are at hand, else their stored
outputs), algebraic cross-checks, and the committed golden fixtures produced by
the reference's CUDA kernels on a B200 (tests/golden/, written by tests/test_parity_ref_gpu.py)."""
import os

import numpy as np
import pytest
import torch

import refdata
from oracle import ba as OB, corr as OC, graph as OG, lie as OL, pin_lie, refimport
from dpvo_b200 import synthetic

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
needs_ref = pytest.mark.skipif(not pin_lie.available(), reason="reference package neither mounted nor staged in oracle/_ref")


# ------------------------------------------------------------------------------- lietorch
@needs_ref
def test_reference_lietorch_tests_pass_on_the_oracle():
    """dpvo/lietorch/run_tests.py, unmodified, with oracle/lie.py as the native backend"""
    done = pin_lie.run()
    assert len(done) == 26


@needs_ref
def test_reference_lietorch_tests_pass_on_the_oracle_scaled_groups():
    """the same reference tests for RxSO3 and Sim3 (run_tests.py's own tolerances): the oracle side of the
    lietorch groups the CUDA library does not implement yet (SURVEY 8(f))"""
    done = pin_lie.run(groups=("RxSO3", "Sim3"))
    assert len(done) == 26


@pytest.mark.parametrize("gid", [1, 2, 3, 4])
def test_lie_identities_self_contained(gid):
    """same known-answer identities as run_tests.py:16-52, not needing the reference tree"""
    torch.manual_seed(0)
    G = OL.GROUPS[gid]
    a = .2 * torch.randn(2, 3, 4, G.K, dtype=torch.float64)
    assert torch.allclose(G.log(G.exp(a)), a, atol=1e-8)
    X = G.exp(.1 * torch.randn(5, 7, G.K, dtype=torch.float64))
    assert G.log(G.mul(X, G.inv(X))).abs().max() < 1e-8
    X = G.exp(torch.randn(5, 7, G.K, dtype=torch.float64))
    a = torch.randn(5, 7, G.K, dtype=torch.float64)
    Y1, Y2 = G.mul(X, G.exp(a)), G.mul(G.exp(G.adj(X, a)), X)
    assert G.log(G.mul(Y1, G.inv(Y2))).abs().max() < 1e-8
    p = torch.randn(5, 7, 3, dtype=torch.float64)
    ph = torch.cat([p, torch.ones_like(p[..., :1])], -1)
    assert torch.allclose(G.act(X, p), OL.matv(G.matrix(X), ph)[..., :3], atol=1e-8)
    assert torch.allclose(G.adjT(X, a), OL.matv(G.Adj_matrix(X).transpose(-1, -2), a), atol=1e-10)


def test_host_mirror_runs_on_oracle_backend(monkeypatch):
    from oracle import lietorch_backend
    LB = lietorch_backend()
    import dpvo_b200.lietorch.groups as Gm
    monkeypatch.setattr(Gm, "_B", LB)
    from dpvo_b200.lietorch import SE3
    torch.manual_seed(1)
    X = SE3.exp(torch.randn(1, 6, 6, dtype=torch.float64))
    a = torch.zeros(1, 1, 6, dtype=torch.float64, requires_grad=True)
    (SE3.exp(a) * X).log().sum().backward()       # broadcasting + autograd through the op table
    assert a.grad.shape == (1, 1, 6) and torch.isfinite(a.grad).all()
    assert SE3.Identity(3, 2).data.shape == (3, 2, 7)


# ----------------------------------------------------------------------------------- corr
def test_corr_two_formulations_agree():
    g = torch.Generator().manual_seed(2)
    f1 = torch.randn(1, 7, 16, 3, 3, generator=g, dtype=torch.float64)
    f2 = torch.randn(1, 3, 16, 20, 24, generator=g, dtype=torch.float64)
    coords = torch.rand(1, 50, 2, 3, 3, generator=g, dtype=torch.float64) * torch.tensor([32.0, 28.0]).view(1, 1, 2, 1, 1) - 4
    ii = torch.randint(0, 7, (50,), generator=g)
    jj = torch.randint(0, 3, (50,), generator=g)
    a = OC.corr_forward(f1, f2, coords, ii, jj, 3, chunk=16)
    b = OC.corr_grid_sample(f1, f2, coords, ii, jj, 3)
    assert (a - b).abs().max() < 1e-12
    coords[0, :10] += 500                       # whole windows outside -> exact zeros
    assert OC.corr_forward(f1, f2, coords, ii, jj, 3)[0, :10].abs().max() == 0


def test_patchify_integer_coords_is_a_crop():
    g = torch.Generator().manual_seed(3)
    net = torch.randn(2, 5, 12, 14, generator=g)
    coords = torch.stack([torch.randint(1, 13, (2, 9), generator=g), torch.randint(1, 11, (2, 9), generator=g)], -1).float()
    p = OC.patchify(net, coords, 1)
    for b in range(2):
        for m in range(9):
            x, y = int(coords[b, m, 0]), int(coords[b, m, 1])
            assert torch.equal(p[b, m], net[b, :, y - 1:y + 2, x - 1:x + 2])


def test_corr_oracle_reproduces_reference_kernel_fixture():
    f = os.path.join(GOLD, "corr_ref_fp32.pt")
    if not os.path.exists(f):
        pytest.skip("fixture not generated yet")
    d = torch.load(f)
    out = OC.corr_forward(d["fmap1"].double(), d["fmap2"].double(), d["coords"].double(), d["ii"], d["jj"], d["radius"])
    assert (out - d["out"].double()).abs().max().item() <= 2e-6 * d["out"].abs().max().item()
    a = d["fmap1"].double().requires_grad_(True)
    b = d["fmap2"].double().requires_grad_(True)
    OC.corr_forward(a, b, d["coords"].double(), d["ii"], d["jj"], d["radius"]).backward(d["grad"].double())
    assert (a.grad - d["fmap1_grad"].double()).abs().max().item() <= 3e-5 * a.grad.abs().max().item()
    assert (b.grad - d["fmap2_grad"].double()).abs().max().item() <= 3e-5 * b.grad.abs().max().item()


# ------------------------------------------------------------------------------------- BA
def _ba_problem(seed=4, n=6, M=8):
    g = torch.Generator().manual_seed(seed)
    dt = torch.float64
    poses = OL.se3_exp(0.05 * torch.randn(n, 6, dtype=dt, generator=g))
    poses[0] = torch.tensor([0, 0, 0, 0, 0, 0, 1.0], dtype=dt)
    intr = torch.tensor([[80.0, 80.0, 80.0, 60.0]], dtype=dt).repeat(n, 1)
    m = n * M
    cx = torch.randint(5, 155, (m,), generator=g).to(dt)
    cy = torch.randint(5, 115, (m,), generator=g).to(dt)
    offs = torch.tensor([-1.0, 0.0, 1.0], dtype=dt)
    patches = torch.zeros(m, 3, 3, 3, dtype=dt)
    patches[:, 0] = cx[:, None, None] + offs[None, None, :]
    patches[:, 1] = cy[:, None, None] + offs[None, :, None]
    patches[:, 2] = (0.3 + 0.7 * torch.rand(m, dtype=dt, generator=g))[:, None, None]
    kk, jj = torch.meshgrid(torch.arange(m), torch.arange(n), indexing="ij")
    kk, jj = kk.reshape(-1), jj.reshape(-1)
    ii = kk // M
    coords = OB.transform(poses[None], patches[None], intr[None], ii, jj, kk)
    target = coords[0, :, 1, 1] + torch.randn(len(kk), 2, dtype=dt, generator=g)
    weight = torch.rand(len(kk), 2, dtype=dt, generator=g)
    return poses, patches, intr, target, weight, ii, jj, kk, n


def test_fastba_equals_python_ba_with_aligned_constants():
    """SURVEY 8(c): one cuda_ba iteration == dpvo/ba.py:BA once damping (1 vs ep), residual gate
    (128 vs 250) and bounds are aligned and no clamp is active"""
    poses, patches, intr, target, weight, ii, jj, kk, n = _ba_problem()
    lm = torch.tensor([1e-4], dtype=torch.float64)
    p1, q1 = OB.fastba_forward(poses, patches, intr, target, weight, lm, ii, jj, kk, 1, n, 1)
    p2, q2 = OB.python_ba(poses[None], patches[None], intr[None], target[None], weight[None], 1e-4, ii, jj, kk,
                          [-64, -64, 2 * 80 + 64, 2 * 60 + 64], ep=1.0, fixedp=1, resid_gate=128.0)
    assert (p1 - poses).abs().max() > 1e-3
    assert (p1 - p2[0]).abs().max() < 1e-10 and (q1 - q2[0]).abs().max() < 1e-10
    c1 = OB.fastba_reproject(poses, patches, intr, ii, jj, kk)
    c2 = OB.transform(poses[None], patches[None], intr[None], ii, jj, kk)[0].permute(0, 3, 1, 2)
    assert (c1 - c2).abs().max() < 1e-10


def test_python_ba_and_transform_equal_the_reference_files():
    """dpvo/ba.py and dpvo/projective_ops.py imported unmodified from the reference sources where they are at hand,
    else their stored outputs (tests/golden/ref_python_ba.pt)"""
    poses, patches, intr, target, weight, ii, jj, kk, n = _ba_problem(seed=5)
    bounds = [-64, -64, 160 + 64, 120 + 64]

    def compute(_):
        with refimport.reference_modules():
            import dpvo.ba as RBA
            import dpvo.projective_ops as RP
            from dpvo.lietorch import SE3
            c_ref, v_ref, (Ji, Jj, Jz) = RP.transform(SE3(poses[None]), patches[None], intr[None], ii, jj, kk, jacobian=True)
            Gs, pt = RBA.BA(SE3(poses[None].clone()), patches[None].clone(), intr[None], target[None], weight[None], 1e-4,
                            ii, jj, kk, bounds, ep=10.0, fixedp=1)
            return dict(coords=c_ref, valid=v_ref, Ji=Ji, Jj=Jj, Jz=Jz, poses=Gs.data.clone(), patches=pt.clone())

    R = refdata.reference("python_ba", refimport if refimport.available() else None, compute)
    c, v, (Ji2, Jj2, Jz2) = OB.transform(poses[None], patches[None], intr[None], ii, jj, kk, jacobian=True)
    p2, q2 = OB.python_ba(poses[None], patches[None], intr[None], target[None], weight[None], 1e-4, ii, jj, kk,
                          bounds, ep=10.0, fixedp=1)
    for k, b in (("coords", c), ("valid", v), ("Ji", Ji2), ("Jj", Jj2), ("Jz", Jz2), ("poses", p2), ("patches", q2)):
        assert (R[k] - R.pick(k, b)).abs().max() < 1e-12, k


def test_ba_oracle_reproduces_reference_kernel_fixture():
    f = os.path.join(GOLD, "ba_ref_fast12.pt")
    if not os.path.exists(f):
        pytest.skip("fixture not generated yet")
    d = torch.load(f)
    n = d["t1"]
    p, q = OB.fastba_forward(d["poses"].double(), d["patches"].double(), d["intrinsics"].double(), d["target"].double(),
                             d["weight"].double(), torch.tensor([1e-4], dtype=torch.float64), d["ii"], d["jj"], d["kk"],
                             d["t0"], n, 2)
    assert ((p[:n] - d["poses_out"].double()).abs().max() / p[:n].abs().max()).item() < 1e-4
    live = d["live"]
    assert ((q[live, 2, 0, 0] - d["depth_out"].double()[live]).abs().max() / q[live, 2, 0, 0].abs().max()).item() < 1e-4
    ix, jx = OG.neighbors(d["kk"], d["jj"])
    assert torch.equal(ix, d["neighbors_ix"]) and torch.equal(jx, d["neighbors_jx"])
    rep = OB.fastba_reproject(d["poses"].double(), d["patches"].double(), d["intrinsics"].double(), d["ii"], d["jj"], d["kk"])
    assert (rep[None] - d["reproject"].double()).abs().max().item() < 0.2      # fixture stored in fp16


# ---------------------------------------------------------------------------------- graph
def test_neighbors_against_definition():
    g = torch.Generator().manual_seed(6)
    ii = torch.randint(0, 9, (200,), generator=g)
    jj = torch.randint(0, 5, (200,), generator=g)
    ix, jx = OG.neighbors(ii, jj)
    for e in range(200):
        grp = sorted([k for k in range(200) if ii[k] == ii[e]], key=lambda k: (int(jj[k]), k))
        pos = grp.index(e)
        assert int(ix[e]) == (grp[pos - 1] if pos > 0 else -1)
        assert int(jx[e]) == (grp[pos + 1] if pos + 1 < len(grp) else -1)


def test_group_edges_is_the_unique_inverse_partition():
    g = torch.Generator().manual_seed(7)
    ii = torch.randint(3, 30, (500,), generator=g)
    jj = torch.randint(3, 30, (500,), generator=g)
    r = OG.group_edges(ii, jj)
    _, inv = torch.unique(ii * 12345 + jj, return_inverse=True)        # net.py:88 / blocks.py:41
    assert np.array_equal(r["group_of"], inv.numpy().astype(np.int32))


def test_synthetic_graph_sizes_match_survey():
    ii, jj, kk = synthetic.replay_edges(36, 96, 13, 22)
    assert len(kk) == 47712 and len(kk.unique()) == 2208
    ii, jj, kk = synthetic.replay_edges(30, 48, 11, 16)
    assert len(kk) == 14496 and len(kk.unique()) == 816
    assert torch.equal(ii, kk // 48)
