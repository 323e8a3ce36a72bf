"""cuda_ba.forward / reproject on the device vs the fp64 CPU oracle.  north_star bar: poses and
inverse depths within 1e-4 relative."""
import pytest
import torch

import refdata
from oracle import ba as OB
from dpvo_b200 import synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _problem(config, n_frames, seed, sigma=1.0):
    st = synthetic.make_state(config, n_frames, device="cpu", features=False, seed=seed)
    g = torch.Generator().manual_seed(seed)
    P = 3
    coords = OB.fastba_reproject(st.poses.double(), st.patches.double(), st.intrinsics.double(), st.ii, st.jj, st.kk)
    target = (coords[:, :, 1, 1] + sigma * torch.randn(st.E, 2, generator=g).double()).float()
    weight = torch.rand(st.E, 2, generator=g)
    return st, target, weight


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp(min=1e-12)).item()


@pytest.mark.parametrize("config,n_frames,iters", [("fast", 12, 1), ("fast", 30, 2), ("default", 36, 2)])
def test_ba_forward_matches_oracle(ext, config, n_frames, iters):
    st, target, weight = _problem(config, n_frames, 21)
    lm = torch.tensor([1e-4])
    t0, t1 = st.t0, st.n
    rp, rpatch = OB.fastba_forward(st.poses.double(), st.patches.double(), st.intrinsics.double(), target.double(),
                                   weight.double(), lm.double(), st.ii, st.jj, st.kk, t0, t1, iters)
    poses = st.poses.clone().to(DEV)[None]
    patches = st.patches.clone().to(DEV)[None]
    ext[1].forward(poses, patches, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], lm.to(DEV),
                   st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV), st.cfg["M"], t0, t1, iters, False)
    torch.cuda.synchronize()
    dp = (rp - st.poses.double()).abs().max().item()
    assert dp > 1e-4, "degenerate problem: BA did not move the poses"
    assert _rel(poses[0].cpu().double()[:t1], rp[:t1]) < 1e-4
    live = st.kk.unique()
    assert _rel(patches[0].cpu().double()[live, 2], rpatch[live, 2]) < 1e-4
    # untouched state stays bit-identical: fixed poses, x/y of patches, patches without edges
    assert torch.equal(poses[0, :t0].cpu(), st.poses[:t0])
    assert torch.equal(patches[0, :, :2].cpu(), st.patches[:, :2])
    # the update is a real correction, not noise: compare step against oracle step
    assert _rel(poses[0].cpu().double()[t0:t1] - st.poses.double()[t0:t1], rp[t0:t1] - st.poses.double()[t0:t1]) < 2e-3


@pytest.mark.parametrize("t0", [2, 12])
def test_ba_many_free_poses(ext, t0):
    """wide optimisation windows (28 and 18 free poses of the 32 the on-chip solver holds): the Schur tiles no
    longer fit one round of the CTA, the Cholesky runs 28 panels"""
    st, target, weight = _problem("fast", 30, 23, sigma=0.5)
    lm = torch.tensor([1e-4])
    t1 = st.n
    rp, rpatch = OB.fastba_forward(st.poses.double(), st.patches.double(), st.intrinsics.double(), target.double(),
                                   weight.double(), lm.double(), st.ii, st.jj, st.kk, t0, t1, 2)
    poses = st.poses.clone().to(DEV)[None]
    patches = st.patches.clone().to(DEV)[None]
    ext[1].forward(poses, patches, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], lm.to(DEV),
                   st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV), st.cfg["M"], t0, t1, 2, False)
    torch.cuda.synchronize()
    assert _rel(poses[0].cpu().double()[:t1], rp[:t1]) < 1e-4
    live = st.kk.unique()
    assert _rel(patches[0].cpu().double()[live, 2], rpatch[live, 2]) < 1e-4
    assert torch.equal(poses[0, :t0].cpu(), st.poses[:t0])


def test_ba_is_deterministic(ext):
    st, target, weight = _problem("fast", 30, 22)
    lm = torch.tensor([1e-4], device=DEV)
    outs = []
    for _ in range(2):
        poses = st.poses.clone().to(DEV)[None]
        patches = st.patches.clone().to(DEV)[None]
        ext[1].forward(poses, patches, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], lm,
                       st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV), st.cfg["M"], st.t0, st.n, 2, False)
        outs.append((poses.cpu(), patches.cpu()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


@pytest.mark.parametrize("config,n_frames", [("fast", 30), ("default", 36)])
def test_ba_grouped_entry_matches_plain_entry(ext, config, n_frames):
    """dpvo_ba_forward_grouped on groupings built by the caller vs cuda_ba.forward (which builds them): the same
    arithmetic on the same groups; the members of a kk group may arrive in another order (the caller's grouping
    uses jj as a secondary key, cuda_ba.forward's does not), which moves fp32 sums by an ulp or two -- hence a
    1e-5 relative bar rather than bit equality (two runs of either entry ARE bit-identical: test_ba_is_deterministic)"""
    from dpvo_b200.net import EdgeGroups
    from dpvo_b200 import fastba
    st, target, weight = _problem(config, n_frames, 27)
    lm = torch.tensor([1e-4], device=DEV)
    ii, jj, kk = st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV)
    p1, q1 = st.poses.clone().to(DEV)[None], st.patches.clone().to(DEV)[None]
    ext[1].forward(p1, q1, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], lm, ii, jj, kk,
                   st.cfg["M"], st.t0, st.n, 2, False)
    p2, q2 = st.poses.clone().to(DEV)[None], st.patches.clone().to(DEV)[None]
    gk, gp = EdgeGroups(kk, None, jj), EdgeGroups(ii, jj, None)       # kk groups may carry any member order
    fastba.BA_grouped(p2, q2, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], lm, ii, jj, kk,
                      st.t0, st.n, 2, gk, gp)
    live = st.kk.unique().to(DEV)
    assert _rel(p2[0, :st.n], p1[0, :st.n]) < 1e-5 and _rel(q2[0, live, 2], q1[0, live, 2]) < 1e-5


def test_ba_structure_only(ext):
    """t1 - t0 == 0: depth-only branch (ba_cuda.cu:521-531)"""
    st, target, weight = _problem("fast", 12, 23)
    lm = torch.tensor([1e-4])
    rp, rpatch = OB.fastba_forward(st.poses.double(), st.patches.double(), st.intrinsics.double(), target.double(),
                                   weight.double(), lm.double(), st.ii, st.jj, st.kk, st.n, st.n, 2)
    poses = st.poses.clone().to(DEV)[None]
    patches = st.patches.clone().to(DEV)[None]
    ext[1].forward(poses, patches, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], lm.to(DEV),
                   st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV), st.cfg["M"], st.n, st.n, 2, False)
    assert torch.equal(poses[0].cpu(), st.poses)
    live = st.kk.unique()
    assert _rel(patches[0].cpu().double()[live, 2], rpatch[live, 2]) < 1e-4


def test_ba_outliers_and_clamps(ext):
    """huge residuals are gated (>=128 px), depths are clamped as ba_cuda.cu:218-221"""
    st, target, weight = _problem("fast", 12, 24, sigma=60.0)
    st.patches[::7, 2] = 19.9
    st.patches[3::7, 2] = 2e-4
    lm = torch.tensor([1e-4])
    rp, rpatch = OB.fastba_forward(st.poses.double(), st.patches.double(), st.intrinsics.double(), target.double(),
                                   weight.double(), lm.double(), st.ii, st.jj, st.kk, st.t0, st.n, 2)
    poses = st.poses.clone().to(DEV)[None]
    patches = st.patches.clone().to(DEV)[None]
    ext[1].forward(poses, patches, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], lm.to(DEV),
                   st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV), st.cfg["M"], st.t0, st.n, 2, False)
    live = st.kk.unique()
    d = patches[0].cpu().double()[live, 2, 0, 0]
    r = rpatch[live, 2, 0, 0]
    # the residual gate (|r| < 128 px) and the clamp branches are discontinuous, so an edge that sits
    # on a threshold may fall on different sides in fp32 and fp64: require agreement for >= 99 % of
    # the patches and bounded drift of the poses
    close = (d - r).abs() <= 1e-3 * r.abs() + 1e-6
    assert close.float().mean().item() > 0.99, close.float().mean().item()
    # both clamp branches of ba_cuda.cu:218-221 were exercised by this problem, on the oracle and on the device
    assert (r == 1.0).any() and (d == 1.0).any(), "no depth took the d > 20 -> 1.0 branch"
    lo = float(torch.tensor(1e-4, dtype=torch.float32))
    assert (r <= 1e-4 * (1 + 1e-6)).any() and (d == lo).any(), "no depth was clamped to 1e-4"
    assert (d >= float(torch.tensor(1e-4, dtype=torch.float32))).all() and (d <= 20.0).all()
    assert _rel(poses[0].cpu().double()[:st.n], rp[:st.n]) < 2e-2


def test_reproject_both_modes(ext):
    st, _, _ = _problem("fast", 20, 25)
    ii, jj, kk = st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV)
    out = ext[1].reproject(st.poses.to(DEV)[None], st.patches.to(DEV)[None], st.intrinsics.to(DEV)[None], ii, jj, kk)
    ref = OB.fastba_reproject(st.poses.double(), st.patches.double(), st.intrinsics.double(), st.ii, st.jj, st.kk)
    assert out.shape == (1, st.E, 2, 3, 3)
    assert (out[0].cpu().double() - ref).abs().max().item() < 2e-3       # pixels, fp32 vs fp64
    out2 = ext[3].reproject_clamped(st.poses.to(DEV)[None], st.patches.to(DEV)[None], st.intrinsics.to(DEV)[None], ii, jj, kk)
    ref2 = OB.transform(st.poses.double()[None], st.patches.double()[None], st.intrinsics.double()[None], st.ii, st.jj, st.kk)
    assert (out2[0].cpu().double() - ref2[0].permute(0, 3, 1, 2)).abs().max().item() < 2e-3


def _wide_graph(n_frames=40, M=24, seed=60):
    """a long window with a few loop-closure style long-range edges: the shape global BA sees (dpvo.py:312-326)"""
    st = synthetic.make_state(dict(M=M, lifetime=8, removal=40, opt_window=39, ht=480, wd=640, intrinsics=(320.0, 320.0, 320.0, 240.0)),
                              n_frames, device="cpu", features=False, seed=seed, buffer=n_frames + 2, mem=n_frames + 2)
    # long-range edges: patches of frames 0..2 observed again in the last three frames
    g = torch.Generator().manual_seed(seed)
    kk_l = torch.arange(0, 3 * M).repeat_interleave(3)
    jj_l = torch.arange(n_frames - 3, n_frames).repeat(3 * M)
    st.ii = torch.cat([st.ii, kk_l // M]); st.jj = torch.cat([st.jj, jj_l]); st.kk = torch.cat([st.kk, kk_l])
    coords = OB.fastba_reproject(st.poses.double(), st.patches.double(), st.intrinsics.double(), st.ii, st.jj, st.kk)
    target = (coords[:, :, 1, 1] + torch.randn(st.E, 2, generator=g).double()).float()
    weight = torch.rand(st.E, 2, generator=g)
    return st, target, weight


@pytest.mark.parametrize("eff_impl,t0", [(True, 1), (False, 1), (True, 20)])
def test_ba_wide_window_and_eff_impl_match_oracle_and_reference_kernel(ext, ref_ext, eff_impl, t0):
    """cuda_ba.forward with eff_impl=True (block_e.cu path of the reference) and / or more than 32 free poses: our
    per-frame Schur product (ba_wide.cu) vs the dense fp64 oracle and vs the reference's own kernel, 1e-4 relative"""
    st, target, weight = _wide_graph()
    lm = torch.tensor([1e-4])
    rp, rq = OB.fastba_forward(st.poses.double(), st.patches.double(), st.intrinsics.double(), target.double(), weight.double(),
                               lm.double(), st.ii, st.jj, st.kk, t0, st.n, 2)
    live = st.kk.unique()

    def run(mod):
        poses, patches = st.poses.clone().to(DEV)[None], st.patches.clone().to(DEV)[None]
        mod.forward(poses, patches, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], lm.to(DEV),
                    st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV), st.cfg["M"], t0, st.n, 2, eff_impl)
        return poses[0, :st.n].cpu().double(), patches[0].cpu().double()[live, 2]

    ours = run(ext[1])
    R = refdata.reference("ba_wide_%s_t%d" % ("eff" if eff_impl else "dense", t0), ref_ext,
                          lambda rx: dict(zip(("poses", "depth"), run(rx[1]))))
    assert st.n - t0 > 32 or eff_impl
    for p, q, pick in ((ours[0], ours[1], lambda x: x), (R["poses"].double(), R["depth"].double(), lambda x: R.pick("depth", x))):
        assert torch.isfinite(p).all() and torch.isfinite(q).all()
        assert _rel(p, rp[:st.n]) < 1e-4
        assert ((q - pick(rq[live, 2])).abs().max() / rq[live, 2].abs().max()).item() < 1e-4
    assert (ours[0] - st.poses[:st.n].double()).abs().max().item() > 1e-4      # the step moved the poses
    if t0 > 1:
        assert torch.equal(ours[0][:t0].float(), st.poses[:t0])                 # poses before t0 stay fixed


def test_ba_wide_rejects_patch_ids_outside_their_frame(ext):
    st, target, weight = _wide_graph(n_frames=36, M=8)
    kk_bad = st.kk.clone()
    kk_bad[5] = kk_bad[5] + 8                      # patch no longer belongs to frame ii[5]
    poses, patches = st.poses.clone().to(DEV)[None], st.patches.clone().to(DEV)[None]
    with pytest.raises(RuntimeError):
        ext[1].forward(poses, patches, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], torch.tensor([1e-4], device=DEV),
                       st.ii.to(DEV), st.jj.to(DEV), kk_bad.to(DEV), 8, 1, st.n, 1, True)


def test_solve_system_matches_dense_restatement(ext):
    """cuda_ba.solve_system (ba.cpp:120-180): A = J^T J with 7x7 blocks, damping, solve of the leading freen poses"""
    g = torch.Generator().manual_seed(70)
    n, r = 12, 40
    ii = torch.randint(0, n, (r,), generator=g)
    jj = (ii + 1 + torch.randint(0, n - 1, (r,), generator=g)) % n
    Ji = torch.randn(r, 7, 7, generator=g) * 0.5 + torch.eye(7)
    Jj = torch.randn(r, 7, 7, generator=g) * 0.5 - torch.eye(7)
    res = torch.randn(r, 7, generator=g)
    for freen in (-1, 9):
        out, = ext[1].solve_system(Ji.to(DEV), Jj.to(DEV), ii.to(DEV), jj.to(DEV), res.to(DEV), 1e-3, 1e-4, freen)
        ref = OB.posegraph_solve(Ji.double(), Jj.double(), ii, jj, res.double(), 1e-3, 1e-4, freen)
        assert out.shape == (n, 7) and out.dtype == torch.float32
        assert (out.cpu().double() - ref).abs().max().item() <= 1e-5 * max(1.0, ref.abs().max().item())
        if freen > 0:
            assert torch.equal(out[freen:].cpu(), torch.zeros(n - freen, 7))
