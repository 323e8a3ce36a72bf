"""Our kernels AND the CPU oracle against the reference's OWN CUDA kernels, compiled from the reference sources
into oracle/_ref by oracle/build_ref.py where those sources are at hand, and otherwise read from the outputs of
those kernels stored under tests/golden/ (tests/refdata.py).

This is what pins the oracle for altcorr / fastba, for which the reference ships no golden vectors:
the oracle must reproduce the reference kernels' outputs on the same seeded inputs, and so must we.
The reference kernels use unordered float atomics (ba_cuda.cu:339-373) and fp16 accumulation
(correlation_kernel.cu:121-131), so agreement is to a tolerance, stated per test.
"""
import os

import pytest
import torch

import refdata
from oracle import ba as OB, corr as OC, graph as OG
from dpvo_b200 import synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ref(ref_ext):
    """the reference kernels (oracle/_ref), or None where only their stored outputs are available"""
    return ref_ext


def _corr_case(seed, M, dtype, H=30, W=40, S1=40, S2=5):
    g = torch.Generator().manual_seed(seed)
    f1 = (torch.randn(1, S1, 128, 3, 3, generator=g) / 4).to(dtype)
    f2 = (torch.randn(1, S2, 128, H, W, generator=g) / 4).to(dtype)
    offs = torch.arange(3).float() - 1
    coords = torch.zeros(1, M, 2, 3, 3)
    coords[0, :, 0] = (torch.rand(M, generator=g) * (W + 10) - 5)[:, None, None] + 1.1 * offs[None, None, :]
    coords[0, :, 1] = (torch.rand(M, generator=g) * (H + 10) - 5)[:, None, None] + 0.9 * offs[None, :, None]
    ii = torch.randint(0, S1, (M,), generator=g)
    jj = torch.randint(0, S2, (M,), generator=g)
    return f1, f2, coords, ii, jj


def test_corr_forward_fp32_three_way(ext, ref):
    f1, f2, coords, ii, jj = _corr_case(31, 400, torch.float32)
    args = (f1.to(DEV), f2.to(DEV), coords.to(DEV), ii.to(DEV), jj.to(DEV), 3)
    R = refdata.reference("corr_fwd_fp32", ref, lambda rx: dict(out=rx[0].forward(*args)[0].cpu()))
    o, = ext[0].forward(*args)
    orc = OC.corr_forward(f1.double(), f2.double(), coords, ii, jj, 3)
    s = orc.abs().max().item()
    r = R["out"].double()
    assert (r - R.pick("out", orc)).abs().max().item() <= 2e-6 * s      # oracle == reference kernel
    assert (R.pick("out", o.cpu().double()) - r).abs().max().item() <= 2e-6 * s   # ours == reference kernel


def test_corr_forward_fp16_ours_is_closer_to_exact_than_reference(ext, ref):
    f1, f2, coords, ii, jj = _corr_case(32, 400, torch.half)
    args = (f1.to(DEV), f2.to(DEV), coords.to(DEV), ii.to(DEV), jj.to(DEV), 3)
    orc = OC.corr_forward(f1.double(), f2.double(), coords, ii, jj, 3)

    def compute(rx):
        r, = rx[0].forward(*args)
        return dict(out=r.cpu(), err_vs_exact=(r.cpu().double() - orc).abs().max().item())

    R = refdata.reference("corr_fwd_fp16", ref, compute)
    o, = ext[0].forward(*args)
    er = R["err_vs_exact"]
    eo = (o.cpu().double() - orc).abs().max().item()
    s = orc.abs().max().item()
    assert eo <= 2.0 ** -10 * s + 1e-4
    assert er <= 3e-2 * s            # half accumulation over 128 channels + half blend
    assert eo <= er                  # fp32 accumulation is at least as accurate
    assert (R.pick("out", o.cpu().double()) - R["out"].double()).abs().max().item() <= 3e-2 * s


def test_corr_backward_three_way(ext, ref):
    f1, f2, coords, ii, jj = _corr_case(33, 80, torch.float32, H=20, W=24, S1=20, S2=3)
    g = torch.Generator().manual_seed(34)
    grad = torch.randn(1, 80, 7, 7, 3, 3, generator=g)
    args = (f1.to(DEV), f2.to(DEV), coords.to(DEV), ii.to(DEV), jj.to(DEV), grad.to(DEV), 3)

    def compute(rx):
        r1, r2 = rx[0].backward(*args)
        return dict(fmap1_grad=r1.cpu(), fmap2_grad=r2.cpu())

    R = refdata.reference("corr_bwd_fp32", ref, compute)
    o1, o2 = ext[0].backward(*args)
    a = f1.double().requires_grad_(True)
    b = f2.double().requires_grad_(True)
    OC.corr_forward(a, b, coords, ii, jj, 3).backward(grad.double())
    for ours, k, orc in ((o1, "fmap1_grad", a.grad), (o2, "fmap2_grad", b.grad)):
        s = orc.abs().max().item()
        theirs = R[k].double()
        assert (theirs - R.pick(k, orc)).abs().max().item() <= 3e-5 * s
        assert (R.pick(k, ours.cpu().double()) - theirs).abs().max().item() <= 3e-5 * s


def test_patchify_matches_reference(ext, ref):
    g = torch.Generator().manual_seed(35)
    net = torch.randn(1, 384, 30, 40, generator=g).to(DEV)
    coords = torch.stack([torch.randint(1, 39, (1, 96), generator=g), torch.randint(1, 29, (1, 96), generator=g)], -1).float().to(DEV)
    R = refdata.reference("patchify", ref, lambda rx: {"r%d" % radius: rx[0].patchify_forward(net, coords, radius)[0].cpu()
                                                       for radius in (0, 1)})
    for radius in (0, 1):
        o, = ext[0].patchify_forward(net, coords, radius)
        assert R.equal("r%d" % radius, o.cpu())
        assert R.equal("r%d" % radius, OC.patchify_raw(net.cpu(), coords.cpu(), radius))


def test_neighbors_matches_reference(ext, ref):
    ii, jj, kk = synthetic.replay_edges(30, 48, 11, 16)
    R = refdata.reference("neighbors", ref, lambda rx: dict(zip(("ix", "jx"), [t.cpu() for t in rx[1].neighbors(kk.to(DEV), jj.to(DEV))])))
    o = ext[1].neighbors(kk.to(DEV), jj.to(DEV))
    orc = OG.neighbors(kk, jj)
    for k, b, c in zip(("ix", "jx"), o, orc):
        assert R.equal(k, b.cpu()) and R.equal(k, c)


@pytest.mark.parametrize("config,n_frames", [("fast", 30), ("default", 36)])
def test_ba_three_way(ext, ref, config, n_frames):
    st = synthetic.make_state(config, n_frames, device="cpu", features=False, seed=41)
    g = torch.Generator().manual_seed(42)
    coords = OB.fastba_reproject(st.poses.double(), st.patches.double(), st.intrinsics.double(), st.ii, st.jj, st.kk)
    target = (coords[:, :, 1, 1] + torch.randn(st.E, 2, generator=g).double()).float()
    weight = torch.rand(st.E, 2, generator=g)
    lm = torch.tensor([1e-4])
    rp, rpatch = OB.fastba_forward(st.poses.double(), st.patches.double(), st.intrinsics.double(), target.double(),
                                   weight.double(), lm.double(), st.ii, st.jj, st.kk, st.t0, st.n, 2)
    live = st.kk.unique()

    def run(mod):
        poses = st.poses.clone().to(DEV)[None]
        patches = st.patches.clone().to(DEV)[None]
        mod.forward(poses, patches, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], lm.to(DEV),
                    st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV), st.cfg["M"], st.t0, st.n, 2, False)
        return poses[0, :st.n].cpu().double(), patches[0].cpu().double()[live, 2]

    R = refdata.reference("ba_%s%d" % (config, n_frames), ref, lambda rx: dict(zip(("poses", "depth"), run(rx[1]))))
    ours = run(ext[1])

    def rel(a, b, bmax=None):
        return ((a - b).abs().max() / (b.abs().max() if bmax is None else bmax)).item()

    # oracle == reference kernel, ours == reference kernel, all to north_star's 1e-4 relative
    assert rel(R["poses"].double(), rp[:st.n]) < 1e-4 and rel(R["depth"].double(), R.pick("depth", rpatch[live, 2]), rpatch[live, 2].abs().max()) < 1e-4
    assert rel(ours[0], R["poses"].double()) < 1e-4 and rel(R.pick("depth", ours[1]), R["depth"].double(), R.absmax("depth")) < 1e-4


def test_reproject_matches_reference(ext, ref):
    st = synthetic.make_state("fast", 20, device=DEV, features=False, seed=43)
    args = (st.poses[None], st.patches[None], st.intrinsics[None], st.ii, st.jj, st.kk)
    R = refdata.reference("reproject", ref, lambda rx: dict(out=rx[1].reproject(*args).cpu()))
    o = ext[1].reproject(*args)
    assert (R["out"] - R.pick("out", o.cpu())).abs().max().item() < 1e-3


def test_write_golden_fixtures_from_reference_kernels(ref):
    """Not a check of ours: regenerates the small fixtures committed under tests/golden/ from the
    REFERENCE kernels, into $DPVO_GOLDEN_OUT.  tests/test_oracle_cpu.py then holds the CPU oracle to
    them without a GPU."""
    out_dir = os.environ.get("DPVO_GOLDEN_OUT")
    if not out_dir or ref is None:
        pytest.skip("set DPVO_GOLDEN_OUT and build oracle/_ref to regenerate fixtures")
    os.makedirs(out_dir, exist_ok=True)
    f1, f2, coords, ii, jj = _corr_case(51, 48, torch.float32, H=16, W=20, S1=12, S2=2)
    c, = ref[0].forward(f1.to(DEV), f2.to(DEV), coords.to(DEV), ii.to(DEV), jj.to(DEV), 3)
    g = torch.Generator().manual_seed(52)
    grad = torch.randn(1, 48, 7, 7, 3, 3, generator=g)
    g1, g2 = ref[0].backward(f1.to(DEV), f2.to(DEV), coords.to(DEV), ii.to(DEV), jj.to(DEV), grad.to(DEV), 3)
    torch.save(dict(fmap1=f1, fmap2=f2, coords=coords, ii=ii, jj=jj, radius=3, out=c.cpu(), grad=grad,
                    fmap1_grad=g1.cpu(), fmap2_grad=g2.cpu(), source="ref_cuda_corr (correlation_kernel.cu) on B200"),
               os.path.join(out_dir, "corr_ref_fp32.pt"))
    st = synthetic.make_state("fast", 12, device="cpu", features=False, seed=53, buffer=16)
    coords2 = OB.fastba_reproject(st.poses.double(), st.patches.double(), st.intrinsics.double(), st.ii, st.jj, st.kk)
    target = (coords2[:, :, 1, 1] + torch.randn(st.E, 2, generator=g).double()).float()
    weight = torch.rand(st.E, 2, generator=g)
    poses = st.poses.clone().to(DEV)[None]
    patches = st.patches.clone().to(DEV)[None]
    ref[1].forward(poses, patches, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None],
                   torch.tensor([1e-4], device=DEV), st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV), 48, st.t0, st.n, 2, False)
    ix, jx = ref[1].neighbors(st.kk.to(DEV), st.jj.to(DEV))
    rep = ref[1].reproject(st.poses.to(DEV)[None], st.patches.to(DEV)[None], st.intrinsics.to(DEV)[None],
                           st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV))
    live = st.kk.unique()
    torch.save(dict(poses=st.poses[:st.n], patches=st.patches[:st.n * 48], intrinsics=st.intrinsics[:st.n],
                    target=target, weight=weight, ii=st.ii, jj=st.jj, kk=st.kk, t0=st.t0, t1=st.n,
                    poses_out=poses[0, :st.n].cpu(), depth_out=patches[0, :st.n * 48, 2, 0, 0].cpu(), live=live,
                    neighbors_ix=ix.cpu(), neighbors_jx=jx.cpu(), reproject=rep.cpu().half(),
                    source="ref_cuda_ba (ba_cuda.cu, ba.cpp) on B200"),
               os.path.join(out_dir, "ba_ref_fast12.pt"))
