"""The drop-in, exercised: the reference's UNMODIFIED Python host code (packed by oracle/build_ref.py into
oracle/_ref/dpvo_ref_py.zip) running on top of OUR native modules -- dpvo/altcorr/correlation.py,
dpvo/fastba/ba.py, dpvo/lietorch (with the reference's own run_tests.py), dpvo/net.py:Update, and the whole
DPVO class of dpvo/dpvo.py on a synthetic stream -- and one DPVO.update() (dpvo.py:328-360) from an identical
state on our kernels vs the reference's own CUDA kernels (oracle/_ref), poses and inverse depths compared at
north_star's 1e-4 relative bar."""
import importlib
import os
import sys

import pytest
import torch

import refdata
from oracle import ba as OB, corr as OC, refimport
from dpvo_b200 import synthetic

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def refpy(ext):
    if not refimport.staged():
        pytest.skip("oracle/_ref/dpvo_ref_py.zip not staged")
    with refimport.reference_python(native=ext[:3]):
        import dpvo.altcorr.correlation as C
        import dpvo.fastba as FB
        import dpvo.lietorch as LT
        import dpvo.projective_ops as PO
        import dpvo.net as RN
        assert C.__file__.startswith(refimport.REF_ZIP) and C.cuda_corr is ext[0] and sys.modules["cuda_ba"] is ext[1]
        yield dict(corr=C, fastba=FB, lietorch=LT, pops=PO, net=RN)


def _corr_case(seed, M, H=24, W=32, S1=30, S2=4):
    g = torch.Generator().manual_seed(seed)
    f1 = torch.randn(1, S1, 128, 3, 3, generator=g) / 4
    f2 = torch.randn(1, S2, 128, H, W, generator=g) / 4
    offs = torch.arange(3).float() - 1
    coords = torch.zeros(1, M, 2, 3, 3)
    coords[0, :, 0] = (torch.rand(M, generator=g) * (W + 6) - 3)[:, None, None] + 1.05 * offs[None, None, :]
    coords[0, :, 1] = (torch.rand(M, generator=g) * (H + 6) - 3)[:, None, None] + 0.95 * offs[None, :, None]
    return f1, f2, coords, torch.randint(0, S1, (M,), generator=g), torch.randint(0, S2, (M,), generator=g)


def test_reference_altcorr_autograd_on_our_kernels(refpy):
    """dpvo/altcorr/correlation.py:4-30 CorrLayer (forward AND backward through autograd) on our cuda_corr"""
    f1, f2, coords, ii, jj = _corr_case(91, 120)
    a = f1.to(DEV).requires_grad_(True)
    b = f2.to(DEV).requires_grad_(True)
    out = refpy["corr"].corr(a, b, coords.to(DEV), ii.to(DEV), jj.to(DEV), 3, 1)     # dropout = 1: no subsampling
    g = torch.Generator().manual_seed(92)
    grad = torch.randn(out.shape, generator=g)
    out.backward(grad.to(DEV))
    a64 = f1.double().requires_grad_(True)
    b64 = f2.double().requires_grad_(True)
    ref = OC.corr_forward(a64, b64, coords, ii, jj, 3)
    ref.backward(grad.double())
    s = ref.abs().max().item()
    assert (out.detach().cpu().double() - ref.detach()).abs().max().item() <= 1e-5 * s
    for mine, theirs in ((a.grad, a64.grad), (b.grad, b64.grad)):
        assert (mine.cpu().double() - theirs).abs().max().item() <= 3e-5 * theirs.abs().max().item()


def test_reference_patchify_bilinear_autograd_on_our_kernels(refpy):
    """correlation.py:33-69 PatchLayer + the Python-side bilinear blend on our patchify kernels"""
    g = torch.Generator().manual_seed(93)
    net = torch.randn(2, 16, 20, 28, generator=g)
    coords = torch.stack([torch.rand(2, 40, generator=g) * 24 + 1.5, torch.rand(2, 40, generator=g) * 16 + 1.5], -1)
    x = net.to(DEV).requires_grad_(True)
    out = refpy["corr"].patchify(x, coords.to(DEV), 1)
    grad = torch.randn(out.shape, generator=g)
    out.backward(grad.to(DEV))
    x64 = net.double().requires_grad_(True)
    # bilinear sampling of the 3x3 window around each (fractional) centre == F.grid_sample, align_corners
    H, W = net.shape[-2:]
    offs = torch.tensor([-1.0, 0.0, 1.0], dtype=torch.float64)
    gx = coords[..., 0].double()[:, :, None, None] + offs[None, None, None, :]
    gy = coords[..., 1].double()[:, :, None, None] + offs[None, None, :, None]
    gx, gy = torch.broadcast_tensors(gx, gy)
    grid = torch.stack([2 * gx / (W - 1) - 1, 2 * gy / (H - 1) - 1], -1).view(2, 40 * 3, 3, 2)
    ref = torch.nn.functional.grid_sample(x64, grid, mode="bilinear", align_corners=True)       # [2,C,120,3]
    ref = ref.view(2, 16, 40, 3, 3).permute(0, 2, 1, 3, 4)
    ref.backward(grad.double())
    assert (out.detach().cpu().double() - ref.detach()).abs().max().item() < 1e-5
    assert (x.grad.cpu().double() - x64.grad).abs().max().item() < 1e-4


def test_reference_fastba_wrapper_on_our_kernels(refpy):
    """dpvo/fastba/ba.py:7-8 BA(...) -> our cuda_ba.forward, vs the fp64 oracle at north_star's 1e-4"""
    st = synthetic.make_state("fast", 20, device="cpu", features=False, seed=94)
    g = torch.Generator().manual_seed(95)
    coords = OB.fastba_reproject(st.poses.double(), st.patches.double(), st.intrinsics.double(), st.ii, st.jj, st.kk)
    target = (coords[:, :, 1, 1] + torch.randn(st.E, 2, generator=g).double()).float()
    weight = torch.rand(st.E, 2, generator=g)
    lm = torch.tensor([1e-4])
    rp, rq = OB.fastba_forward(st.poses.double(), st.patches.double(), st.intrinsics.double(), target.double(), weight.double(),
                               lm.double(), st.ii, st.jj, st.kk, st.t0, st.n, 2)
    poses, patches = st.poses.clone().to(DEV)[None], st.patches.clone().to(DEV)[None]
    refpy["fastba"].BA(poses, patches, st.intrinsics.to(DEV)[None], target.to(DEV)[None], weight.to(DEV)[None], lm.to(DEV),
                       st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV), st.t0, st.n, M=st.cfg["M"], iterations=2, eff_impl=False)
    live = st.kk.unique()
    assert ((poses[0, :st.n].cpu().double() - rp[:st.n]).abs().max() / rp[:st.n].abs().max()).item() < 1e-4
    assert ((patches[0].cpu().double()[live, 2] - rq[live, 2]).abs().max() / rq[live, 2].abs().max()).item() < 1e-4


def test_reference_lietorch_run_tests_cuda_on_our_backend(refpy, ext):
    """the GPU half of dpvo/lietorch/run_tests.py:270-290 (forward identities + Jacobian checks, the file's own
    tolerances), the reference's groups.py / group_ops.py / gradcheck.py on OUR lietorch_backends"""
    z = refimport.REF_ZIP
    saved = list(sys.path)
    sys.path[:0] = [z + "/dpvo/lietorch", z + "/dpvo"]
    for m in ("lietorch", "gradcheck", "run_tests"):
        sys.modules.pop(m, None)
    try:
        assert sys.modules["lietorch_backends"] is ext[2]
        torch.manual_seed(1234)
        rt = importlib.import_module("run_tests")
        import lietorch as LT
        n = 0
        for Group in (LT.SO3, LT.RxSO3, LT.SE3, LT.Sim3):
            for fn in (rt.test_exp_log, rt.test_inv, rt.test_adj, rt.test_act):
                fn(Group, device="cuda"); n += 1
            tol = 1e-3 if Group is LT.Sim3 else 1e-8
            rt.test_exp_log_grad(Group, device="cuda", tol=tol)
            rt.test_inv_log_grad(Group, device="cuda", tol=tol)
            for fn in (rt.test_adj_grad, rt.test_adjT_grad, rt.test_act_grad, rt.test_matrix_grad,
                       rt.extract_translation_grad, rt.test_vec_grad, rt.test_fromvec_grad):
                fn(Group, device="cuda")
            n += 9
        assert n == 52
    finally:
        sys.path[:] = saved
        for m in ("lietorch", "gradcheck", "run_tests"):
            sys.modules.pop(m, None)


def test_reference_transform_jacobians_on_our_lietorch(refpy):
    """dpvo/projective_ops.py:53-113 transform(jacobian=True) (SE3 mul / inv / act4 / adjT through our
    lietorch_backends) vs the oracle restatement, which is pinned bit-exactly to the same file on the CPU"""
    st = synthetic.make_state("fast", 14, device="cpu", features=False, seed=96, noise=0.02)
    SE3 = refpy["lietorch"].SE3
    args = (st.ii, st.jj, st.kk)
    x, v, (Ji, Jj, Jz) = refpy["pops"].transform(SE3(st.poses.to(DEV)[None]), st.patches.to(DEV)[None], st.intrinsics.to(DEV)[None],
                                                 *[a.to(DEV) for a in args], jacobian=True)
    ox, ov, (oJi, oJj, oJz) = OB.transform(st.poses.double()[None], st.patches.double()[None], st.intrinsics.double()[None],
                                           *args, jacobian=True)
    for mine, theirs in ((x, ox), (v, ov), (Ji, oJi), (Jj, oJj), (Jz, oJz)):
        assert (mine.cpu().double() - theirs).abs().max().item() <= 2e-4 * max(1.0, theirs.abs().max().item())


@pytest.mark.parametrize("config,n_frames", [("fast", 14)])
def test_reference_update_module_vs_ours_same_weights(ext, config, n_frames):
    """dpvo/net.py:Update (torch, autocast as dpvo.py:332, calling OUR cuda_ba.neighbors) vs dpvo_b200.net.Update
    (tcgen05) with the same state_dict, both against the reference module in fp32: ours no worse than 2x the
    reference's own mixed-precision error.  The reference module runs live where its package is staged, else its
    stored outputs stand in (tests/refdata.py); either way ours is also held, on every element, to the fp32
    restatement oracle/update.py with the same weights."""
    from dpvo_b200.net import Update
    from oracle import update as OU
    st = synthetic.make_state(config, n_frames, device="cpu", features=False)
    E = st.E
    torch.manual_seed(1234)
    weights = OU.Update(3).state_dict()              # net.py:28-72 construction order: the reference module's seeded weights
    ours = Update(3).to(DEV).eval()
    ours.load_state_dict(weights)
    mod32 = OU.Update(3).to(DEV).eval()
    mod32.load_state_dict(weights)
    g = torch.Generator().manual_seed(64)
    net = (torch.randn(1, E, 384, generator=g) * 0.5).to(DEV)
    inp = (torch.randn(1, E, 384, generator=g) * 0.25).half().to(DEV)
    corr = (torch.randn(1, E, 882, generator=g) * 2).half().to(DEV)
    ii, jj, kk = st.ii.to(DEV), st.jj.to(DEV), st.kk.to(DEV)

    def err(a, b):
        return (a.float() - b.float()).abs().max().item()

    def compute(_):
        with refimport.reference_python(native=ext[:3]):
            import dpvo.net as RN
            ref_mod = RN.Update(3).to(DEV).eval()
            ref_mod.load_state_dict(weights)
            with torch.no_grad():
                rn, (rd, rw, _) = ref_mod(net, inp.float(), corr.float(), None, ii, jj, kk)
                with torch.autocast("cuda", dtype=torch.half):
                    an, (ad, aw, _) = ref_mod(net, inp, corr, None, ii, jj, kk)
        return dict(net=rn.float(), delta=rd.float(), weight=rw.float(),
                    autocast_err_net=err(an, rn), autocast_err_delta=err(ad, rd), autocast_err_weight=err(aw, rw))

    R = refdata.reference("update_module_%s%d" % (config, n_frames), refimport if refimport.staged() else None, compute)
    with torch.no_grad():
        on, (od, ow, _) = ours(net, inp, corr, None, ii, jj, kk)
        n32, (d32, w32, _) = mod32(net, inp.float(), corr.float(), None, ii, jj, kk)

    mine = {"net": on, "delta": od, "weight": ow}
    e = {k: err(R.pick(k, mine[k]), R[k].to(DEV)) for k in mine}
    print("ours vs fp32:", e["net"], e["delta"], e["weight"],
          " autocast vs fp32:", R["autocast_err_net"], R["autocast_err_delta"], R["autocast_err_weight"])
    for k, o32, bar in (("net", n32, 2e-2), ("delta", d32, 1e-2), ("weight", w32, 5e-3)):
        assert e[k] <= max(2 * R["autocast_err_" + k], bar), k
        assert err(mine[k], o32) <= max(2 * R["autocast_err_" + k], bar), k


# ------------------------------------------------------------------------------ the whole DPVO class
@pytest.fixture(scope="module")
def slam_fast():
    if not refimport.staged():
        pytest.skip("oracle/_ref/dpvo_ref_py.zip not staged")
    from oracle import ref_pipeline as RP
    try:
        RP.ref_native()
    except ImportError:
        pytest.skip("oracle/_ref kernels not built")
    r = RP.RefDPVO("fast", native="ours", update="reference", seed=1234)
    r.feed(RP.make_stream("fast", 20, seed=3))
    yield r
    r.close()


def _rel(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max()).item()


def test_reference_dpvo_class_runs_on_our_modules(slam_fast):
    """dpvo/dpvo.py, unmodified: 20 frames through DPVO.__call__ (patchify, motion probe, initialisation with 12
    updates, per-frame update + keyframe) with cuda_corr / cuda_ba / lietorch_backends all ours"""
    s = slam_fast.slam
    assert s.is_initialized and s.n >= 8
    assert s.pg.ii.numel() > 0 and s.pg.net.shape[1] == s.pg.ii.numel()
    assert torch.isfinite(s.pg.poses_[:s.n]).all() and torch.isfinite(s.pg.patches_[:s.n]).all()
    q = s.pg.poses_[:s.n, 3:]
    assert (q.norm(dim=-1) - 1).abs().max().item() < 1e-4


def test_one_dpvo_update_ours_vs_reference_kernels(slam_fast):
    """ONE DPVO.update() from an identical mid-stream state: (a) reference kernels + reference Update (the
    reference CUDA pipeline), (b) our kernels + reference Update, (c) our kernels + our Update.
    Same target/weight => BA outputs at north_star's 1e-4; the full update differs by the fp16-accumulated
    correlation of the reference (3e-2 on corr) so its bar is the update's own mixed-precision noise."""
    r = slam_fast
    snap = r.snapshot()
    outs = {}
    for name, native, upd in (("ref", "ref", "reference"), ("ours_kernels", "ours", "reference"), ("ours_all", "ours", "ours")):
        r.restore(snap)
        r.use(native, upd)
        outs[name] = r.update_once()
    r.restore(snap)
    r.use("ours", "reference")
    n = r.slam.n
    a, b, c = outs["ref"], outs["ours_kernels"], outs["ours_all"]
    print("n=%d E=%d" % (n, r.slam.pg.ii.numel()))
    for nm, o in (("ours_kernels", b), ("ours_all", c)):
        print(nm, "vs reference CUDA pipeline: pose rel %.3g, depth rel %.3g, target abs %.3g px, weight abs %.3g, net abs %.3g" %
              (_rel(o["poses"], a["poses"]), _rel(o["depth"], a["depth"]), (o["target"] - a["target"]).abs().max().item(),
               (o["weight"] - a["weight"]).abs().max().item(), (o["net"] - a["net"]).abs().max().item()))
    for o in (b, c):
        assert torch.isfinite(o["poses"]).all() and torch.isfinite(o["depth"]).all()
        assert (o["target"] - a["target"]).abs().max().item() < 0.25          # px; reference corr is fp16-accumulated
        assert (o["weight"] - a["weight"]).abs().max().item() < 0.05
        assert _rel(o["poses"], a["poses"]) < 2e-3 and _rel(o["depth"], a["depth"]) < 2e-2


def test_dpvo_update_ba_stage_matches_reference_kernels_given_same_target(slam_fast):
    """the BA stage of DPVO.update() in isolation: the target / weight produced by the reference pipeline fed to
    both cuda_ba.forward implementations through the reference's fastba.BA -> 1e-4 relative on poses and depths"""
    r = slam_fast
    snap = r.snapshot()
    r.use("ref", "reference")
    ref_out = r.update_once()
    s = r.slam
    t0 = max(s.n - s.cfg.OPTIMIZATION_WINDOW, 1)
    res = {}
    for native in ("ref", "ours"):
        r.restore(snap)
        r.use(native)
        lm = torch.as_tensor([1e-4], device=DEV)
        r.mods["dpvo.fastba"].BA(s.poses, s.patches, s.intrinsics, ref_out["target"], ref_out["weight"], lm,
                                 s.pg.ii, s.pg.jj, s.pg.kk, t0, s.n, M=s.M, iterations=2, eff_impl=False)
        res[native] = (s.pg.poses_[:s.n].clone(), s.pg.patches_[:s.n, :, 2, 1, 1].clone())
    r.restore(snap)
    r.use("ours", "reference")
    assert _rel(res["ours"][0], res["ref"][0]) < 1e-4 and _rel(res["ours"][1], res["ref"][1]) < 1e-4
