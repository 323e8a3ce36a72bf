"""The step the bench times -- UpdateRunner.step(): reproject_clamped -> corr_fwd_tc on the real feature ring ->
tcgen05 Update -> grouped BA -- end to end on BASELINE configs[1] (default, E = 47,712) and configs[2] (fast,
E = 14,496), eager and as a CUDA graph, against
  (1) the composed fp32 oracle (oracle/ba.py transform + oracle/corr.py + oracle/update.py + fastba_forward fp64), and
  (2) the reference CUDA pipeline (oracle/ref_pipeline.py:RefCudaStep: the reference's own correlation and BA
      kernels from oracle/_ref around the torch Update under autocast, exactly DPVO.update's data flow), run live
      where oracle/_ref is built and otherwise read from its stored errors and outputs (tests/refdata.py).
Bars.  BA stage given the same target/weight: north_star's 1e-4 relative on poses and inverse depths.  Whole
update: ours may be no further from the fp32 oracle than 2x what the reference CUDA pipeline is (its fp16
correlation accumulation and autocast GEMMs set the noise floor of this path)."""
import pytest
import torch

import refdata
from oracle import ba as OB, corr as OC, update as OU
from dpvo_b200 import synthetic
from dpvo_b200.runner import UpdateRunner

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _rel(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max()).item()


@torch.no_grad()
def composed_oracle_step(st, mod32, net, kk_ring, jj_ring, iters=2):
    """fp32 everywhere (fp64 BA), oracle functions only, on the device for speed"""
    poses, patches, intr = st.poses[None], st.patches[None], st.intrinsics[None]
    coords = OB.transform(poses, patches, intr, st.ii, st.jj, st.kk).permute(0, 1, 4, 2, 3).contiguous()
    g, f1, f2 = st.gmap.float().contiguous(), st.fmap1.float().contiguous(), st.fmap2.float().contiguous()
    c0 = OC.corr_forward(g, f1, coords, kk_ring, jj_ring, 3, chunk=128)
    c1 = OC.corr_forward(g, f2, coords / 4, kk_ring, jj_ring, 3, chunk=2048)
    corr = torch.stack([c0, c1], -1).view(1, st.E, -1)
    net, (delta, weight, _) = mod32(net, st.imap[:, kk_ring].float(), corr, None, st.ii, st.jj, st.kk)
    target = coords[..., 1, 1] + delta
    # the BA restatement runs on the host (fp64)
    lm = torch.tensor([1e-4], dtype=torch.float64)
    p, q = OB.fastba_forward(st.poses.cpu().double(), st.patches.cpu().double(), st.intrinsics.cpu().double(), target[0].cpu().double(),
                             weight[0].cpu().double(), lm, st.ii.cpu(), st.jj.cpu(), st.kk.cpu(), st.t0, st.n, iters)
    p, q = p.to(poses.device), q.to(poses.device)
    return dict(poses=p[:st.n], depth=q[:, 2, 1, 1], target=target, weight=weight, net=net, corr=corr, coords=coords)


@pytest.mark.parametrize("config,n_frames", [("fast", 30), ("default", 36)])
@pytest.mark.parametrize("graph", [False, True])
def test_full_update_step_vs_oracle_and_reference_pipeline(ext, ref_ext, config, n_frames, graph):
    st = synthetic.make_state(config, n_frames, device=DEV, seed=1234)
    run = UpdateRunner(st, seed=1234)
    torch.manual_seed(1234)
    mod32 = OU.Update(3).to(DEV).eval()
    mod32.load_state_dict(run.update.state_dict())
    live = st.kk.unique()
    poses0, patches0 = st.poses.clone(), st.patches.clone()

    ora = composed_oracle_step(st, mod32, torch.zeros(1, st.E, 384, device=DEV), run.kk_ring, run.jj_ring)

    def errs(x):
        return dict(pose=_rel(x["poses"], ora["poses"]), depth=_rel(x["depth"][live], ora["depth"][live]),
                    target=(x["target"] - ora["target"]).abs().max().item(), weight=(x["weight"] - ora["weight"]).abs().max().item(),
                    net=(x["net"] - ora["net"]).abs().max().item())

    def reference_pipeline(rx):
        from oracle.ref_pipeline import RefCudaStep
        refp = RefCudaStep(st, mod32)
        rt, rw, rcorr = refp.step()
        er = errs(dict(poses=refp.poses[:st.n], depth=refp.patches[:, 2, 1, 1], target=rt, weight=rw, net=refp.net.float()))
        r_corr = (rcorr.float() - ora["corr"]).abs().max().item() / ora["corr"].abs().max().item()
        return dict({"err_" + k: v for k, v in er.items()}, corr_rel_err=r_corr, poses=refp.poses[:st.n].clone(),
                    depth=refp.patches[live, 2, 1, 1].clone())

    # the reference CUDA pipeline's errors against the fp32 oracle set the bars of the whole update
    R = refdata.reference("step_%s%d" % (config, n_frames), ref_ext, reference_pipeline)

    if graph:
        run.capture()
        run.reset(); run.net.zero_()
        tgt, wgt = run.step_graph()
    else:
        tgt, wgt = run.step()
    torch.cuda.synchronize()
    ours = dict(poses=st.poses[:st.n].clone(), depth=st.patches[:, 2, 1, 1].clone(), target=tgt, weight=wgt, net=run.net)

    # correlation on the real ring (36 x 120 x 160 channels-last, reprojected coords): ours vs fp32 oracle
    e_corr = (run.corr_buf[..., :882].float() - ora["corr"]).abs().max().item() / ora["corr"].abs().max().item()
    r_corr = R["corr_rel_err"]

    eo, er = errs(ours), {k: R["err_" + k] for k in ("pose", "depth", "target", "weight", "net")}
    print("\n[%s graph=%s E=%d] corr rel err vs fp32 oracle: ours %.3g, reference kernel %.3g" % (config, graph, st.E, e_corr, r_corr))
    print("  ours      vs fp32 oracle:", {k: "%.3g" % v for k, v in eo.items()})
    print("  reference vs fp32 oracle:", {k: "%.3g" % v for k, v in er.items()})
    print("  ours vs reference CUDA pipeline: pose %.3g depth %.3g" % (_rel(ours["poses"], R["poses"].to(DEV)),
                                                                      _rel(R.pick("depth", ours["depth"][live]), R["depth"].to(DEV))))
    assert e_corr <= 2.0 ** -9 and e_corr <= r_corr
    for k in eo:
        assert eo[k] <= max(2 * er[k], {"pose": 1e-4, "depth": 1e-4, "target": 1e-2, "weight": 5e-3, "net": 2e-2}[k]), (k, eo[k], er[k])

    # BA stage alone on the path's own target / weight: our grouped BA vs the reference kernel vs the fp64 oracle at 1e-4
    lm = torch.tensor([1e-4], device=DEV)
    if ref_ext is not None:
        p_ref, q_ref = poses0.clone()[None], patches0.clone()[None]
        ref_ext[1].forward(p_ref, q_ref, st.intrinsics[None], tgt, wgt, lm, st.ii, st.jj, st.kk, st.cfg["M"], st.t0, st.n, 2, False)
        assert _rel(ours["poses"], p_ref[0, :st.n]) < 1e-4 and _rel(ours["depth"][live], q_ref[0, :, 2, 1, 1][live]) < 1e-4
    p_o, q_o = OB.fastba_forward(poses0.cpu().double(), patches0.cpu().double(), st.intrinsics.cpu().double(), tgt[0].cpu().double(),
                                 wgt[0].cpu().double(), lm.cpu().double(), st.ii.cpu(), st.jj.cpu(), st.kk.cpu(), st.t0, st.n, 2)
    p_o, q_o = p_o.to(DEV), q_o.to(DEV)
    assert _rel(ours["poses"], p_o[:st.n]) < 1e-4 and _rel(ours["depth"][live], q_o[:, 2, 1, 1][live]) < 1e-4


def test_recurrent_state_over_three_updates_tracks_the_oracle(ext):
    """three consecutive updates (the recurrent `net` carried in place, poses / depths updated by BA each time) on
    fast: drift against the fp32 composed oracle stays at the mixed-precision noise level"""
    st = synthetic.make_state("fast", 30, device=DEV, seed=11)
    run = UpdateRunner(st, seed=5)
    mod32 = OU.Update(3).to(DEV).eval()
    mod32.load_state_dict(run.update.state_dict())
    so = synthetic.make_state("fast", 30, device=DEV, seed=11)
    net = torch.zeros(1, st.E, 384, device=DEV)
    live = st.kk.unique()
    for it in range(3):
        o = composed_oracle_step(so, mod32, net, run.kk_ring, run.jj_ring)
        net = o["net"]
        so.poses[:so.n] = o["poses"].float()
        so.patches[:, 2] = o["depth"].float()[:, None, None]
        run.step()
        e_net = (run.net - net).abs().max().item()
        e_pose, e_depth = _rel(st.poses[:st.n], so.poses[:so.n]), _rel(st.patches[live, 2, 1, 1], so.patches[live, 2, 1, 1])
        print("update %d: net abs %.3g, pose rel %.3g, depth rel %.3g" % (it, e_net, e_pose, e_depth))
        assert e_net < 5e-2 and e_pose < 2e-3 and e_depth < 2e-2
