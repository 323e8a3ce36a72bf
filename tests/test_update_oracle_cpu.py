"""oracle/update.py held to the REFERENCE's own dpvo/net.py:Update -- through the committed fixtures
(tests/golden/update_ref_*.pt, written by oracle/make_golden_update.py from the imported reference
module) and against the imported module itself (live where the reference sources are at hand, else its stored
outputs)."""
import os

import pytest
import torch

import refdata
from oracle import update as OU, refimport
from oracle.make_golden_update import CASES, make_inputs, small_graph, loop_scatter_softmax_sum

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("name", sorted(CASES))
def test_update_oracle_reproduces_reference_module_fixture(name):
    d = torch.load(os.path.join(GOLD, "update_ref_%s.pt" % name))
    M, lifetime, removal, frames, wseed, dseed = CASES[name]
    ii, jj, kk = small_graph(M, lifetime, removal, frames)
    assert torch.equal(ii, d["ii"]) and torch.equal(jj, d["jj"]) and torch.equal(kk, d["kk"])
    net, inp, corr, x = make_inputs(ii.numel(), dseed)
    for t, s in zip((net, inp, corr, x), d["input_sums"]):
        assert abs(float(t.double().sum()) - s) < 1e-6 * max(1.0, abs(s))
    torch.manual_seed(d["weight_seed"])
    mod = OU.Update(3).eval()
    for k, v in mod.state_dict().items():       # same construction order => same seeded weights as the reference module
        assert abs(float(v.double().sum()) - d["param_sums"][k]) < 1e-9 * max(1.0, abs(d["param_sums"][k])), k
    with torch.no_grad():
        on, (od, ow, _) = mod(net, inp, corr, None, ii, jj, kk)
        agg = mod.agg_ij(x, ii * 12345 + jj)
    # fp32 on both sides, same op order: equal up to the BLAS summation order of the host that wrote the fixture
    assert (on - d["out_net"]).abs().max().item() <= 2e-5 * d["out_net"].abs().max().item()
    assert (od - d["out_delta"]).abs().max().item() <= 1e-5
    assert (ow - d["out_weight"]).abs().max().item() <= 1e-5
    _, inv = torch.unique(ii * 12345 + jj, return_inverse=True)
    assert (agg - d["softagg_rows"][:, inv]).abs().max().item() <= 1e-5


def test_scatter_restatement_against_loop_definition():
    g = torch.Generator().manual_seed(5)
    E = 300
    key = torch.randint(0, 17, (E,), generator=g) * 12345 + torch.randint(0, 3, (E,), generator=g)
    fx, gx = torch.randn(1, E, 32, generator=g).double(), 3 * torch.randn(1, E, 32, generator=g).double()
    _, inv = torch.unique(key, return_inverse=True)
    y = OU.scatter_sum(fx * OU.scatter_softmax(gx, inv, dim=1), inv, dim=1)
    assert (y - loop_scatter_softmax_sum(fx, gx, key)).abs().max().item() < 1e-12


def test_update_oracle_equals_imported_reference_module_live():
    """the reference module run live where its sources are at hand (bit for bit: same host, same op order), else its
    stored outputs (tests/golden/ref_update_live.pt) to the fixture test's bars above"""
    ii, jj, kk = small_graph(5, 4, 6, 9)
    net, inp, corr, _ = make_inputs(ii.numel(), 123)
    torch.manual_seed(7)
    mine = OU.Update(3).eval()

    def compute(_):
        with refimport.reference_modules():
            import dpvo.net as RN
            theirs = RN.Update(3).eval()
            theirs.load_state_dict(mine.state_dict())          # identical key names
            with torch.no_grad():
                rn, (rd, rw, _) = theirs(net, inp, corr, None, ii, jj, kk)
        return dict(net=rn, delta=rd, weight=rw)

    R = refdata.reference("update_live", refimport if refimport.available() else None, compute)
    with torch.no_grad():
        on, (od, ow, _) = mine(net, inp, corr, None, ii, jj, kk)
    if R.stored is None:
        assert torch.equal(on, R["net"]) and torch.equal(od, R["delta"]) and torch.equal(ow, R["weight"])
    else:
        assert (R.pick("net", on) - R["net"]).abs().max().item() <= 2e-5 * R.absmax("net")
        assert (R.pick("delta", od) - R["delta"]).abs().max().item() <= 1e-5
        assert (R.pick("weight", ow) - R["weight"]).abs().max().item() <= 1e-5


def test_packed_inference_weights_follow_the_parameters():
    """dpvo_b200.net.Update keeps fp16 copies of its dense weights for the kernels; loading a checkpoint (or any
    in-place parameter change) after a forward must refresh them (ADVICE r01)"""
    from dpvo_b200.net import Update
    torch.manual_seed(0)
    u = Update(3).eval()
    p1 = u.packed()
    w_before = p1["c1a"][0].clone()
    assert u.packed() is p1                                   # unchanged parameters: no repacking
    torch.manual_seed(1)
    other = OU.Update(3).state_dict()
    u.load_state_dict(other)
    p2 = u.packed()
    assert not torch.equal(p2["c1a"][0], w_before)
    assert torch.equal(p2["c1a"][0], other["c1.0.weight"].half())
    with torch.no_grad():
        u.c1[0].weight.mul_(2.0)                              # an optimiser-style in-place step
    assert torch.equal(u.packed()["c1a"][0], (other["c1.0.weight"] * 2).half())
