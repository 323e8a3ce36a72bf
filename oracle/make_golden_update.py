"""ORACLE tooling (test infrastructure): golden vectors of the update operator, produced by the
REFERENCE's own module -- dpvo/net.py:27-92 `Update` (with dpvo/blocks.py:15-48 GatedResidual /
SoftAgg) imported unmodified from /root/reference through oracle/refimport.py.

    python -m oracle.make_golden_update          # writes tests/golden/update_ref_{a,b}.pt

What the reference module cannot bring along in this container is replaced by stand-ins on sys.path
(oracle/shims): `torch_scatter` (pytorch-scatter 2.1.2, not vendored under /root/reference, restated
in oracle/update.py from its published definition -- and cross-checked below against a per-group
torch.softmax loop that shares no code with it) and `fastba.neighbors` (oracle/graph.py, itself
pinned bit-exactly to the reference's CUDA kernel by tests/golden/ba_ref_fast12.pt).  Everything
else -- layer structure, residual order, LayerNorm eps, the ii*12345+jj grouping key, the masks on
the neighbour inputs, the heads -- is the reference's code executing.

The fixtures hold inputs and outputs only; the weights are re-created by the consumer with
`torch.manual_seed(seed); Update(3)` (same construction order as net.py:28-72, checked through the
per-parameter checksums stored here).
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import refimport  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
CASES = {
    # name: (M patches/frame, lifetime, removal, frames, weight seed, data seed)
    "a": (6, 5, 8, 10, 1234, 71),
    "b": (4, 3, 5, 12, 99, 72),
}


def small_graph(M, lifetime, removal, frames):
    from dpvo_b200.synthetic import replay_edges
    return replay_edges(frames, M, lifetime, removal)


def loop_scatter_softmax_sum(fx, gx, key):
    """independent restatement of blocks.py:41-43 for the cross-check: python loop over groups"""
    uniq = torch.unique(key)
    out = torch.zeros(1, len(uniq), fx.shape[-1], dtype=fx.dtype)
    for n, u in enumerate(uniq.tolist()):
        sel = key == u
        w = torch.softmax(gx[0, sel], dim=0)
        out[0, n] = (fx[0, sel] * w).sum(0)
    return out


def group_rows(x, key):
    """[1, G, C]: the row of x shared by the edges of each group of `key`, groups in ascending key order;
    x == group_rows(x, key)[:, inverse] with inverse from torch.unique(key, return_inverse=True)"""
    _, inv = torch.unique(key, return_inverse=True)
    first = torch.zeros(int(inv.max()) + 1, dtype=torch.long).scatter_(0, inv.flip(0), torch.arange(key.numel() - 1, -1, -1))
    rows = x[:, first].clone()
    assert torch.equal(rows[:, inv], x), "rows differ inside a group"
    return rows


def make_inputs(E, dseed):
    """the seeded inputs of a case (CPU generator: identical on every host); the fixture stores their
    checksums instead of the tensors"""
    g = torch.Generator().manual_seed(dseed)
    net = torch.randn(1, E, 384, generator=g) * 0.5
    inp = torch.randn(1, E, 384, generator=g) * 0.25
    corr = torch.randn(1, E, 882, generator=g) * 2
    x = torch.randn(1, E, 384, generator=g)
    return net, inp, corr, x


def make_case(name):
    M, lifetime, removal, frames, wseed, dseed = CASES[name]
    ii, jj, kk = small_graph(M, lifetime, removal, frames)
    E = ii.numel()
    net, inp, corr, x = make_inputs(E, dseed)
    with refimport.reference_modules():
        import dpvo.net as RN
        torch.manual_seed(wseed)
        mod = RN.Update(3).eval()
        with torch.no_grad():
            out_net, (delta, weight, _) = mod(net, inp, corr, None, ii, jj, kk)
            # SoftAgg alone, against the loop restatement (pins the scatter stand-ins independently)
            agg = mod.agg_ij(x, ii * 12345 + jj)
            y = loop_scatter_softmax_sum(mod.agg_ij.f(x), mod.agg_ij.g(x), ii * 12345 + jj)
            _, inv = torch.unique(ii * 12345 + jj, return_inverse=True)
            agg_loop = mod.agg_ij.h(y)[:, inv]
            assert (agg - agg_loop).abs().max().item() < 1e-5, "scatter stand-in disagrees with the loop definition"
        sums = {k: float(v.double().sum()) for k, v in mod.state_dict().items()}
    # SoftAgg gives every edge of an (ii, jj) group the same row: store one row per group, in ascending key order
    agg_rows = group_rows(agg, ii * 12345 + jj)
    return dict(ii=ii, jj=jj, kk=kk, weight_seed=wseed, data_seed=dseed,
                input_sums=[float(t.double().sum()) for t in (net, inp, corr, x)],
                out_net=out_net, out_delta=delta, out_weight=weight, softagg_rows=agg_rows,
                param_sums=sums, source="dpvo/net.py:Update + dpvo/blocks.py (reference, imported unmodified), fp32 CPU, torch %s" % torch.__version__)


def main():
    if not refimport.available():
        raise SystemExit("reference tree not mounted; fixtures can only be regenerated in the build container")
    os.makedirs(GOLD, exist_ok=True)
    for name in CASES:
        d = make_case(name)
        path = os.path.join(GOLD, "update_ref_%s.pt" % name)
        torch.save(d, path)
        print("wrote %s: E=%d, %.1f KB" % (path, d["ii"].numel(), os.path.getsize(path) / 1e3))


if __name__ == "__main__":
    main()
