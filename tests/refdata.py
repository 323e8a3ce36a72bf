"""Outputs of the reference project -- its own CUDA kernels (oracle/_ref) or its Python modules -- for the seeded
cases of the tests that compare against it.

Where the reference is at hand they are computed live.  Elsewhere they come from tests/golden/ref_<case>.pt, which the
same tests write when DPVO_GOLDEN_OUT names a directory and the reference is at hand (the GPU cases on a B200).
Small arrays are stored whole.  A large array is stored as a fixed sample of its elements, with the max-abs of the
whole array, the SHA-256 of its bytes (used by the tests that compare bit for bit) and the flat indices of the sample;
`Ref.pick` applies the same indices to the array under test, so one assertion reads the same either way."""
import hashlib
import math
import os

import pytest
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SAMPLE = 1024            # elements kept of an array larger than this


def _index(numel):
    """SAMPLE distinct flat indices spread over an array of `numel` elements: k * stride mod numel, the stride coprime
    to numel near numel / golden ratio.  Plain integer arithmetic, so the stored samples do not depend on the random
    number generator of any library version."""
    stride = max(1, int(numel * 0.6180339887498949))
    while math.gcd(stride, numel) != 1:
        stride += 1
    return torch.tensor(sorted(k * stride % numel for k in range(SAMPLE)), dtype=torch.long)


def _sha(x):
    return hashlib.sha256(x.detach().cpu().contiguous().numpy().tobytes()).hexdigest()


class Ref:
    def __init__(self, arrays, stored):
        self.arrays, self.stored = arrays, stored        # live: name -> full tensor / float; stored: the golden dict

    def __getitem__(self, k):
        """the reference array (its stored sample where it was sampled) or scalar"""
        if self.stored is None:
            return self.arrays[k]
        e = self.stored[k]
        return e["val"] if isinstance(e, dict) else e

    def pick(self, k, x):
        """the elements of `x` (shaped as reference array `k`) that `self[k]` holds"""
        if self.stored is None or not isinstance(self.stored[k], dict) or not self.stored[k]["sampled"]:
            return x
        e = self.stored[k]
        assert tuple(x.shape) == tuple(e["shape"]), (k, tuple(x.shape), e["shape"])
        return x.reshape(-1)[e["idx"].long().to(x.device)]

    def absmax(self, k):
        """max |.| over the whole reference array"""
        if self.stored is None or not isinstance(self.stored[k], dict):
            return self[k].abs().max().item()
        return self.stored[k]["absmax"]

    def equal(self, k, x):
        """`x` is bit for bit the reference array `k`"""
        if self.stored is None:
            return torch.equal(self.arrays[k].to(x.device), x)
        e = self.stored[k]
        return tuple(x.shape) == tuple(e["shape"]) and x.dtype == getattr(torch, e["dtype"]) and _sha(x) == e["sha256"]


def _store(arrays):
    out = {}
    for k, v in arrays.items():
        if not torch.is_tensor(v):
            out[k] = v
            continue
        v = v.detach().cpu().contiguous()
        e = {"shape": tuple(v.shape), "dtype": str(v.dtype).replace("torch.", ""), "sha256": _sha(v),
             "absmax": v.abs().max().item() if v.is_floating_point() else None}
        e["sampled"] = v.numel() > SAMPLE
        if e["sampled"]:
            e["idx"] = _index(v.numel()).int()
            e["val"] = v.reshape(-1)[e["idx"].long()].clone()
        else:
            e["val"] = v.clone()
        out[k] = e
    return out


def reference(case, ref_ext, compute):
    """the reference outputs of `case`: compute(ref_ext) -> {name: tensor or float} where oracle/_ref is built,
    else tests/golden/ref_<case>.pt"""
    if ref_ext is not None:
        arrays = compute(ref_ext)
        out_dir = os.environ.get("DPVO_GOLDEN_OUT")
        if out_dir:
            os.makedirs(out_dir, exist_ok=True)
            torch.save(_store(arrays), os.path.join(out_dir, "ref_%s.pt" % case))
        return Ref(arrays, None)
    path = os.path.join(GOLD, "ref_%s.pt" % case)
    if not os.path.exists(path):
        pytest.fail("no stored reference outputs for %s (%s) and oracle/_ref is not built" % (case, path))
    return Ref(None, torch.load(path))
