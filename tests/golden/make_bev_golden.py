"""Generate golden vectors for the BEV projection by running the REFERENCE's own
`MinkUNetBaseBEV.sparse2super` (utils/models/minkunet_bev.py:169-230) on CPU.

Needs a checkout of the reference at oracle/_ref/ (tests/refharness.py):
    python tests/golden/make_bev_golden.py
The reference imports MinkowskiEngine at module scope; an empty stand-in module
satisfies the import (sparse2super itself is plain torch).  torch is pinned to
one thread so index_put_ on duplicate pixels is the deterministic
"highest row wins" (SURVEY.md 8a-11).
"""
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

OUT = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(os.path.dirname(os.path.dirname(OUT)), "oracle", "_ref")


def _import_reference_model():
    me = types.ModuleType("MinkowskiEngine")
    mods = types.ModuleType("MinkowskiEngine.modules")
    rb = types.ModuleType("MinkowskiEngine.modules.resnet_block")
    rb.BasicBlock = type("BasicBlock", (), {"expansion": 1})
    rb.Bottleneck = type("Bottleneck", (), {"expansion": 4})
    me.modules = mods
    mods.resnet_block = rb
    sys.modules.update({"MinkowskiEngine": me, "MinkowskiEngine.modules": mods,
                        "MinkowskiEngine.modules.resnet_block": rb})
    sys.path.insert(0, REF)
    import utils.models.minkunet_bev as ref  # noqa
    return ref


def _bare_model(ref, bound, pool=(5, 3, 1)):
    m = object.__new__(ref.MinkUNetBaseBEV)
    nn.Module.__init__(m)
    m.mapping_bound_2d = bound
    m.mapping_boundaries = [[-bound, bound], [-bound, bound], [-10, 8]]
    m.pool2D = nn.MaxPool2d(*pool)
    return m


class _ST:  # the three attributes sparse2super touches (x.C, x.F, x.device)
    def __init__(self, C, F):
        self.C, self.F, self.device = C, F, F.device


def make_case(rng, n, batch, bound, channels, dup_frac=0.3, voxel=0.05):
    lim = int(bound / voxel) + 3  # a few rows fall outside the strict bounds
    xy = rng.integers(-lim, lim, size=(n, 2))
    z = rng.integers(-40, 40, size=(n, 1))
    ndup = int(n * dup_frac)
    if ndup:
        src = rng.integers(0, n, size=ndup)
        dst = rng.integers(0, n, size=ndup)
        xy[dst] = xy[src]  # several z-voxels per pixel
    b = np.sort(rng.integers(0, batch, size=(n, 1)), axis=0)
    b[0], b[-1] = 0, batch - 1
    coords = np.concatenate([b, xy, z], axis=1).astype(np.int32)
    # keep rows unique as a SparseTensor would
    _, first = np.unique(coords, axis=0, return_index=True)
    coords = coords[np.sort(first)]
    feats = rng.standard_normal((coords.shape[0], channels)).astype(np.float32)
    feats = np.maximum(feats, 0) + (rng.random(feats.shape) < 0.1) * feats  # mostly post-ReLU, some negatives
    return coords, feats.astype(np.float32)


def main():
    torch.set_num_threads(1)
    ref = _import_reference_model()
    rng = np.random.default_rng(20240617)
    cases = {}
    for name, (n, batch, bound, ch) in {
        "small": (600, 2, 2.0, 8),
        "wide": (1500, 3, 3.0, 5),
        "edge": (400, 1, 1.0, 3),
    }.items():
        coords, feats = make_case(rng, n, batch, bound, ch)
        m = _bare_model(ref, bound)
        F = torch.from_numpy(feats).clone().requires_grad_(True)
        out = m.sparse2super(_ST(torch.from_numpy(coords), F))
        gw = torch.from_numpy(rng.standard_normal(tuple(out.shape)).astype(np.float32))
        (out * gw).sum().backward()
        cases[name] = dict(coords=coords, feats=feats, bound=np.float64(bound), out=out.detach().numpy(),
                           grad_out=gw.numpy(), grad_feats=F.grad.numpy())
    # full-size image (bound 50 -> 2000x2000), few channels; store non-zeros only
    coords, feats = make_case(rng, 20000, 2, 50.0, 4, dup_frac=0.2)
    m = _bare_model(ref, 50.0)
    out = m.sparse2super(_ST(torch.from_numpy(coords), torch.from_numpy(feats))).numpy()
    nz = np.nonzero(out.reshape(-1))[0]
    cases["full50"] = dict(coords=coords, feats=feats, bound=np.float64(50.0), out_shape=np.array(out.shape),
                           nz_index=nz.astype(np.int64), nz_value=out.reshape(-1)[nz])
    flat = {f"{k}/{kk}": vv for k, v in cases.items() for kk, vv in v.items()}
    np.savez_compressed(os.path.join(OUT, "bev_reference.npz"), **flat)
    print({k: {kk: getattr(vv, "shape", vv) for kk, vv in v.items()} for k, v in cases.items()})


if __name__ == "__main__":
    main()
