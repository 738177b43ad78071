"""Golden vectors for the losses, the BEV label image and the dataset-side filters, produced by the REFERENCE's own
code (needs a checkout of the reference at oracle/_ref/, tests/refharness.py):

    python tests/golden/make_reference_golden.py        -> tests/golden/reference_step_products.npz

  * utils/losses/losses.py:56-97,129-187       DICELoss, SoftDICELoss (7 classes, and the 19-class `is_kitti` branch):
                                                loss value and d loss / d logits
  * utils/datasets/semantickitti_bev.py:433-464 PC2ImgConverter.getBEVImageNew, arguments prepared as at :137-153,:244-249
  * utils/datasets/semantickitti_bev.py:155-172 filter_bounds;  utils/datasets/dataset.py:58-72 random_sample (seeded)
The reference is not part of this repository: tests/test_golden_reference.py replays these inputs through
lidog_b200/lidog/{losses,step,datapath}.py on the CPU (everywhere) and on the device (-m gpu)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import refharness as rh  # noqa: E402
from tests.golden.inputs import REGENERATED, seeded_inputs, sha256  # noqa: E402
from tests.test_reference_unchanged import _reference_class  # noqa: E402


def main():
    from oracle import me_cpu
    inputs = seeded_inputs()
    out = {}
    with rh.reference(me_cpu):
        ref = rh.load_file("utils/losses/losses.py", "losses")
        g = torch.Generator().manual_seed(7)
        for C, kitti in ((7, False), (19, True)):
            logits = (torch.randn(3000, C, generator=g) * 2).float()
            target = torch.randint(-1, C, (3000,), generator=g)
            target[:40], target[40:70] = 1, min(6, C - 1)
            target[target == 3] = 4  # a class that never occurs (tmask)
            out[f"loss{C}_logits"], out[f"loss{C}_target"] = logits.numpy(), target.numpy()
            for name, crit in (("dice", ref.DICELoss(ignore_label=-1)),
                               ("softdice", ref.SoftDICELoss(ignore_label=-1, is_kitti=kitti))):
                x = logits.clone().requires_grad_(True)
                v = crit(x, target)
                v.backward()
                out[f"loss{C}_{name}"], out[f"loss{C}_{name}_grad"] = np.float64(v.item()), x.grad.numpy()
    Conv = _reference_class("utils/datasets/semantickitti_bev.py", "PC2ImgConverter")
    for tag, bound, img in (("kitti", 50.0, 167), ("nusc", 30.0, 100)):
        q, colab = inputs[f"bev_{tag}_coords"], inputs[f"bev_{tag}_colabels"]
        bounds = [[-bound, bound], [-bound, bound], [-10, 8]]
        conv = Conv(imgChannel=1, xRange=bounds[0], yRange=bounds[1], zRange=bounds[2], xGridSize=2 * bound / img,
                    yGridSize=2 * bound / img, zGridSize=0.3)
        bl, _ = conv.getBEVImageNew((q * 0.05).astype(np.float32), colab)
        out[f"bev_{tag}_coords"], out[f"bev_{tag}_colabels"] = q, colab
        out[f"bev_{tag}_image"], out[f"bev_{tag}_bound_img"] = bl.astype(np.int32), np.array([bound, img])
    # dataset-side filter + augmentation: plain numpy on `self.*` attributes / module-level scipy
    import ast
    src = open(rh.REF + "/utils/datasets/semantickitti_bev.py").read()
    fb = next(n for n in ast.walk(ast.parse(src)) if isinstance(n, ast.FunctionDef) and n.name == "filter_bounds")
    ns = {"np": np}
    exec(compile(ast.Module(body=[fb], type_ignores=[]), "semantickitti_bev.py", "exec"), ns)

    class Self:
        grid_bounds = [[-60, 60], [-60, 60], [-10, 8]]  # semantickitti_bev.py:137
    cloud = inputs["filter_points"]
    out["filter_points"], out["filter_keep"] = cloud, np.asarray(ns["filter_bounds"](Self(), cloud))
    from scipy.linalg import expm, norm
    asrc = open(rh.REF + "/utils/common/augmentation.py").read()
    ans = {"np": np, "expm": expm, "norm": norm}
    for node in ast.parse(asrc).body:
        if isinstance(node, ast.ClassDef) and node.name in ("RandomRotation", "RandomScale"):
            exec(compile(ast.Module(body=[node], type_ignores=[]), "augmentation.py", "exec"), ans)
    np.random.seed(1234)  # configs/lidog/single/semantickitti.yaml:32
    pts32 = inputs["aug_points"]
    aug = ans["RandomScale"](0.95, 1.05)(ans["RandomRotation"]()(pts32.copy()))  # order of train_lidog's Compose
    out["aug_points"], out["aug_result"] = pts32, np.asarray(aug)
    assert out["aug_result"].dtype == np.float64  # float32 @ float64: what sparse_quantize then receives
    out = {(k + "_sha256" if k in REGENERATED else k): (np.array(sha256(v)) if k in REGENERATED else v)
           for k, v in out.items()}
    np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_step_products.npz"), **out)
    print({k: getattr(v, "shape", v) for k, v in out.items()})


if __name__ == "__main__":
    main()
