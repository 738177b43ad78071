"""Seeded inputs and digests shared by the golden-data generators and the tests that replay their fixtures."""
import hashlib

import numpy as np

# inputs reference_step_products.npz does not store (it would exceed 1 MB): seeded_inputs() regenerates them, the
# fixture keeps `<name>_sha256` of each to prove the regenerated arrays are the ones the reference saw
REGENERATED = ("bev_kitti_coords", "bev_nusc_coords", "aug_points")


def sha256(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def sample_index(n: int, k: int) -> np.ndarray:
    """A fixed, sorted sample of min(k, n) of the indices 0..n-1."""
    return np.sort(np.random.default_rng(0).choice(n, size=min(k, n), replace=False))


def seeded_inputs():
    """The seeded inputs of reference_step_products.npz: voxel coordinates and colabels of two synthetic scans (BEV
    label image), the bounds-filter cloud and the augmentation cloud."""
    from oracle import voxel as ov
    from lidog_b200.lidog import synth
    out = {}
    for tag, seed, shape in (("kitti", 5, "kitti"), ("nusc", 3, "nuscenes")):
        pts, lab = synth.make_scan(seed, shape)
        keep = (np.abs(pts[:, 0]) < 35) & (np.abs(pts[:, 1]) < 35)
        pts, lab = pts[keep][::3], lab[keep][::3]
        q, _, colab, _, _ = ov.sparse_quantize(pts, np.ones((len(pts), 1), np.float32), lab, -1, True, True, False, 0.05)
        out[f"bev_{tag}_coords"], out[f"bev_{tag}_colabels"] = q.astype(np.int32), colab.astype(np.int32)
    rng = np.random.default_rng(11)
    cloud = np.concatenate([rng.uniform(-70, 70, (4000, 2)), rng.uniform(-12, 10, (4000, 1))], 1).astype(np.float32)
    cloud[:200, :2] = rng.uniform(-3.5, 3.5, (200, 2)).astype(np.float32)  # around the ego box
    out["filter_points"] = cloud
    out["aug_points"] = rng.uniform(-40, 40, (3000, 3)).astype(np.float32)
    return out
