"""shared builders for the parity tests"""
import numpy as np
import torch

from detzero_b200.config import AttrDict

SMALL_RANGE = [-9.6, -9.6, -2, 9.6, 9.6, 4]
VOXEL = [0.1, 0.1, 0.15]
WAYMO_RANGE = [-75.2, -75.2, -2, 75.2, 75.2, 4]


def config1_cloud(n=20000, seed=0, pc_range=WAYMO_RANGE, c=5):
    """SURVEY.md §8d config 1: uniform cloud + 2 % out-of-range + 5 % exact duplicates / on-lattice coordinates"""
    g = np.random.default_rng(seed)
    lo, hi = np.array(pc_range[:3], np.float32), np.array(pc_range[3:], np.float32)
    p = g.uniform(lo, hi, (n, 3)).astype(np.float32)
    n_out = n // 50
    p[:n_out] = p[:n_out] * 1.2 + np.array([3.0, -3.0, 5.0], np.float32)          # outside (some in z only)
    n_dup = n // 20
    src = g.integers(n_out, n, n_dup)
    dst = g.integers(n_out, n, n_dup)
    p[dst[: n_dup // 2]] = p[src[: n_dup // 2]]                                     # exact duplicates
    k = g.integers(-700, 700, (n_dup - n_dup // 2, 3)).astype(np.float32)
    p[dst[n_dup // 2:]] = (k * np.array(VOXEL, np.float32)).astype(np.float32)      # exactly on the lattice
    p[g.integers(0, n, 8), 0] = hi[0]                                               # x == upper bound exactly
    feats = np.concatenate([np.tanh(g.uniform(0, 2, (n, 1))), g.uniform(0, 1, (n, max(c - 4, 1)))], axis=1)
    return np.concatenate([p, feats.astype(np.float32)], axis=1)[:, :c].astype(np.float32)


def clustered_cloud(n, seed, pc_range=SMALL_RANGE, c=5):
    """points concentrated on a few surfaces so that voxels have neighbours (exercises the rulebook)"""
    g = np.random.default_rng(seed)
    lo, hi = np.array(pc_range[:3], np.float32), np.array(pc_range[3:], np.float32)
    xy = g.uniform(lo[:2], hi[:2], (n, 2))
    z = np.where(g.random(n) < 0.6, g.normal(0.0, 0.05, n), g.uniform(0, 2.5, n))
    wall = g.random(n) < 0.3
    xy[wall, 0] = np.round(xy[wall, 0] / 3.0) * 3.0 + g.normal(0, 0.03, wall.sum())
    p = np.concatenate([xy, z[:, None]], axis=1)
    f = np.concatenate([np.tanh(g.uniform(0, 2, (n, 1))), g.uniform(0, 1, (n, c - 4))], axis=1)
    return np.concatenate([p, f], axis=1).astype(np.float32)


def merge_sweeps_inputs(seed=3):
    """three sweeps of 500 points (x y z intensity elongation NLZ-flag, 90 % NLZ == -1), small-angle poses, 0.1 s apart"""
    g = np.random.default_rng(seed)

    def pose():
        a = g.uniform(-0.2, 0.2)
        p = np.eye(4); p[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]; p[:3, 3] = g.uniform(-3, 3, 3)
        return p
    infos = [{'pose': pose(), 'time_stamp': 1550000000000000 - 100000 * k} for k in range(3)]
    pts = []
    for k in range(3):
        a = g.normal(0, 20, (500, 6)).astype(np.float32); a[:, 5] = np.where(g.random(500) < 0.9, -1, 1)
        pts.append(a)
    return infos, pts


def iou_boxes(seed=7, n=300):
    """rotated boxes (x y z dx dy dz heading); boxes 100..199 sit within ~0.2 m of boxes 0..99, so many pairs overlap partly"""
    g = np.random.default_rng(seed)
    b = np.concatenate([g.uniform(-10, 10, (n, 3)), g.uniform(1, 5, (n, 3)), g.uniform(-3.2, 3.2, (n, 1))], 1).astype(np.float32)
    b[100:200, :2] = b[:100, :2] + g.normal(0, 0.2, (100, 2)).astype(np.float32)
    return b


from detzero_b200.synthetic import model_cfg, CLASS_NAMES    # noqa: E402,F401  (one definition, shared with bench.py)


def rel_err(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()
