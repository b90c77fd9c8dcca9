"""Direct rulebook path of the bf16-plane layers (mask pass -> scatter -> tile pass, no row-major table) against the table
path: the same masks, digests and histogram, a tile-major table that equals the row-major table row for row, and
bit-identical backbone features.  Run on the B200 box: pytest -m gpu."""
import numpy as np
import pytest
import torch

import oracle
from oracle import det_ref, weights
from tests import util
from detzero_b200 import ops

pytestmark = pytest.mark.gpu

SCHED_BINS = 4096


def _coords(seed, B, shape, density):
    """random sites plus full x = 0 and x = W-1 columns in some (z, y) rows of every frame: the x-clipping of the mask pass and
    lines that end on a bitmap word boundary (W not a multiple of 32) are exercised"""
    idx = weights.random_sparse_coords(seed, B, shape, density)
    D, H, W = shape
    g = np.random.default_rng(seed + 7)
    edge = []
    for b in range(B):
        for z, y in zip(g.integers(0, D, 6), g.integers(0, H, 6)):
            edge += [(b, z, y, 0), (b, z, y, 1), (b, z, y, W - 2), (b, z, y, W - 1)]
    idx = np.unique(np.concatenate([idx, np.array(edge, np.int32)]), axis=0).astype(np.int32)
    return idx[g.permutation(len(idx))]


def _ws_parts(sws, cap):
    """hist | tile_mask | tickets | masks | keys views of a schedule workspace (csrc/rulebook.cu)"""
    tiles = (cap + 127) // 128
    i32 = sws.view(torch.int32)
    off = SCHED_BINS + tiles + 8
    masks = i32[off:off + cap]
    keys = sws[(off + cap) * 4:(off + cap) * 4 + cap * 2].view(torch.int16)
    return i32[:SCHED_BINS], masks, keys


def _check_tiles(order, tab_tiles, cap, n, K, tab, masks):
    """tab_tiles rows (via plane K) == the row-major table; order a permutation; tile masks = OR of their rows' masks"""
    tiles = (cap + 127) // 128
    tn = (n + 127) // 128
    o = order[:n].cpu().numpy()
    assert np.array_equal(np.sort(o), np.arange(n))
    assert np.array_equal(np.sort(order[cap:cap + tiles].cpu().numpy()), np.arange(tiles))
    tt = tab_tiles[:tn].cpu().numpy()
    rows = tt[:, K, :].reshape(-1)
    assert np.array_equal(rows[:n], o) and np.all(rows[n:] == -1)
    planes = tt[:, :K, :].transpose(1, 0, 2).reshape(K, -1)
    want = tab[:n, :K].cpu().numpy().T                                      # canonical row order
    assert np.array_equal(planes[:, :n], want[:, o])
    assert np.all(planes[:, n:] == -1)
    m = masks[:n].cpu().numpy().astype(np.int64)
    assert np.array_equal(m, tab[:n, 27].cpu().numpy().astype(np.int64))
    tm = np.zeros(tn, np.int64)
    np.bitwise_or.at(tm, np.arange(n) // 128, m[o])
    assert np.array_equal(order[cap + tiles:cap + tiles + tn].cpu().numpy().astype(np.int64), tm)


@pytest.mark.parametrize('ks,with_perm,perm_walk', [((3, 3, 3), True, True), ((3, 3, 3), True, False), ((3, 3, 3), False, False),
                                                    ((1, 3, 3), True, True), ((3, 1, 1), True, True)])
@pytest.mark.parametrize('frame_major', [False, True])
def test_direct_subm_equals_table_path(cuda, ks, with_perm, perm_walk, frame_major):
    shape, B = [7, 20, 67], 3
    idx = _coords(5, B, shape, 0.25)
    if not with_perm:                               # an index without perm: the rows must be in lattice order
        idx = idx[np.lexsort(idx.T[::-1])]
    n = cap = len(idx)
    K = ks[0] * ks[1] * ks[2]
    c = torch.from_numpy(idx).to(cuda)
    d_n = torch.tensor([n], dtype=torch.int32, device=cuda)
    index = ops.grid_index_from_coords(c, d_n, cap, B, shape, with_perm=with_perm)
    sws_a, sws_b = ops.new_sched_ws(cap, cuda), ops.new_sched_ws(cap, cuda)
    tab = ops.rulebook_subm(c, d_n, cap, index, list(ks), layout='row', sched_ws=sws_a, frame_major=frame_major)
    ops.rulebook_subm_masks(c, d_n, cap, index, list(ks), sws_b, frame_major=frame_major, perm_walk=perm_walk)
    ha, ma, ka = _ws_parts(sws_a, cap)
    hb, mb, kb = _ws_parts(sws_b, cap)
    assert torch.equal(ha, hb) and torch.equal(ma[:n], mb[:n]) and torch.equal(ka[:n], kb[:n])
    order, tab_tiles = ops.rulebook_schedule_direct(c, d_n, cap, index, list(ks), [1, 1, 1], [0, 0, 0], True, sws_b, B, frame_major)
    _check_tiles(order, tab_tiles, cap, n, K, tab, mb)
    assert torch.equal(ops.tiles_to_rows(tab_tiles, order, d_n, cap)[:n], tab[:n])


@pytest.mark.parametrize('ks,stride,pad', [((3, 3, 3), (2, 2, 2), (1, 1, 1)), ((3, 1, 1), (2, 1, 1), (0, 0, 0)),
                                           ((3, 3, 3), (2, 2, 2), (0, 1, 1))])
@pytest.mark.parametrize('frame_major', [False, True])
def test_direct_conv_equals_table_path(cuda, ks, stride, pad, frame_major):
    shape, B = [9, 22, 66], 3
    idx = _coords(11, B, shape, 0.2)
    n_in = len(idx)
    c = torch.from_numpy(idx).to(cuda)
    d_n = torch.tensor([n_in], dtype=torch.int32, device=cuda)
    index = ops.grid_index_from_coords(c, d_n, n_in, B, shape, with_perm=True)
    out_cap = 2 * n_in
    K = ks[0] * ks[1] * ks[2]
    sws_a, sws_b = ops.new_sched_ws(out_cap, cuda), ops.new_sched_ws(out_cap, cuda)
    oc_a, dn_a, _, tab, odhw_a = ops.rulebook_conv(c, d_n, n_in, index, list(ks), list(stride), list(pad), out_cap, layout='row',
                                                   sched_ws=sws_a, frame_major=frame_major)
    oc_b, dn_b, oi_b, odhw_b = ops.rulebook_conv_masks(c, d_n, n_in, index, list(ks), list(stride), list(pad), out_cap, sws_b,
                                                       frame_major=frame_major)
    n = int(dn_a.item())
    assert n == int(dn_b.item()) and odhw_a == odhw_b and torch.equal(oc_a[:n], oc_b[:n])
    ha, ma, ka = _ws_parts(sws_a, out_cap)
    hb, mb, kb = _ws_parts(sws_b, out_cap)
    assert torch.equal(ha, hb) and torch.equal(ma[:n], mb[:n]) and torch.equal(ka[:n], kb[:n])
    order, tab_tiles = ops.rulebook_schedule_direct(oc_b, dn_b, out_cap, index, list(ks), list(stride), list(pad), False, sws_b, B,
                                                    frame_major)
    _check_tiles(order, tab_tiles, out_cap, n, K, tab, mb)


def _waymo_batch(cuda, B):
    clouds = [util.clustered_cloud(40000, 300 + b, util.WAYMO_RANGE) for b in range(B)]
    ref = oracle.Point2VoxelCPU3d(util.VOXEL, util.WAYMO_RANGE, 5, 5, 150000)
    feats, coords = [], []
    for b, p in enumerate(clouds):
        v, c, n = ref.point_to_voxel(p)
        feats.append(det_ref.mean_vfe(v, n)); coords.append(np.pad(c, ((0, 0), (1, 0)), constant_values=b))
    return torch.cat(feats).to(cuda), torch.from_numpy(np.concatenate(coords).astype(np.int32)).to(cuda)


@pytest.mark.parametrize('kind', ['VoxelBackBone8x', 'VoxelResBackBone8x'])
def test_backbone_direct_tiles_bit_identical(cuda, kind):
    """batch 8 on the 1504 x 1504 x 41 lattice: the direct path and the table path give the same features, bit for bit"""
    from detzero_b200.det import cp_modules
    from detzero_b200.spconv.pytorch import _SparseConv
    B = 8
    feats, coords = _waymo_batch(cuda, B)
    for mode in ('bf16x2', 'bf16'):
        cfg = util.model_cfg(kind).BACKBONE_3D
        cfg.COMPUTE_MODE = mode
        m = cp_modules[kind](model_cfg=cfg, input_channels=5, grid_size=[1504, 1504, 40]).eval()
        weights.load_seeded(m, 7)
        m = m.to(cuda)
        def run():
            # the first frame sizes the strided convs' outputs from a guess; an overflow raises the capacity hint and asks for a re-run
            for attempt in range(6):
                try:
                    with torch.no_grad():
                        bd = m({'voxel_features': feats, 'voxel_coords': coords, 'batch_size': B})
                    return [(name, t.indices.cpu(), t.features.cpu()) for name, t in
                            list(bd['multi_scale_3d_features'].items()) + [('out', bd['encoded_spconv_tensor'])]]
                except RuntimeError as e:
                    if 'overflow' not in str(e):
                        raise
            raise AssertionError('capacity hints did not settle')

        outs = []
        try:
            for direct in (True, False):
                _SparseConv.DIRECT_TILES = direct
                outs.append(run())
        finally:
            _SparseConv.DIRECT_TILES = True
        for (name, ia, fa), (_, ib, fb) in zip(*outs):
            assert torch.equal(ia, ib), (mode, name)
            assert torch.equal(fa.view(torch.int32), fb.view(torch.int32)), (mode, name)
