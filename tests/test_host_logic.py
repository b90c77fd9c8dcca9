"""Host-side logic that needs no GPU: module-attached caches (ADVICE r1 high), capacity-overflow reporting in
CenterPoint.post_processing (ADVICE r1 medium), explicit table layout (ADVICE r1 low)."""
import gc

import pytest
import torch
import torch.nn as nn


def test_fold_bn_cache_lives_on_the_module_and_tracks_changes():
    from detzero_b200.spconv import pytorch as sp
    assert not hasattr(sp, '_fold_cache'), 'no global id()-keyed cache: ids and allocator addresses are recycled'
    outs = []
    for seed in (1, 2, 3, 4):                       # models built and freed one after the other (the round-1 failure pattern)
        torch.manual_seed(seed)
        bn = nn.BatchNorm1d(16, eps=1e-3).eval()
        with torch.no_grad():
            bn.running_mean.normal_(); bn.running_var.uniform_(0.5, 1.5); bn.weight.uniform_(0.5, 1.5); bn.bias.normal_()
        scale, shift = sp.fold_bn(bn, None)
        want = bn.weight / torch.sqrt(bn.running_var + 1e-3)
        assert torch.allclose(scale, want) and torch.allclose(shift, bn.bias - bn.running_mean * want)
        assert '_dz_fold' in bn.__dict__
        s2, _ = sp.fold_bn(bn, None)
        assert s2 is scale                           # cache hit
        with torch.no_grad():
            bn.weight.mul_(2.0)                      # in-place update (what load_state_dict does) invalidates it
        s3, _ = sp.fold_bn(bn, None)
        assert torch.allclose(s3, 2 * want)
        outs.append(scale)
        del bn
        gc.collect()


def test_dense_and_refine_weight_caches_live_on_the_module():
    from detzero_b200.det import dense
    from detzero_b200.refine import modules as rm
    from detzero_b200 import _lib
    assert not hasattr(dense, '_pack_cache') and not hasattr(rm, '_w_cache')
    conv = nn.Conv2d(8, 4, 3)
    a = dense.pack_conv_weight(conv, _lib.DZ_F32)
    assert dense.pack_conv_weight(conv, _lib.DZ_F32) is a and '_dz_pack' in conv.__dict__
    conv2 = nn.Conv2d(8, 4, 3)
    assert not torch.equal(dense.pack_conv_weight(conv2, _lib.DZ_F32), a)
    lin = nn.Linear(8, 4)
    w = rm._w2d(lin)
    assert rm._w2d(lin) is w and torch.equal(w, lin.weight.detach())
    with torch.no_grad():
        lin.weight.add_(1.0)
    assert torch.equal(rm._w2d(lin), lin.weight.detach())


class _FakeLevel:
    def __init__(self, count, cap, producer):
        self._count = torch.tensor([count], dtype=torch.int32)
        self._cap, self._n, self._producer = cap, None, producer

    def set_num(self, n):
        from detzero_b200.spconv.pytorch import SparseConvTensor
        return SparseConvTensor.set_num(self, n)


class _Producer:
    _cap_hint = 0


def test_post_processing_raises_every_hint_before_reporting_overflow():
    from detzero_b200.det.centerpoint import CenterPoint
    pa, pb, pc = _Producer(), _Producer(), _Producer()
    levels = {'x_conv1': _FakeLevel(50, 100, pa), 'x_conv2': _FakeLevel(300, 200, pb), 'x_conv3': _FakeLevel(700, 400, pc)}
    bd = {'final_boxes_count': torch.tensor([2], dtype=torch.int32), 'final_boxes_padded': torch.zeros(1, 500, 9),
          'multi_scale_3d_features': levels, 'overflow_flag': torch.tensor([2], dtype=torch.int32)}
    with pytest.raises(RuntimeError, match='overflow in 2 place'):
        CenterPoint.post_processing(None, bd)
    assert (pa._cap_hint, pb._cap_hint, pc._cap_hint) == (50, 300, 700)     # ALL hints grew, not only the first overflowing one
    # the device flag alone (counts were clamped by a replayed graph) is enough to raise
    ok = {'x_conv1': _FakeLevel(50, 100, pa)}
    bd = {'final_boxes_count': torch.tensor([0], dtype=torch.int32), 'final_boxes_padded': torch.zeros(1, 500, 9),
          'multi_scale_3d_features': ok, 'overflow_flag': torch.tensor([1], dtype=torch.int32)}
    with pytest.raises(RuntimeError, match='overflow'):
        CenterPoint.post_processing(None, bd)
    bd['overflow_flag'] = torch.tensor([0], dtype=torch.int32)
    pred, _ = CenterPoint.post_processing(None, bd)
    assert len(pred) == 1 and pred[0]['pred_boxes'].shape[0] == 0
    # counts are re-read on every call (a replayed graph reuses the same output objects)
    ok['x_conv1']._count = torch.tensor([70], dtype=torch.int32)
    CenterPoint.post_processing(None, bd)
    assert ok['x_conv1']._n == 70


def test_overflow_flag_counts_clamped_levels():
    from detzero_b200.det.centerpoint import CenterPoint
    levels = {'a': _FakeLevel(50, 100, None), 'b': _FakeLevel(300, 200, None)}
    bd = {'final_boxes_count': torch.zeros(1, dtype=torch.int32), 'multi_scale_3d_features': levels}
    assert int(CenterPoint._overflow_flag(None, bd).item()) == 1
    bd['voxel_wanted'] = (torch.tensor([10], dtype=torch.int32), 5, None)
    assert int(CenterPoint._overflow_flag(None, bd).item()) == 2


def test_first_run_capacity_growth_is_per_dimension():
    from detzero_b200.spconv import pytorch as sp
    conv_out = sp.SparseConv3d(64, 128, (3, 1, 1), stride=(2, 1, 1), padding=0, bias=False)
    worst = 1
    for k, s in zip(conv_out.kernel_size, conv_out.stride):
        worst *= -(-k // s)
    assert worst == 2                                 # one z = 2 input reaches two outputs: a 1.0 factor could overflow


def test_tracker_and_crop_oracle_restatements():
    """oracle pieces behind tests/test_gpu_track.py: overlap area is the numerator of the (reference-pinned) rotated IoU; 3-D IoU of
    a box with itself is 1; the crop mask equals an independent float64 point-in-rotated-box test away from the faces"""
    import numpy as np
    import oracle
    g = np.random.default_rng(1)
    b = np.concatenate([g.uniform(-5, 5, (40, 3)), g.uniform(1, 4, (40, 3)), g.uniform(-3.2, 3.2, (40, 1))], 1).astype(np.float32)
    ov, iou = oracle.boxes_overlap_bev(b, b), oracle.boxes_iou_bev(b, b)
    area = (b[:, 3] * b[:, 4])
    assert np.allclose(iou, ov / np.maximum(area[:, None] + area[None] - ov, 1e-8), atol=1e-6)
    assert np.allclose(np.diag(oracle.boxes_iou3d(b, b)), 1.0, atol=3e-2)          # the 1e-2 corner margin again
    assert np.allclose(oracle.iou2d(b[:, [0, 1, 3, 4]], b[:, [0, 1, 3, 4]]).diagonal(), 1.0)
    p = g.uniform(-8, 8, (20000, 3)).astype(np.float32)
    m = oracle.points_in_boxes(p, b)
    P, B = p.astype(np.float64), b.astype(np.float64)
    for t in range(0, 40, 7):
        c, s = np.cos(-B[t, 6]), np.sin(-B[t, 6])
        lx = (P[:, 0] - B[t, 0]) * c - (P[:, 1] - B[t, 1]) * s
        ly = (P[:, 0] - B[t, 0]) * s + (P[:, 1] - B[t, 1]) * c
        inside = (np.abs(P[:, 2] - B[t, 2]) <= B[t, 5] / 2) & (np.abs(lx) < B[t, 3] / 2) & (np.abs(ly) < B[t, 4] / 2)
        near = (np.abs(np.abs(lx) - B[t, 3] / 2) < 1e-3) | (np.abs(np.abs(ly) - B[t, 4] / 2) < 1e-3) | (np.abs(np.abs(P[:, 2] - B[t, 2]) - B[t, 5] / 2) < 1e-3)
        assert np.array_equal(m[t][~near] == 1, inside[~near])


def test_frame_file_format_and_result_pkl(tmp_path):
    """reference on-disk formats: (N, 6) float32 frame files read straight into a (pinned-able) buffer; result.pkl round trip"""
    import numpy as np
    from detzero_b200 import io as dzio
    g = np.random.default_rng(0)
    pts = g.normal(0, 10, (1234, 6)).astype(np.float32)
    path = str(tmp_path / '0007.npy')
    dzio.write_frame_npy(path, pts)
    assert np.array_equal(np.load(path), pts)                       # byte-compatible with what the reference reads (waymo_dataset.py:97)
    buf = torch.empty((2000, 6), dtype=torch.float32)
    assert dzio.read_frame_into(path, buf) == 1234 and np.array_equal(buf[:1234].numpy(), pts)
    with pytest.raises(ValueError):
        dzio.read_frame_into(path, torch.empty((10, 6), dtype=torch.float32))
    np.save(str(tmp_path / 'bad.npy'), pts.astype(np.float64))
    with pytest.raises(ValueError):
        dzio.read_frame_into(str(tmp_path / 'bad.npy'), buf)
    boxes = torch.zeros(2, 500, 9)
    boxes[0, :3, 7], boxes[0, :3, 8], boxes[1, :1, 8] = torch.tensor([.9, .8, .7]), torch.tensor([1., 3., 2.]), 1.
    annos = dzio.gathered_to_annos(boxes, torch.tensor([3, 1]), ['Vehicle', 'Pedestrian', 'Cyclist'], sequence_name='seg-1')
    dzio.save_result_pkl(str(tmp_path / 'result.pkl'), annos)
    back = dzio.sequence_list_to_dict(dzio.load_result_pkl(str(tmp_path / 'result.pkl')))
    assert list(back['seg-1']['0000']['name']) == ['Vehicle', 'Cyclist', 'Pedestrian'] and back['seg-1']['0001']['boxes_lidar'].shape == (1, 7)


def test_merge_sweeps_restatement_matches_reference_source():
    """the oracle's merge_sweeps against the output of the reference's own DatasetTemplate.merge_sweeps statements
    (detection/detzero_det/datasets/dataset.py) on the same inputs, stored by tests/golden/make_golden_host.py"""
    import os
    import numpy as np
    from oracle import det_ref
    from tests import util
    want = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'host.npz'))['merge_sweeps']
    infos, pts = util.merge_sweeps_inputs()
    got = det_ref.merge_sweeps(infos[0], infos, pts)
    assert np.array_equal(want, got)
