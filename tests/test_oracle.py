"""CPU tests (-m "not gpu"): pin the oracle against the golden vectors produced by the reference's own modules
(tests/golden/make_golden.py), cross-check the two voxelizer restatements and the sparse-conv restatement against
torch's dense conv3d, and check the host logic + that the C-ABI library exports every declared symbol."""
import json
import os
import re

import numpy as np
import pytest
import torch

import oracle
from oracle import det_ref, spconv_ref, weights
from tests import util

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, 'golden', 'detector.npz'))
TINY_RANGE = [-4.8, -4.8, -2, 4.8, 4.8, 4]
SEED = 1234


def tiny_batch():
    clouds = [util.clustered_cloud(6000, 101, TINY_RANGE), util.clustered_cloud(3500, 102, TINY_RANGE)]
    vox = oracle.Point2VoxelCPU3d(util.VOXEL, TINY_RANGE, 5, 5, 200000)
    v, c, n = [], [], []
    for b, p in enumerate(clouds):
        vv, cc, nn = vox.point_to_voxel(p)
        v.append(vv); n.append(nn); c.append(np.pad(cc, ((0, 0), (1, 0)), constant_values=b))
    return np.concatenate(v), np.concatenate(c).astype(np.int32), np.concatenate(n)


def test_voxelizer_c_vs_python_restatement():
    """BASELINE config[0] shape (reduced n): the C and pure-Python restatements of Point2VoxelCPU3d agree bit for bit,
    incl. out-of-range points, duplicates, on-lattice coordinates and the voxel cap"""
    pts = util.config1_cloud(3000, seed=0)
    for max_voxels in (200000, 700):
        v, c, n = oracle.Point2VoxelCPU3d(util.VOXEL, util.WAYMO_RANGE, 5, 5, max_voxels).point_to_voxel(pts)
        pv, pc, pn = oracle.points_to_voxel_py(pts, util.VOXEL, util.WAYMO_RANGE, 5, max_voxels)
        assert np.array_equal(c, pc) and np.array_equal(n, pn) and np.array_equal(v.view(np.uint32), pv.view(np.uint32))
        assert len(c) <= max_voxels
    assert (n <= 5).all() and len(np.unique(c, axis=0)) == len(c)


def test_voxelizer_properties_full_size():
    """size-independent properties at the BASELINE size (180 K points): voxels unique, counts consistent, every kept
    point lies inside its voxel, first-appearance order"""
    from detzero_b200.det.dataset import synth_waymo_cloud
    pts = synth_waymo_cloud(0)[:, :5]
    v, c, n = oracle.Point2VoxelCPU3d(util.VOXEL, util.WAYMO_RANGE, 5, 5, 200000).point_to_voxel(pts)
    assert len(np.unique(c, axis=0)) == len(c)
    lo = np.array(util.WAYMO_RANGE[:3], np.float32)
    first = v[:, 0, :3]
    cc = np.floor((first - lo) / np.array(util.VOXEL, np.float32)).astype(np.int32)[:, ::-1]
    assert np.array_equal(cc, c)
    assert n.sum() <= len(pts) and n.min() >= 1


def test_sparse_conv_restatement_vs_dense_conv3d():
    shape, B, cin, cout = [9, 20, 20], 2, 4, 6
    idx = weights.random_sparse_coords(3, B, shape, 0.1)
    f = torch.randn(len(idx), cin, dtype=torch.float64)
    x = spconv_ref.dense_from_sparse(f, idx, shape, B)
    for ks, st, pd in [(3, 1, 1), (3, 2, 1), (3, 2, (0, 1, 1)), ((3, 1, 1), (2, 1, 1), 0)]:
        w = torch.randn(cout, *spconv_ref._triple(ks), cin, dtype=torch.float64)
        d = torch.nn.functional.conv3d(x, w.permute(0, 4, 1, 2, 3), stride=spconv_ref._triple(st), padding=spconv_ref._triple(pd))
        if st == 1:
            o = spconv_ref.sparse_conv_native(f, w, spconv_ref.rulebook_subm(idx, shape, ks), len(idx))
            oi = idx
        else:
            oi, oshape, pairs = spconv_ref.rulebook_conv(idx, shape, ks, st, pd)
            assert list(d.shape[2:]) == oshape
            o = spconv_ref.sparse_conv_native(f, w, pairs, len(oi))
            mask = torch.ones_like(d[:, 0], dtype=torch.bool)
            mask[oi[:, 0], oi[:, 1], oi[:, 2], oi[:, 3]] = False
            assert d.permute(0, 2, 3, 4, 1)[mask].abs().max() == 0         # exactly zero outside the out-site set
            key = ((oi[:, 0].astype(np.int64) * oshape[0] + oi[:, 1]) * oshape[1] + oi[:, 2]) * oshape[2] + oi[:, 3]
            assert (np.diff(key) > 0).all()                                  # sorted ascending (b,z,y,x)
        ref = d[oi[:, 0], :, oi[:, 1], oi[:, 2], oi[:, 3]]
        assert (o - ref).abs().max() < 1e-12


def _ref_sd(kind, seed):
    """seeded state dict with the reference module's key names/shapes (recorded by make_golden.py)"""
    with open(os.path.join(HERE, 'golden', 'state_dict_keys.json')) as f:
        keys = json.load(f)[kind]
    return {k: weights.seeded_tensor(k, shape, seed) for k, shape in keys}


@pytest.mark.parametrize('kind', ['VoxelBackBone8x', 'VoxelResBackBone8x'])
def test_oracle_backbone_matches_reference_golden(kind):
    voxels, coords, num = tiny_batch()
    feats = det_ref.mean_vfe(voxels, num)
    assert np.array_equal(feats.numpy(), GOLD['mean_vfe'])
    lv = det_ref.voxel_backbone(_ref_sd(kind, SEED), '', feats, coords, [41, 96, 96], 2, res=(kind == 'VoxelResBackBone8x'))
    assert np.array_equal(lv['out'].idx, GOLD[kind + '.out_idx'])
    assert util.rel_err(lv['out'].f, GOLD[kind + '.out_feat']) < 1e-6
    for name in ('x_conv1', 'x_conv2', 'x_conv3', 'x_conv4'):
        assert lv[name].f.shape[0] == int(GOLD['%s.%s.n' % (kind, name)][0])
        s = GOLD['%s.%s.sum' % (kind, name)]
        assert abs(lv[name].f.double().abs().sum().item() - s[1]) < 1e-5 * s[1]


def test_oracle_dense_chain_matches_reference_golden():
    voxels, coords, num = tiny_batch()
    lv = det_ref.voxel_backbone(_ref_sd('VoxelResBackBone8x', SEED), '', det_ref.mean_vfe(voxels, num), coords, [41, 96, 96], 2, res=True)
    sf = det_ref.height_compression(lv['out'])
    s2d = det_ref.bev_backbone(_ref_sd('BaseBEVBackbone', SEED + 1), '', sf, [5, 5], [1, 2], [1, 2])
    assert util.rel_err(s2d, GOLD['spatial_features_2d']) < 1e-5
    names = ['center', 'center_z', 'dim', 'rot', 'iou', 'hm']
    maps = det_ref.center_head_maps(_ref_sd('CenterHead', SEED + 2), '', s2d, names)
    for n in names:
        assert util.rel_err(maps[n], GOLD['head.' + n]) < 1e-5, n
    post = dict(MAX_OBJ_PER_SAMPLE=100, SCORE_THRESH=0.03, POST_CENTER_LIMIT_RANGE=[-80, -80, -10.0, 80, 80, 10.0],
                NMS_THRESH=0.7, NMS_PRE_MAXSIZE=4096, NMS_POST_MAXSIZE=500)
    gmaps = {n: torch.from_numpy(GOLD['head.' + n]) for n in names}
    got = det_ref.generate_predicted_boxes(gmaps, TINY_RANGE, util.VOXEL, 8, post, use_iou=True)
    for b in range(2):
        assert np.array_equal(got[b]['pred_boxes'].numpy(), GOLD['final.%d.boxes' % b])
        assert np.array_equal(got[b]['pred_scores'].numpy(), GOLD['final.%d.scores' % b])
        assert np.array_equal(got[b]['pred_labels'].numpy(), GOLD['final.%d.labels' % b])


def test_product_state_dict_keys_match_reference():
    """checkpoint compatibility: the product module trees expose exactly the reference's state-dict keys and shapes"""
    from detzero_b200.det import cp_modules
    with open(os.path.join(HERE, 'golden', 'state_dict_keys.json')) as f:
        ref = json.load(f)
    cfg = util.model_cfg()
    mods = {
        'VoxelBackBone8x': cp_modules['VoxelBackBone8x'](model_cfg=cfg.BACKBONE_3D, input_channels=5, grid_size=[96, 96, 40]),
        'VoxelResBackBone8x': cp_modules['VoxelResBackBone8x'](model_cfg=cfg.BACKBONE_3D, input_channels=5, grid_size=[96, 96, 40]),
        'BaseBEVBackbone': cp_modules['BaseBEVBackbone'](model_cfg=cfg.BACKBONE_2D, input_channels=256),
        'CenterHead': cp_modules['CenterHead'](model_cfg=cfg.DENSE_HEAD, input_channels=512, num_class=3, class_names=util.CLASS_NAMES,
                                               grid_size=[96, 96, 40], point_cloud_range=TINY_RANGE, voxel_size=util.VOXEL),
    }
    for kind, m in mods.items():
        mine = {k: list(v.shape) for k, v in m.state_dict().items()}
        theirs = {k: s for k, s in ref[kind]}
        assert mine == theirs, kind


def test_rotated_iou_restatement_properties():
    g = np.random.default_rng(0)
    b = np.concatenate([g.uniform(-5, 5, (50, 3)), g.uniform(1, 4, (50, 3)), g.uniform(-3.2, 3.2, (50, 1))], 1).astype(np.float32)
    iou = oracle.boxes_iou_bev(b, b)
    assert np.allclose(np.diag(iou), 1.0, atol=2e-2)                 # the 1e-2 corner margin inflates self-overlap a little
    assert np.allclose(iou, iou.T, atol=1e-4)
    axis = b.copy(); axis[:, 6] = 0
    a, c = axis[:10], axis[10:20]
    x1 = np.maximum(a[:, None, 0] - a[:, None, 3] / 2, c[None, :, 0] - c[None, :, 3] / 2)
    x2 = np.minimum(a[:, None, 0] + a[:, None, 3] / 2, c[None, :, 0] + c[None, :, 3] / 2)
    y1 = np.maximum(a[:, None, 1] - a[:, None, 4] / 2, c[None, :, 1] - c[None, :, 4] / 2)
    y2 = np.minimum(a[:, None, 1] + a[:, None, 4] / 2, c[None, :, 1] + c[None, :, 4] / 2)
    inter = np.clip(x2 - x1, 0, None) * np.clip(y2 - y1, 0, None)
    ref = inter / (a[:, None, 3] * a[:, None, 4] + c[None, :, 3] * c[None, :, 4] - inter)
    assert np.abs(oracle.boxes_iou_bev(a, c) - ref).max() < 2e-2


def test_c_abi_exports_every_declared_symbol():
    """the library loads and exports every function include/detzero_b200.h declares (no compute without a GPU)"""
    from detzero_b200 import _lib
    root = os.path.dirname(HERE)
    lib_path = os.path.join(root, 'detzero_b200', 'libdetzero_b200.so')
    if not os.path.exists(lib_path):
        import __graft_entry__ as g
        g.build()
    hdr = open(os.path.join(root, 'include', 'detzero_b200.h')).read()
    declared = set(re.findall(r'\b(dz_[a-z0-9_]+)\s*\(', hdr))
    l = _lib.lib()
    for name in declared:
        assert hasattr(l, name), name
    assert declared == set(_lib.exported_symbols())
    assert l.dz_sm_arch() == 100 and l.dz_version() >= 100


def test_product_path_fails_loudly_without_cuda():
    """no CPU fallback: ops on CPU tensors raise instead of silently computing elsewhere"""
    from detzero_b200.spconv.pytorch import SparseConvTensor
    with pytest.raises(RuntimeError):
        SparseConvTensor(torch.zeros(4, 5), torch.zeros(4, 4, dtype=torch.int32), [41, 96, 96], 1)


def test_config_semantics(tmp_path):
    from detzero_b200.config import AttrDict, cfg_from_list, cfg_from_yaml_file
    base = tmp_path / 'base.yaml'
    base.write_text('POINT_CLOUD_RANGE: [-1, -1, -1, 1, 1, 1]\nDATA_PROCESSOR:\n  - NAME: shuffle_points\n')
    top = tmp_path / 'top.yaml'
    top.write_text('CLASS_NAMES: [A, B]\nDATA_CONFIG:\n  _BASE_CONFIG_: base.yaml\nMODEL:\n  NAME: CenterPoint\n  VFE:\n    NAME: MeanVFE\nOPT:\n  LR: 0.003\n  STEPS: [35, 45]\n')
    c = cfg_from_yaml_file(str(top), AttrDict())
    assert c.DATA_CONFIG.POINT_CLOUD_RANGE[3] == 1 and c.MODEL.VFE.NAME == 'MeanVFE'
    assert c.DATA_CONFIG.DATA_PROCESSOR[0].NAME == 'shuffle_points'
    cfg_from_list(['OPT.LR', '0.01', 'OPT.STEPS', '1,2'], c)
    assert c.OPT.LR == 0.01 and c.OPT.STEPS == [1, 2]


def test_data_processor_and_collate():
    from detzero_b200.det.dataset import SyntheticWaymoDataset, default_waymo_1sweep_cfg, mask_points_by_range
    ds = SyntheticWaymoDataset(default_waymo_1sweep_cfg(), util.CLASS_NAMES, num_frames=2, n_points=5000)
    assert list(ds.grid_size) == [1504, 1504, 40] and ds.max_num_voxels == 200000 and ds.max_points_per_voxel == 5
    items = [ds[0], ds[1]]
    assert items[0]['points'].shape[1] == 5
    batch = ds.collate_batch(items)
    assert batch['points'].shape[1] == 6 and batch['batch_size'] == 2
    assert (batch['points'][:batch['points_per_frame'][0], 0] == 0).all() and (batch['points'][batch['points_per_frame'][0]:, 0] == 1).all()
    p = np.array([[75.2, 0, 0], [75.3, 0, 0], [0, -75.2, 9]], np.float32)
    assert mask_points_by_range(p, util.WAYMO_RANGE).tolist() == [True, False, True]    # inclusive bound, z unfiltered


def test_rotated_iou_restatement_matches_compiled_reference():
    """the C restatement of the rotated-BEV IoU agrees bit for bit with the reference's own iou3d_cpu.cpp (compiled by
    oracle/build_ref.py; its output on these boxes is stored by tests/golden/make_golden_host.py)"""
    want = np.load(os.path.join(HERE, 'golden', 'host.npz'))['iou_bev']
    b = util.iou_boxes()
    assert np.array_equal(want, oracle.boxes_iou_bev(b, b))


def test_yaml_config_builds_registry_model():
    """the shipped YAML (same keys as the reference's centerpoint_1sweep.yaml) builds the detector through the registry"""
    from detzero_b200.config import AttrDict, cfg_from_yaml_file
    from detzero_b200.det import build_network
    from detzero_b200.det.dataset import SyntheticWaymoDataset
    root = os.path.join(os.path.dirname(HERE), 'detzero_b200')
    cfg = cfg_from_yaml_file(os.path.join(root, 'cfgs', 'det_model_cfgs', 'centerpoint_1sweep.yaml'), AttrDict())
    assert cfg.DATA_CONFIG.POINT_CLOUD_RANGE == [-75.2, -75.2, -2, 75.2, 75.2, 4]
    ds = SyntheticWaymoDataset(cfg.DATA_CONFIG, cfg.CLASS_NAMES, training=False, num_frames=1, n_points=1000)
    model = build_network(cfg.MODEL, len(cfg.CLASS_NAMES), ds)
    names = [type(m).__name__ for m in model.module_list]
    assert names == ['MeanVFE', 'VoxelResBackBone8x', 'HeightCompression', 'BaseBEVBackbone', 'CenterHead']
    assert model.backbone3d.sparse_shape == [41, 1504, 1504] and model.vfe.max_voxels == 200000


def test_row_major_table_helper_matches_k_major():
    """ops.table_to_rows: the host-side conversion between the two rulebook table layouts of include/detzero_b200.h
    (k-major (K, cap) <-> row-major (cap, 32) with the neighbour bit mask in column 27); pure torch, runs on the CPU"""
    from detzero_b200 import ops
    g = np.random.default_rng(4)
    idx = weights.random_sparse_coords(9, 1, [7, 12, 12], 0.15)
    pairs = spconv_ref.rulebook_subm(idx, [7, 12, 12], 3)
    n = len(idx)
    nbr = torch.full((27, n), -1, dtype=torch.int32)
    for k, (i_in, i_out) in enumerate(pairs):
        nbr[k, torch.as_tensor(np.asarray(i_out), dtype=torch.long)] = torch.as_tensor(np.asarray(i_in), dtype=torch.int32)
    tab = ops.table_to_rows(nbr)
    assert tab.shape == (n, 32) and torch.equal(tab[:, :27].t().contiguous(), nbr)
    bits = ((nbr >= 0).to(torch.int64) << torch.arange(27)[:, None]).sum(0)
    assert torch.equal(tab[:, 27].to(torch.int64), bits) and torch.all(tab[:, 28:] == 0)
    assert int(bits[0]) & (1 << 13)                      # every site is its own centre-tap neighbour


def test_bench_cpu_arm_produces_detections():
    """the CPU arm of bench.py (`--impl reference` / cpu_baseline) runs the oracle chain on the bench workload with the same
    head calibration as the GPU arm: a frame must reach post-processing with real work (500 boxes into the rotated NMS)"""
    import sys
    argv, sys.argv = sys.argv, ['bench.py']
    try:
        import bench
        torch.set_num_threads(min(8, os.cpu_count() or 1))
        out = bench.cpu_frame_fn('VoxelBackBone8x')(0)
    finally:
        sys.argv = argv
    d = out[0]
    assert d['pred_boxes'].shape == (500, 7) and d['pred_scores'].shape == (500,)
    assert float(d['pred_scores'].max()) > 0.3 and int(d['pred_labels'].min()) >= 1
