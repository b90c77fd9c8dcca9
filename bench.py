#!/usr/bin/env python
"""bench.py -- Waymo-shape frames/sec through the B200-native DetZero hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W             # BASELINE configs[1] (default): this framework, one rank per GPU
    python bench.py --impl reference --steps K --warmup W      # the reference algorithm's CPU path (oracle port), same config
    python bench.py --config 3|4|5 ...                         # the other BASELINE configurations (see below)
    python bench.py --dump-outputs DIR ...                     # config 2: + the last timed step's detections as DIR/*.npy

--config 2 (default; BASELINE configs[1]): CenterPoint 1-sweep VoxelBackBone8x, synthetic 180 K-pt Waymo-range clouds, 8 frames
    per step and GPU (the reference's BATCH_SIZE_PER_GPU, centerpoint_1sweep.yaml:88).  A step = raw points -> hard voxelization
    (+MeanVFE) -> rulebooks -> sparse backbone -> BEV scatter -> BEV backbone -> CenterHead -> decode -> rotated NMS
    (-> per-step NCCL all-gather of the boxes when N > 1: dist.SequenceGather, ONE collective, NMS writes into its send buffer).
    Sparse convs default to the fp32-level `bf16x2` mode; the other modes are measured in the same run (`config.also`).
--config 3 (BASELINE configs[2]): 5-sweep (~900 K pts) DynamicMeanVFE -> VoxelResBackBone8x in bf16 -> BEV -> head, plus the
    sparse-conv GB/s sweep over the voxel count (`config.sweep`).
--config 4 (BASELINE configs[3]): PRM + GRM refiner, 256 tracks x 200 boxes, 256 and 1024 points per crop; tracks/s.
--config 5 (BASELINE configs[4]): a 199-frame sequence sharded frame i -> rank i % W, per-sequence NCCL box gather inside the
    timed region, then PRM/GRM on tracks sharded by id and the second gather; strong scaling, frames/s.

Timing: CUDA events around every step on the launching stream, L2 flushed (256 MiB write) between steps outside the timed
intervals, max over ranks of the summed step times.  `value` has the input resident in HBM; `e2e` includes the pinned-host ->
device copy of the step's inputs and the device -> host read of the results through the public API.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_POINTS = 180000
NUM_CLOUDS = 4
ALSO_MODES = ['tf32x3', 'tf32', 'bf16', 'bf16x2']


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', type=int, default=2, choices=[2, 3, 4, 5], help='BASELINE.json configs[config-1]')
    ap.add_argument('--backbone', default=None, choices=['VoxelBackBone8x', 'VoxelResBackBone8x'])
    ap.add_argument('--mode', default=os.environ.get('DZ_MODE', 'tf32'),
                    help='dense BEV/head convs: tf32 (tcgen05; what the reference gets from cuDNN by default, SURVEY A.6) | fp32 (exact FMA)')
    ap.add_argument('--sp-mode', default=os.environ.get('DZ_SP_MODE'),
                    help='sparse-conv arithmetic: bf16x2 (default: fp32-level, 2 bf16 planes, tcgen05) | tf32x3 (fp32-level, 3 TF32 passes) | '
                         'fp32 (exact FMA, spconv default) | tf32 | bf16')
    ap.add_argument('--batch', type=int, default=None,
                    help='frames per step and GPU; config 2 default 8 = the reference config (centerpoint_1sweep.yaml:88 BATCH_SIZE_PER_GPU)')
    ap.add_argument('--no-also', action='store_true', help='config 2: skip the extra sparse-conv modes (config.also)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='launch kernels eagerly instead of replaying a CUDA graph')
    ap.add_argument('--no-schedule', action='store_true', help='run the tensor-core sparse convs without the mask-grouped tile schedule')
    ap.add_argument('--layer-times', action='store_true', help='print per-layer sparse-conv times of the traced step to stderr')
    ap.add_argument('--stage-times', action='store_true', help='print a per-stage device time table to stderr')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='config 2: write the detections of the last timed step (rank 0) to DIR/<name>.npy, float32')
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != 'ours' or args.config != 2):
        ap.error('--dump-outputs is implemented for --impl ours --config 2')
    return args


def make_model_cfg(backbone, mode, sp_mode, vfe='MeanVFE'):
    from detzero_b200 import synthetic
    cfg = synthetic.model_cfg(backbone, mode)
    cfg.BACKBONE_3D.COMPUTE_MODE = sp_mode
    cfg.VFE.NAME = vfe
    if os.environ.get('DZ_NO_OVERLAP'):
        cfg.BACKBONE_3D.OVERLAP_RULEBOOKS = False      # diagnostic: rulebooks inline on the main stream
    return cfg


def tune_head_for_bench(model):
    """The seeded random weights give a flat heatmap and a negative IoU map, i.e. no detections and an idle post-processing
    stage.  Re-scale the heatmap / IoU head outputs (same rule for the GPU arm and the CPU arm) so that a frame yields
    ~1.5 K candidates above SCORE_THRESH, 500 boxes into the rotated NMS (calibrated with the oracle on frame 0)."""
    import torch
    sd = model.state_dict()
    g = torch.Generator().manual_seed(1234)
    with torch.no_grad():
        sd['dense_head.heads_list.0.hm.0.1.bias'].copy_(torch.randn(64, generator=g) * 0.2)
        sd['dense_head.heads_list.0.hm.1.weight'].mul_(torch.tensor([340.865, 293.364, 329.442]).view(3, 1, 1, 1))
        sd['dense_head.heads_list.0.hm.1.bias'].copy_(torch.tensor([-7.4753, -0.0872, 14.5139]))
        sd['dense_head.heads_list.0.iou.1.bias'].fill_(0.85)
    return {k: v.detach().clone() for k, v in model.state_dict().items()}


def build_inputs(batch, num_batches=NUM_CLOUDS, seed0=0):
    from detzero_b200 import synthetic
    from detzero_b200.det.dataset import SyntheticWaymoDataset, default_waymo_1sweep_cfg
    ds = SyntheticWaymoDataset(default_waymo_1sweep_cfg(), synthetic.CLASS_NAMES, training=False, num_frames=num_batches * batch,
                               n_points=N_POINTS, seed0=seed0)
    batches = []
    for i in range(num_batches):
        items = [ds[i * batch + j] for j in range(batch)]
        for it in items:                    # fixed shape for CUDA-graph replay: pad with far out-of-range points (dropped by
            p = it['points']                # the voxelizer exactly like any other out-of-range point)
            if p.shape[0] < N_POINTS:
                pad = np.full((N_POINTS - p.shape[0], p.shape[1]), 1.0e4, dtype=np.float32)
                it['points'] = np.concatenate([p, pad], axis=0)
        batches.append(ds.collate_batch(items))
    return ds, batches


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(',')
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower() == 'active':
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}
        return {'sm_mhz': float(np.median(self.samples)), 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}


def hbm_peak():
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        return json.load(open(peaks_path)), 'measured'
    return {'hbm_gbs': 6650.0, 'bf16_tflops_sustained': 1450.0}, 'fallback'


# ------------------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference path (voxelizer C restatement + spconv 'Native' + torch-CPU convs)
# ------------------------------------------------------------------------------------------------------------------
def cpu_frame_fn(backbone, seed=3):
    import torch
    import oracle
    from oracle import det_ref, weights
    from tests import util
    from detzero_b200.det import build_network
    ds, batches = build_inputs(1)
    model = build_network(make_model_cfg(backbone, 'fp32', 'fp32'), 3, ds).eval()
    weights.load_seeded(model, seed)
    sd = tune_head_for_bench(model)
    vox = oracle.Point2VoxelCPU3d(util.VOXEL, util.WAYMO_RANGE, 5, 5, 200000)
    post = dict(MAX_OBJ_PER_SAMPLE=500, SCORE_THRESH=0.03, POST_CENTER_LIMIT_RANGE=[-80, -80, -10.0, 80, 80, 10.0],
                NMS_THRESH=0.7, NMS_PRE_MAXSIZE=4096, NMS_POST_MAXSIZE=500)
    res = backbone == 'VoxelResBackBone8x'

    def run(i):
        pts = batches[i % len(batches)]['points'][:, 1:]
        with torch.no_grad():
            v, c, n = vox.point_to_voxel(pts)
            lv = det_ref.voxel_backbone(sd, 'backbone3d.', det_ref.mean_vfe(v, n), np.pad(c, ((0, 0), (1, 0))), [41, 1504, 1504], 1, res)
            s2d = det_ref.bev_backbone(sd, 'backbone2d.', det_ref.height_compression(lv['out']), [5, 5], [1, 2], [1, 2])
            maps = det_ref.center_head_maps(sd, 'dense_head.', s2d, ['center', 'center_z', 'dim', 'rot', 'iou', 'hm'])
            return det_ref.generate_predicted_boxes(maps, util.WAYMO_RANGE, util.VOXEL, 8, post, use_iou=True)
    return run


def workload_name(backbone, batch):
    return 'CenterPoint 1-sweep %s, synthetic 180K-pt Waymo-range cloud, fp32, batch %d/GPU' % (backbone, batch)


def run_reference(args):
    """--impl reference: the reference algorithm on the host cores (oracle port; spconv itself cannot be installed
    here).  Same workload as the GPU arm; one step = one FRAME of it (a bounded sample).  Under torchrun only rank 0 works."""
    import torch
    if int(os.environ.get('RANK', '0')) != 0:
        return
    backbone = args.backbone or 'VoxelBackBone8x'
    cores = cpu_threads()
    torch.set_num_threads(cores)
    run = cpu_frame_fn(backbone)
    for i in range(args.warmup):
        run(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        run(i)
    dt = time.perf_counter() - t0
    fps = args.steps / dt
    line = {'impl': 'reference', 'metric': 'Waymo-shape frames/sec', 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 * dt / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
            'config': {'workload': workload_name(backbone, args.batch or 8),
                       'arm': 'oracle port of the reference algorithm on the host CPU (spconv cannot be installed here); one step = ONE frame '
                              'of the workload (bounded sample): CPU frames/s does not depend on the batch size'},
            'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                             'sample': '%d frames of the same workload, one frame per step, torch threads=%d' % (args.steps, cores)},
            'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


def cpu_threads():
    """threads the CPU arm uses: the oracle port (numpy rulebooks + torch gather/mm/index_add + oneDNN convs) stops scaling
    -- and on a 128-core host gets ~30x SLOWER from oversubscription -- beyond ~16 threads"""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get('DZ_CPU_THREADS', '16'))))


def cpu_baseline(backbone):
    import torch
    cores = cpu_threads()
    torch.set_num_threads(cores)
    run = cpu_frame_fn(backbone)
    run(0)
    t0 = time.perf_counter()
    n = 0
    while n < 2 or (time.perf_counter() - t0 < 12.0 and n < 8):
        run(n)
        n += 1
    dt = time.perf_counter() - t0
    return {'value': n / dt, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
            'sample': '%d frames of the same workload (oracle port: C voxelizer + spconv-Native restatement + torch-CPU convs)' % n}


# ------------------------------------------------------------------------------------------------------------------
class Env:
    """ranks, device, timing helpers shared by the configurations"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.rank = int(os.environ.get('RANK', '0'))
        self.local = int(os.environ.get('LOCAL_RANK', '0'))
        assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm'
        torch.cuda.set_device(self.local)
        self.dev = torch.device('cuda', self.local)
        if self.world > 1:
            dist.init_process_group('nccl', device_id=self.dev)
        self.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=self.dev)

    def timed(self, fn, steps, warmup):
        """W untimed + K timed steps, CUDA events per step, L2 flush between steps (outside the timed intervals), barrier +
        synchronize on both sides, max over ranks of the summed step times (ms)"""
        torch, dist = self.torch, self.dist
        for i in range(warmup):
            fn(i)
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        evs = []
        for i in range(steps):
            self.flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn(warmup + i)
            e.record()
            evs.append((s, e))
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        total_ms = sum(s.elapsed_time(e) for s, e in evs)
        t = torch.tensor([total_ms], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def done(self):
        if self.world > 1:
            self.dist.destroy_process_group()


class Detector:
    """one CenterPoint model + its captured CUDA graph for a fixed batch shape"""

    def __init__(self, env, ds, batches, backbone, mode, sp_mode, use_graph=True, vfe='MeanVFE', gather=None, slab=None):
        from detzero_b200 import ops, synthetic
        from detzero_b200.det import build_network
        torch = env.torch
        self.env, self.batches, self.ops = env, batches, ops
        self.model = build_network(make_model_cfg(backbone, mode, sp_mode, vfe), 3, ds).eval()
        synthetic.load_seeded(self.model, 3)
        tune_head_for_bench(self.model)
        self.model = self.model.to(env.dev)
        self.host_pts = [torch.from_numpy(b['points']).pin_memory() for b in batches]
        self.dev_pts = [h.to(env.dev) for h in self.host_pts]
        self.gather = gather                               # dist.SequenceGather (per-step gather) or None
        self.slab = slab if slab is not None else (gather.slot(0, batches[0]['batch_size']) if gather is not None else None)
        self.graph = None
        self.launches_per_step = 0
        self.use_graph = use_graph

    def batch_dict(self, i, pts):
        b = self.batches[i % len(self.batches)]
        d = {'points': pts, 'points_per_frame': b['points_per_frame'], 'frame_id': b['frame_id'], 'batch_size': b['batch_size']}
        if self.slab is not None:
            d['gather_slab'] = self.slab                   # NMS writes straight into the gather's send buffer
        return d

    def settle(self):
        """capacity hints (buffer sizes / launch grids follow the observed sparsity): every input through the public API until no
        overflow is reported"""
        torch = self.env.torch
        for rep in range(2):
            for i in range(len(self.batches)):
                for attempt in range(6):
                    try:
                        with torch.no_grad():
                            self.model(self.batch_dict(i, self.dev_pts[i]))
                        break
                    except RuntimeError as e:
                        if 'overflow' not in str(e):
                            raise
        torch.cuda.synchronize()

    def capture(self):
        if not self.use_graph:
            return
        self.static_pts = self.dev_pts[0].clone()
        self.ops.reset_launch_count()
        self.graph, self.out = self.model.capture_graph(self.batch_dict(0, self.static_pts), warmup=0)
        self.launches_per_step = self.ops.launch_count()

    def step_resident(self, i):
        torch = self.env.torch
        k = i % len(self.batches)
        if self.graph is not None:
            self.static_pts.copy_(self.dev_pts[k], non_blocking=True)      # device->device, part of the step
            self.graph.replay()
            out = self.out
        else:
            with torch.no_grad():
                out = self.model.forward_device(self.batch_dict(i, self.dev_pts[k]))
        if self.gather is not None:
            self.gathered = self.gather.gather()                           # ONE NCCL all-gather, inside the timed region
        self.last_out = out
        return out

    def _prefetch(self, i):
        """pinned host -> device staging copy of step i's points on the copy stream (overlaps the running step's kernels)"""
        torch = self.env.torch
        if not hasattr(self, 'stage'):
            self.stage = torch.empty_like(self.dev_pts[0])
            self.copy_stream = torch.cuda.Stream(device=self.env.dev)
            self.ev_copied, self.ev_consumed = torch.cuda.Event(), torch.cuda.Event()
            self.ev_consumed.record(torch.cuda.current_stream())
        self.copy_stream.wait_event(self.ev_consumed)                          # the previous contents have been moved into the graph's input
        with torch.cuda.stream(self.copy_stream):
            self.stage.copy_(self.host_pts[i % len(self.batches)], non_blocking=True)
            self.ev_copied.record(self.copy_stream)
        self.prefetched = i

    def step_e2e(self, i, out_host, state):
        """one step through the public API from HOST buffers: every call issues one H2D (34.6 MB of points) and one D2H (counts + boxes).
        With the CUDA graph the input is double-buffered like any data loader does: the H2D of step i+1 is issued at the start of step i
        (copy stream, pinned memory) and overlaps its kernels; step i consumes the copy made during step i-1."""
        torch = self.env.torch
        k = i % len(self.batches)
        with torch.no_grad():
            if self.graph is not None:
                if getattr(self, 'prefetched', None) != i:
                    self._prefetch(i)                                          # cold start (first call): not overlapped
                torch.cuda.current_stream().wait_event(self.ev_copied)
                self.static_pts.copy_(self.stage, non_blocking=True)           # device -> device into the graph's static input
                self.ev_consumed.record(torch.cuda.current_stream())
                self._prefetch(i + 1)                                          # next step's H2D, overlapped with this step's replay
                self.graph.replay()
                pred, _ = self.model.post_processing(self.out)                 # the step's D2H (counts, overflow flag) + dicts
            else:
                pts = self.host_pts[k].to(self.env.dev, non_blocking=True)
                pred, _ = self.model(self.batch_dict(i, pts))                  # public API: includes the D2H read of counts
            if self.gather is not None:
                self.gathered = self.gather.gather()
            d2h = 4 * (len(pred) + 8)                                          # the count / flag read inside post_processing
            padded = (self.out if self.graph is not None else self.model.last_batch_dict)['final_boxes_padded'] if (
                self.graph is not None or hasattr(self.model, 'last_batch_dict')) else None
            if padded is not None and padded.shape == out_host.shape:          # every frame's boxes go back to pinned host memory: ONE copy
                out_host.copy_(padded, non_blocking=True)                      # of the fixed-shape (B, 500, 9) result
                d2h += padded.numel() * 4
            else:
                for b, pd in enumerate(pred):
                    n = pd['pred_boxes'].shape[0]
                    out_host[b, :n, :7].copy_(pd['pred_boxes'], non_blocking=True)
                    d2h += n * 7 * 4
            state['d2h'], state['boxes'] = d2h, sum(pd['pred_boxes'].shape[0] for pd in pred)
        return pred


def sparse_conv_roofline(det, layer_times, batch, storage_bytes=4):
    """achieved = algorithmic bytes of all sparse-conv launches of one step / their summed duration (CUDA events on the
    launching stream, one eager traced step); algorithmic bytes per layer = (N_in*Cin + N_out*Cout)*s + pairs*8 + K*Cin*Cout*s
    (+ N_out*Cout*s with a residual), s = storage bytes per value -- SURVEY.md §8d."""
    import torch
    from detzero_b200 import ops
    peaks, which = hbm_peak()
    peak = peaks['hbm_gbs']
    rec = ops.enable_spconv_trace(True)
    with torch.no_grad():
        det.model.forward_device(det.batch_dict(0, det.dev_pts[0]))
    torch.cuda.synchronize()
    ops.enable_spconv_trace(False)
    tot_bytes, tot_ms, tot_flops, layers = 0.0, 0.0, 0.0, []
    s = storage_bytes
    for r in rec:
        if r['nbr'].shape[1] == 32 and r['nbr'].shape[0] != r['K']:      # tensor-core launch: row-major table (cap, 32)
            valid = r['nbr'][:r['n_out'], :r['K']].t() >= 0
            if r['row_order'] is not None:
                valid = valid[:, r['row_order'][:r['n_out']].long()]        # tile order (for the offsets/tile statistic)
        else:
            valid = r['nbr'][:, :r['n_out']] >= 0
        pairs = int(valid.sum().item())
        K, cin, cout = r['K'], r['cin'], r['cout']
        b = (r['n_in'] * cin + r['n_out'] * cout) * s + pairs * 8 + K * cin * cout * s + (r['n_out'] * cout * s if r['residual'] else 0)
        ms = r['start'].elapsed_time(r['end'])
        if layer_times:
            T = (r['n_out'] + 127) // 128
            v = torch.zeros((valid.shape[0], T * 128), dtype=torch.bool, device=valid.device)
            v[:, :r['n_out']] = valid
            touched = int(v.view(valid.shape[0], T, 128).any(2).sum().item())
            print('spconv layer K=%d cin=%d cout=%d n_out=%d pairs=%d offsets/tile=%.1f scheduled=%s  %.1f us  %.0f GB/s' % (
                K, cin, cout, r['n_out'], pairs, touched / max(T, 1), r['row_order'] is not None, 1000 * ms, b / ms / 1e6), file=sys.stderr)
        layers.append({'K': K, 'cin': cin, 'cout': cout, 'n_out': r['n_out'], 'us': round(1000 * ms, 1), 'GBps': round(b / ms / 1e6, 1)})
        tot_bytes += b
        tot_flops += 2.0 * pairs * cin * cout
        tot_ms += ms
    achieved = tot_bytes / (tot_ms / 1000.0) / 1e9 if tot_ms > 0 else 0.0
    return {'bound': 'hbm', 'kernel': 'sparse conv (all %d sparse-conv launches of one step)' % len(rec), 'achieved': achieved,
            'peak': peak, 'peak_source': which, 'unit': 'GB/s', 'frac': achieved / peak,
            'traffic': committed_traffic(det, batch), 'traffic_source': 'committed ncu --set full capture of the same 14 launches '
            '(profiles/r02_ncu_full_spconv_bf16x2_batch8.json, dram__bytes_read.sum + dram__bytes_write.sum); NOT measured in this run -- null for '
            'any other mode / batch / backbone',
            'algorithmic_bytes_per_step': tot_bytes, 'storage_bytes_per_value': s, 'algorithmic_flops_per_step': tot_flops,
            'ms_per_step': tot_ms, 'frames_per_step': batch, 'layers': layers}


def committed_traffic(det, batch):
    """DRAM bytes per step of the sparse-conv launches from the committed ncu capture -- only for the exact configuration it was taken on"""
    path = os.path.join(ROOT, 'profiles', 'r02_ncu_full_spconv_bf16x2_batch8.json')
    try:
        mode = det.model.backbone3d.model_cfg.get('COMPUTE_MODE')
        if mode == 'bf16x2' and batch == 8 and type(det.model.backbone3d).__name__ == 'VoxelBackBone8x' and os.path.exists(path):
            j = json.load(open(path))
            return (j['dram_read_MB'] + j['dram_write_MB']) * 1e6
    except Exception:
        pass
    return None


def dump_outputs(path, pred):
    """what a caller of CenterPoint.forward receives for each frame of the step: pred_boxes (n, 7), pred_scores (n,) and
    pred_labels (n,), as DIR/frame<b>_<key>.npy in float32 (labels are small integers, exact in float32)"""
    os.makedirs(path, exist_ok=True)
    for b, d in enumerate(pred):
        for key in ('pred_boxes', 'pred_scores', 'pred_labels'):
            np.save(os.path.join(path, 'frame%d_%s.npy' % (b, key)), d[key].float().cpu().numpy())


SP_DTYPE = {'fp32': 'fp32 FMA', 'tf32x3': 'tf32x3 (3 TF32 passes, fp32-level)',
            'bf16x2': 'bf16x2 (2 bf16 planes = 16 significand bits in 4 bytes, fp32 accumulate; <= 2e-4 vs the fp32 oracle through the whole backbone)',
            'tf32': 'tf32 (1 pass)', 'bf16': 'bf16 (storage and products)'}


# ------------------------------------------------------------------------------------------------------------------
def run_config2(args):
    from detzero_b200 import synthetic
    from detzero_b200 import dist as dzdist
    env = Env()
    torch = env.torch
    backbone = args.backbone or 'VoxelBackBone8x'
    batch = args.batch or 8
    sp_mode = args.sp_mode or synthetic.DEFAULT_SP_MODE
    if args.no_schedule:
        from detzero_b200.spconv import pytorch as _sp
        _sp._SparseConv.SCHEDULE_TILES = False
    ds, batches = build_inputs(batch, seed0=env.rank * 64)            # each rank takes its own frames
    gather = dzdist.SequenceGather(batch * env.world, K=500, device=env.dev) if env.world > 1 else None
    det = Detector(env, ds, batches, backbone, args.mode, sp_mode, use_graph=not args.no_graph, gather=gather)
    det.settle()
    out_host = torch.empty((batch, 500, 9), dtype=torch.float32).pin_memory()
    state = {'d2h': 0, 'boxes': 0}

    if args.stage_times and env.rank == 0:
        names = [type(m).__name__ for m in det.model.module_list]
        acc, reps = [0.0] * len(names), 6
        with torch.no_grad():
            for f in range(reps + 2):
                bd = det.batch_dict(f, det.dev_pts[f % len(batches)])
                env.flush.zero_()
                evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
                evs[0].record()
                for k, m in enumerate(det.model.module_list):
                    bd = m(bd)
                    evs[k + 1].record()
                torch.cuda.synchronize()
                if f >= 2:
                    for k in range(len(names)):
                        acc[k] += evs[k].elapsed_time(evs[k + 1]) / reps
        print('stage times (eager, us/step): ' + ', '.join('%s %.0f' % (n, 1000 * t) for n, t in zip(names, acc)) +
              ' | total %.0f' % (1000 * sum(acc)), file=sys.stderr)

    det.capture()
    sampler = ClockSampler(env.local)
    sampler.start()
    total_ms = env.timed(det.step_resident, args.steps, args.warmup)
    sampler.stop_flag = True
    if args.dump_outputs and env.rank == 0:
        with torch.no_grad():                               # before the e2e arm replays the graph into the same output buffers
            dump_outputs(args.dump_outputs, det.model.post_processing(det.last_out)[0])
    e2e_ms = env.timed(lambda i: det.step_e2e(i, out_host, state), args.steps, args.warmup)
    with torch.no_grad():                                   # overflow check of the resident-arm configuration (flag + counts)
        det.model.post_processing(det.step_resident(0))
    frames = args.steps * batch * env.world
    value, e2e = frames / (total_ms / 1000.0), frames / (e2e_ms / 1000.0)
    launches = (det.launches_per_step if det.graph is not None else 0) * args.steps
    roof = sparse_conv_roofline(det, args.layer_times, batch, storage_bytes=2 if sp_mode == 'bf16' else 4)

    also = {}
    if not args.no_also and env.world == 1:
        for m in ALSO_MODES:
            if m == sp_mode:
                continue
            d2 = Detector(env, ds, batches, backbone, args.mode, m, use_graph=not args.no_graph)
            d2.settle()
            d2.capture()
            ms2 = env.timed(d2.step_resident, args.steps, max(2, min(args.warmup, 3)))
            r2 = sparse_conv_roofline(d2, False, batch, storage_bytes=2 if m == 'bf16' else 4)
            also[m] = {'value': args.steps * batch / (ms2 / 1000.0), 'unit': 'frames/s', 'ms_per_step': ms2 / args.steps, 'steps': args.steps,
                       'sparse_conv_ms_per_step': r2['ms_per_step'], 'sparse_conv_roofline_frac': r2['frac'], 'precision': SP_DTYPE[m]}
            del d2
            torch.cuda.empty_cache()

    line = {
        'metric': 'Waymo-shape frames/sec', 'value': value, 'unit': 'frames/s', 'n_gpus': env.world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': total_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None,
        'dtype': 'fp32' if (args.mode == 'fp32' and sp_mode == 'fp32') else
                 'sparse convs: %s; dense BEV/head convs: %s products, fp32 accumulate (the reference\'s cuDNN default)' % (SP_DTYPE[sp_mode], args.mode),
        'data': 'synthetic',
        'config': {'workload': workload_name(backbone, batch),
                   'sparse_conv_mode': sp_mode, 'dense_conv_mode': args.mode, 'parallelism': 'frames sharded dp%d' % env.world,
                   'collective': ('per-step all-gather of the padded boxes of all ranks (dist.SequenceGather: ONE ncclAllGather of %d B per rank, '
                                  'NMS writes into the send buffer), inside the timed region' % (gather.send.numel() * 4)) if gather else 'none (1 GPU)',
                   'l2': 'flushed (256 MiB write) between steps, outside the timed intervals',
                   'launch': 'eager' if args.no_graph else 'CUDA graph replay of CenterPoint.forward_device',
                   'detections_last_step': int(state['boxes']), 'also': also},
        'e2e': {'value': e2e, 'unit': 'frames/s', 'h2d_bytes_per_step': int(det.host_pts[0].numel() * 4),
                'd2h_bytes_per_step': int(state['d2h'])},          # boxes of every frame + the count read, last step
        'gpu_launches': launches,
        'clocks': sampler.summary(),
        'roofline': roof,
    }
    if env.rank == 0 and env.world == 1 and not args.no_cpu_baseline:
        line['cpu_baseline'] = cpu_baseline(backbone)
    if env.rank == 0:
        print(json.dumps(line))
    env.done()


# ------------------------------------------------------------------------------------------------------------------
def five_sweep_cloud(seed, n_target=900000, subsample=1.0):
    """BASELINE configs[2]: 5 clouds with ego-motion offsets 0..2 m and time column 0, -0.1 .. -0.4 (SURVEY §8d config 3)"""
    from detzero_b200.det.dataset import synth_waymo_cloud
    parts = [synth_waymo_cloud(seed * 5 + s, n_target // 5, sweep=s, ego_shift=0.5 * s) for s in range(5)]
    pts = np.concatenate(parts, axis=0).astype(np.float32)              # (N, 6): x y z intensity elongation time
    if subsample < 1.0:
        g = np.random.default_rng(seed)
        pts = pts[g.random(pts.shape[0]) < subsample]
    keep = (np.abs(pts[:, 0]) <= 75.2) & (np.abs(pts[:, 1]) <= 75.2)
    return pts[keep]


def run_config3(args):
    """5-sweep ~900 K-pt clouds, DynamicMeanVFE -> VoxelResBackBone8x (bf16) -> BEV -> CenterHead; one frame per step"""
    from detzero_b200 import synthetic
    from detzero_b200.det.dataset import SyntheticWaymoDataset, default_waymo_1sweep_cfg
    env = Env()
    torch = env.torch
    backbone = args.backbone or 'VoxelResBackBone8x'
    sp_mode = args.sp_mode or 'bf16'
    dcfg = default_waymo_1sweep_cfg()
    dcfg.POINT_FEATURE_ENCODING.used_feature_list = ['x', 'y', 'z', 'intensity', 'elongation', 'offset']      # waymo_5sweeps.yaml: + time
    ds = SyntheticWaymoDataset(dcfg, synthetic.CLASS_NAMES, training=False, num_frames=1, n_points=N_POINTS)

    def batches_for(sub, n=NUM_CLOUDS):
        out, npts = [], None
        for i in range(n):
            p = five_sweep_cloud(env.rank * 16 + i, subsample=sub)
            npts = p.shape[0] if npts is None else npts
            p = p[:npts] if p.shape[0] >= npts else np.concatenate([p, np.full((npts - p.shape[0], 6), 1.0e4, np.float32)])
            out.append({'points': np.pad(p, ((0, 0), (1, 0))).astype(np.float32), 'points_per_frame': [npts], 'frame_id': np.array(['s%d' % i]),
                        'batch_size': 1})
        return out
    batches = batches_for(1.0)
    det = Detector(env, ds, batches, backbone, args.mode, sp_mode, use_graph=not args.no_graph, vfe='DynamicMeanVFE')
    det.settle()
    det.capture()
    out_host = torch.empty((1, 500, 9), dtype=torch.float32).pin_memory()
    state = {'d2h': 0, 'boxes': 0}
    sampler = ClockSampler(env.local)
    sampler.start()
    total_ms = env.timed(det.step_resident, args.steps, args.warmup)
    sampler.stop_flag = True
    e2e_ms = env.timed(lambda i: det.step_e2e(i, out_host, state), args.steps, args.warmup)
    frames = args.steps * env.world
    sb = 2 if sp_mode == 'bf16' else 4
    roof = sparse_conv_roofline(det, args.layer_times, 1, storage_bytes=sb)
    with torch.no_grad():
        od = det.model.forward_device(det.batch_dict(0, det.dev_pts[0]))
    n_vox_full = int(od['voxel_count'].item())
    sweep = []
    if env.rank == 0:
        for sub in (0.04, 0.10, 0.26, 1.0):                # ~50 K .. ~400 K+ voxels by sub-sampling the points
            bs = batches_for(sub, 2)
            d2 = Detector(env, ds, bs, backbone, args.mode, sp_mode, use_graph=False, vfe='DynamicMeanVFE')
            d2.settle()
            r = sparse_conv_roofline(d2, False, 1, storage_bytes=sb)
            with torch.no_grad():
                o2 = d2.model.forward_device(d2.batch_dict(0, d2.dev_pts[0]))
            sweep.append({'points': int(bs[0]['points'].shape[0]), 'voxels': int(o2['voxel_count'].item()), 'sparse_conv_ms': r['ms_per_step'],
                          'achieved_GBps': r['achieved'], 'frac': r['frac'], 'layers': r['layers']})
            del d2
            torch.cuda.empty_cache()
    roof.pop('layers', None)
    line = {'metric': 'Waymo-shape frames/sec', 'value': frames / (total_ms / 1000.0), 'unit': 'frames/s', 'n_gpus': env.world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': total_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'sparse convs: %s; dense BEV/head convs: %s' % (SP_DTYPE[sp_mode], args.mode), 'data': 'synthetic',
            'config': {'workload': 'CenterPoint 5-sweep concat (%d pts, %d voxels), DynamicMeanVFE -> %s, %s, batch 1/GPU'
                                   % (batches[0]['points'].shape[0], n_vox_full, backbone, sp_mode),
                       'sparse_conv_mode': sp_mode, 'dense_conv_mode': args.mode, 'parallelism': 'frames sharded dp%d' % env.world,
                       'l2': 'flushed (256 MiB write) between steps, outside the timed intervals',
                       'launch': 'eager' if args.no_graph else 'CUDA graph replay', 'sweep': sweep},
            'e2e': {'value': frames / (e2e_ms / 1000.0), 'unit': 'frames/s', 'h2d_bytes_per_step': int(det.host_pts[0].numel() * 4),
                    'd2h_bytes_per_step': int(state['d2h'])},
            'gpu_launches': (det.launches_per_step if det.graph is not None else 0) * args.steps, 'clocks': sampler.summary(), 'roofline': roof}
    if env.rank == 0:
        print(json.dumps(line))
    env.done()


# ------------------------------------------------------------------------------------------------------------------
def prm_gflop(qpts):
    """PRM flops per track (SURVEY §8a a17: 17.65 GFLOP at 256 query pts): the query encoder (32->128->128->256 on 200 x qpts points)
    scales with qpts, the rest does not"""
    enc = 2.0 * 200 * (32 * 128 + 128 * 128 + 128 * 256) / 1e9
    return 17.65 + (qpts - 256) * enc


class Refiner:
    """PRM (+ GRM) on a chunk of tracks; inputs of the reference's shapes (SURVEY Appendix B)"""

    def __init__(self, env, mode, tracks, qpts, with_grm=True):
        from detzero_b200 import synthetic
        from detzero_b200.refine import GeometryTransformer, PositionTransformer
        torch = env.torch
        self.env, self.tracks = env, tracks
        cfg = synthetic.prm_cfg()
        cfg.COMPUTE_MODE = mode
        self.prm = PositionTransformer(cfg, 32, 32).eval()
        synthetic.load_seeded(self.prm, 4321)
        self.prm = self.prm.to(env.dev)
        self.grm = None
        if with_grm:
            cfg = synthetic.grm_cfg()
            cfg.COMPUTE_MODE = mode
            self.grm = GeometryTransformer(cfg, 11, 4).eval()
            synthetic.load_seeded(self.grm, 4322)
            self.grm = self.grm.to(env.dev)
        self.host = []
        for i in range(2):
            d = synthetic.prm_inputs(100 + i + 8 * env.rank, B=tracks, qpts=qpts)
            if with_grm:
                d.update(synthetic.grm_inputs(200 + i + 8 * env.rank, B=tracks))
            self.host.append({k: (v.pin_memory() if isinstance(v, torch.Tensor) else v) for k, v in d.items()})
        self.dev_in = [{k: v.to(env.dev) for k, v in h.items()} for h in self.host]
        self.h2d = sum(v.numel() * v.element_size() for v in self.host[0].values())

    def run(self, d):
        torch = self.env.torch
        with torch.no_grad():
            out = self.prm(dict(d))['batch_box_preds']
            out2 = self.grm(dict(d))['batch_box_preds'] if self.grm is not None else None
        return out, out2

    def step_resident(self, i):
        return self.run(self.dev_in[i % 2])

    def step_e2e(self, i, host_out):
        d = {k: v.to(self.env.dev, non_blocking=True) for k, v in self.host[i % 2].items()}
        a, b = self.run(d)
        host_out[0].copy_(a, non_blocking=True)
        if b is not None:
            host_out[1].copy_(b, non_blocking=True)


def run_config4(args):
    """GRM + PRM refiner: 256 tracks x 200 boxes, crops of 256 (reference) and 1024 (BASELINE) points; a step = a chunk of tracks"""
    from detzero_b200 import ops
    env = Env()
    torch = env.torch
    mode = args.mode
    chunk = args.batch or 16
    res = {}
    peaks, which = hbm_peak()
    for qpts in (1024, 256):
        rf = Refiner(env, mode, chunk, qpts)
        host_out = (torch.empty((chunk, 200, 7)).pin_memory(), torch.empty((chunk, 7)).pin_memory())
        rf.step_resident(0)
        ops.reset_launch_count()
        rf.step_resident(1)
        launches = ops.launch_count()
        sampler = ClockSampler(env.local)
        sampler.start()
        ms = env.timed(rf.step_resident, args.steps, args.warmup)
        sampler.stop_flag = True
        e2e_ms = env.timed(lambda i: rf.step_e2e(i, host_out), args.steps, args.warmup)
        tracks = args.steps * chunk * env.world
        tps = tracks / (ms / 1000.0)
        gflop = prm_gflop(qpts) + 5.6
        res[qpts] = dict(tps=tps, ms=ms / args.steps, e2e=tracks / (e2e_ms / 1000.0), launches=launches * args.steps, clocks=sampler.summary(),
                         tflops=tps * gflop / 1e3, h2d=rf.h2d, gflop=gflop)
        del rf
        torch.cuda.empty_cache()
    main = res[1024]
    peak = peaks['bf16_tflops_sustained'] * (0.5 if mode == 'tf32' else 1.0)
    line = {'metric': 'refiner tracks/sec (GRM + PRM)', 'value': main['tps'], 'unit': 'tracks/s', 'n_gpus': env.world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': main['ms'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': '%s products, fp32 accumulate and storage' % mode, 'data': 'synthetic',
            'config': {'workload': 'GRM+PRM refiner, 256 tracks x 200 boxes per sequence in chunks of %d tracks per step, 1024 pts/crop (BASELINE) '
                                   '[also 256 pts/crop = the reference config], 48 memory pts/box, GRM 4096 x 11 memory' % chunk,
                       'mode': mode, 'tracks_per_step': chunk, 'parallelism': 'tracks sharded dp%d' % env.world,
                       'l2': 'flushed (256 MiB write) between steps, outside the timed intervals', 'launch': 'eager',
                       'also': {'256 pts/crop': {'value': res[256]['tps'], 'unit': 'tracks/s', 'ms_per_step': res[256]['ms'],
                                                 'e2e': res[256]['e2e'], 'achieved_TFLOPs': res[256]['tflops']}}},
            'e2e': {'value': main['e2e'], 'unit': 'tracks/s', 'h2d_bytes_per_step': int(main['h2d']), 'd2h_bytes_per_step': chunk * (200 * 7 + 7) * 4},
            'gpu_launches': main['launches'], 'clocks': main['clocks'],
            'roofline': {'bound': 'tensor', 'kernel': 'refiner step (point-MLP encoders + MHA + FFN + heads), %.2f GFLOP/track' % main['gflop'],
                         'achieved': main['tflops'], 'peak': peak, 'peak_source': which + (' (bf16 sustained / 2 for TF32)' if mode == 'tf32' else ''),
                         'unit': 'TFLOP/s', 'frac': main['tflops'] / peak, 'traffic': None}}
    if env.rank == 0:
        print(json.dumps(line))
    env.done()


# ------------------------------------------------------------------------------------------------------------------
def run_config5(args):
    """Full det + refine on a 199-frame sequence: frame i -> rank i % W (reference sampler order), per-sequence NCCL box gather inside
    the timed region, PRM/GRM on 256 tracks sharded track j -> rank j % W, second gather.  One step = one whole sequence; strong scaling."""
    from detzero_b200 import dist as dzdist, synthetic
    env = Env()
    torch, dist = env.torch, env.dist
    F, FB, TRACKS, TCHUNK = 199, 5, 256, 16
    backbone = args.backbone or 'VoxelBackBone8x'
    sp_mode = args.sp_mode or synthetic.DEFAULT_SP_MODE
    mine = dzdist.shard_indices(F, env.rank, env.world)                # frames of this rank (tail wraps like the reference sampler)
    while len(mine) % FB:
        mine.append(mine[0])                                           # last batch padded by wrapping
    nb = len(mine) // FB
    ds, pool = build_inputs(FB, num_batches=4, seed0=0)               # 20 distinct clouds, cycled over the sequence
    gather = dzdist.SequenceGather(F, K=500, device=env.dev)
    slab = (torch.zeros((FB, 500, 9), device=env.dev), torch.zeros((FB,), dtype=torch.int32, device=env.dev))
    det = Detector(env, ds, pool, backbone, args.mode, sp_mode, use_graph=not args.no_graph, slab=slab)
    det.settle()
    det.capture()
    my_tracks = list(range(env.rank, TRACKS, env.world))
    n_chunks = (len(my_tracks) + TCHUNK - 1) // TCHUNK
    rf = Refiner(env, args.mode, TCHUNK, 256)
    rf.step_resident(0)
    refined = torch.zeros((n_chunks * TCHUNK, 200, 7), device=env.dev)
    refined_all = torch.empty((env.world * n_chunks * TCHUNK, 200, 7), device=env.dev) if env.world > 1 else refined
    timing = {}

    def sequence(i):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record()
        for k in range(nb):
            det.step_resident(i * nb + k)                                # graph replay: the NMS result lands in `slab`
            f0, f1 = k * FB, min(gather.f_local, k * FB + FB)
            if f1 > f0:                                                  # -> this rank's rows of the sequence send buffer
                gather.boxes[f0:f1].copy_(slab[0][:f1 - f0], non_blocking=True)
                gather.counts[f0:f1].copy_(slab[1][:f1 - f0], non_blocking=True)
        e[1].record()
        boxes, counts = gather.gather()                                  # ONE collective: all boxes of the sequence on every rank (-> tracker)
        e[2].record()
        for c in range(n_chunks):
            a, _ = rf.step_resident(c)
            refined[c * TCHUNK:(c + 1) * TCHUNK].copy_(a, non_blocking=True)
        if env.world > 1:
            dist.all_gather_into_tensor(refined_all, refined)            # the second gather: refined boxes per track
        e[3].record()
        timing['ev'] = e
        return boxes, counts

    total_ms = env.timed(sequence, args.steps, max(1, args.warmup))
    ev = timing['ev']
    parts = {'detect_ms': ev[0].elapsed_time(ev[1]), 'box_gather_us': 1000 * ev[1].elapsed_time(ev[2]), 'refine_ms': ev[2].elapsed_time(ev[3])}
    sampler = ClockSampler(env.local)
    sampler.start()
    b, c = sequence(0)
    torch.cuda.synchronize()
    sampler.stop_flag = True
    line = {'metric': 'Waymo-shape frames/sec (det + gather + refine, whole sequence)', 'value': F * args.steps / (total_ms / 1000.0), 'unit': 'frames/s',
            'n_gpus': env.world, 'steps': args.steps, 'warmup': max(1, args.warmup), 'ms_per_step': total_ms / args.steps, 'higher_is_better': True,
            'scaling': 'strong', 'vs_baseline': None,
            'dtype': 'sparse convs: %s; dense convs + refiner: %s' % (SP_DTYPE[sp_mode], args.mode), 'data': 'synthetic',
            'config': {'workload': 'Full det+refine: 199-frame Waymo-shape sequence (180K-pt clouds, 20 distinct, cycled) sharded frame i -> rank i %% W in '
                                   'batches of %d, ONE NCCL all-gather of the padded boxes per sequence, then PRM+GRM on %d synthetic tracks (200 boxes, '
                                   '256 pts/crop) sharded by id + the second gather' % (FB, TRACKS),
                       'sparse_conv_mode': sp_mode, 'dense_conv_mode': args.mode, 'parallelism': 'frames i %% %d, tracks j %% %d' % (env.world, env.world),
                       'frames_per_rank': len(mine), 'tracks_per_rank': len(my_tracks), 'last_sequence': parts,
                       'gathered_boxes_total': int(c.sum().item()), 'l2': 'flushed (256 MiB write) between sequences',
                       'launch': 'CUDA graph replay per batch of %d frames; refiner eager' % FB},
            'e2e': None, 'gpu_launches': (det.launches_per_step * nb) * args.steps, 'clocks': sampler.summary(), 'roofline': None}
    if env.rank == 0:
        print(json.dumps(line))
    env.done()


def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)
    return {2: run_config2, 3: run_config3, 4: run_config4, 5: run_config5}[args.config](args)


if __name__ == '__main__':
    main()
