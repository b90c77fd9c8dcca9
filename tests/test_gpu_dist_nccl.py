"""NCCL world-size-2 test of the per-sequence box gather ON GPUs (needs >= 2 devices, skipped with one): the detector's
NMS writes into dist.SequenceGather's send buffer, ONE ncclAllGather, frame order = the reference's merge_results_dist
(utils/detzero_utils/common_utils.py:135-138: parts[r][k] -> frame k*W + r, truncated to the sequence length)."""
import json
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

WORKER = r'''
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(sys.argv[0]))))
sys.path.insert(0, sys.argv[6])
import numpy as np, torch, torch.distributed as dist
rank, world, port, num_frames, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], int(sys.argv[4]), sys.argv[5]
os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=port, RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
torch.cuda.set_device(rank)
dev = torch.device('cuda', rank)
dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
from detzero_b200 import dist as dz, ops
idx = dz.shard_indices(num_frames, rank, world)
K, cap = 500, 512
sg = dz.SequenceGather(num_frames, K=K, device=dev)
g = np.random.default_rng(0)
want_counts = []
for j0 in range(0, len(idx), 2):                     # "batches" of 2 frames: the rotated NMS writes straight into the send buffer
    fr = idx[j0:j0 + 2]
    B = len(fr)
    boxes = np.zeros((B, cap, 7), np.float32); scores = np.zeros((B, cap), np.float32); n = np.zeros(B, np.int32)
    for b, f in enumerate(fr):
        m = 5 + f % 7                                # well separated boxes: NMS keeps all m of them
        boxes[b, :m, 0] = 10.0 * np.arange(m); boxes[b, :m, 1] = f; boxes[b, :m, 3:6] = 1.0
        scores[b, :m] = np.linspace(0.9, 0.5, m); n[b] = m
    bs, cs = sg.slot(j0, j0 + B)
    ops.nms_bev(torch.from_numpy(boxes).to(dev), torch.from_numpy(scores).to(dev), torch.zeros((B, cap), dtype=torch.int32, device=dev),
                torch.from_numpy(n).to(dev), 0.7, K, label_offset=1, out=bs, d_out_n=cs)
b_all, c_all = sg.gather()
b2, c2 = dz.gather_sequence_boxes(sg.boxes, sg.counts, num_frames)      # the two-collective form must agree
torch.cuda.synchronize()
assert torch.equal(b_all, b2) and torch.equal(c_all, c2)
if rank == 0:
    json.dump({'tags': b_all[:, 0, 1].tolist(), 'counts': c_all.tolist(), 'second_x': b_all[:, 1, 0].tolist()}, open(out, 'w'))
dist.barrier()
dist.destroy_process_group()
'''


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_sequence_gather_nccl_world2(cuda, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    w = tmp_path / 'worker.py'
    w.write_text(WORKER)
    port, num_frames, out = _free_port(), 7, str(tmp_path / 'out.json')
    procs = [subprocess.Popen([sys.executable, str(w), str(r), '2', str(port), str(num_frames), out, os.path.dirname(HERE)]) for r in range(2)]
    for p in procs:
        assert p.wait(timeout=300) == 0
    res = json.load(open(out))
    assert res['tags'] == [float(f) for f in range(num_frames)]            # frame order restored, truncated to the sequence length
    assert res['counts'] == [5 + f % 7 for f in range(num_frames)]
    assert res['second_x'] == [10.0] * num_frames
