"""Golden vectors for two host-side restatements, from the reference's own code on the inputs of tests/util.py:

    merge_sweeps  DatasetTemplate.merge_sweeps (detection/detzero_det/datasets/dataset.py), its statements executed as they are
    iou_bev       boxes_iou_bev_cpu of utils/detzero_utils/ops/iou3d_nms/src/iou3d_cpu.cpp, compiled by oracle/build_ref.py

    python tests/golden/make_golden_host.py       # needs the reference checkout (ref_import.REF)
"""
import os
import re
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)

from ref_import import REF  # noqa: E402
from oracle import build_ref  # noqa: E402
from tests import util  # noqa: E402


def golden_host():
    out = {}
    src = open(os.path.join(REF, 'detection', 'detzero_det', 'datasets', 'dataset.py')).read()
    m = re.search(r'    @staticmethod\n    def merge_sweeps\(.*?\n        return point_clouds\n', src, re.S)
    ns = {'np': np}
    exec('class _T:\n' + m.group(0), ns)
    infos, pts = util.merge_sweeps_inputs()
    out['merge_sweeps'] = ns['_T'].merge_sweeps(infos[0], infos, pts)
    b = util.iou_boxes()
    iou = torch.zeros(len(b), len(b))
    build_ref.build()
    build_ref.load().boxes_iou_bev_cpu(torch.from_numpy(b), torch.from_numpy(b), iou)
    out['iou_bev'] = iou.numpy()
    np.savez_compressed(os.path.join(HERE, 'host.npz'), **out)
    print('host.npz:', {k: (v.shape, v.dtype) for k, v in out.items()})


if __name__ == '__main__':
    golden_host()
