"""Where the rulebook chain's time goes in the bench workload (config 2: CenterPoint 1-sweep, batch 8, sparse convs in the
default bf16-plane mode).

1. torch.profiler (CUDA activities) over a few CUDA-graph replays of the step: kernel time per stream, every rulebook kernel in
   launch order (occurrence i of a name = the i-th rulebook of that kind in the step), and how long the launching (main) stream
   has no kernel running while its step is in flight -- mostly waiting on the side-stream events of the rulebooks.
2. The rulebook of every sparse conv of the step rebuilt in isolation (CUDA events, median of --reps), table path
   (rulebook kernel writing the row-major table -> schedule -> transpose) against the direct path (mask pass -> scatter ->
   tile pass), and the submanifold mask pass with and without the lattice-order walk.

    python tools/rulebook_timeline.py --out profiles/rulebook_timeline.json [--table] [--timeline-only]
    (--table: the step on the table path; --timeline-only: part 1 only)

Prints a short summary; the JSON has the GPU name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
from detzero_b200 import ops, synthetic  # noqa: E402
from detzero_b200.spconv import pytorch as sp  # noqa: E402

RULEBOOK_KERNELS = ('k_subm_nbr', 'k_conv_nbr', 'k_subm_mask', 'k_conv_mask', 'k_sched_scatter', 'k_sched_tiles', 'k_tiles_direct',
                    'k_conv_mark', 'k_index_to_coords', 'k_clamp_count')


def gpu_info():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = r.stdout.strip()
    except Exception as e:                        # the numbers stay valid; the record says why the limit is missing
        info['power_limit_and_max_sm_clock'] = 'unavailable: %s' % e
    return info


def short(name):
    return name.split('(')[0].split('<')[0].replace('void ', '').strip()


def timeline(det, replays):
    for i in range(3):
        det.step_resident(i)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for i in range(replays):
            det.env.flush.zero_()
            torch.cuda._sleep(1000)                 # marker kernel: the step starts after it
            det.step_resident(i)
            torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, 'trace.json')
        prof.export_chrome_trace(path)
        ev = json.load(open(path))['traceEvents']
    kern = [e for e in ev if e.get('cat') == 'kernel' and 'dur' in e]
    kern.sort(key=lambda e: e['ts'])
    marker = [e for e in kern if 'spin_kernel' in e['name']]
    # replay windows: the kernels between two marker kernels (the L2 flush runs before the marker)
    cuts = [e['ts'] + e['dur'] for e in marker] + [float('inf')]
    kern = [e for e in kern if 'spin_kernel' not in e['name'] and not ('FillFunctor' in e['name'] and e['dur'] > 30)]
    steps = [[] for _ in range(len(cuts) - 1)]
    for e in kern:
        for j in range(len(cuts) - 1):
            if cuts[j] <= e['ts'] < cuts[j + 1]:
                steps[j].append(e)
                break
    steps = [s for s in steps if s]
    per_stream, rb_names, idle, wall = {}, {}, [], []
    for s in steps:
        by = {}
        for e in s:
            by.setdefault(e['args'].get('stream', -1), []).append(e)
        main = min(by, key=lambda k: min(e['ts'] for e in by[k]))      # the stream the step starts on
        t0, t1 = min(e['ts'] for e in s), max(e['ts'] + e['dur'] for e in s)
        wall.append(t1 - t0)
        busy, end = 0.0, t0
        for e in sorted(by[main], key=lambda e: e['ts']):
            a, b = max(e['ts'], end), e['ts'] + e['dur']
            if b > a:
                busy += b - a
            end = max(end, b)
        idle.append((t1 - t0) - busy)
        for k, es in by.items():
            key = 'main' if k == main else str(k)
            per_stream[key] = per_stream.get(key, 0.0) + sum(e['dur'] for e in es) / len(steps)
        occ = {}
        for e in s:
            n = short(e['name'])
            if n in RULEBOOK_KERNELS or 'scan' in n.lower() or 'grid_index' in n.lower():
                j = occ.get(n, 0)
                occ[n] = j + 1
                lst = rb_names.setdefault(n, [])
                if len(lst) <= j:
                    lst.append(0.0)
                lst[j] += e['dur'] / len(steps)
    rb_total = sum(sum(v) for v in rb_names.values())
    return {'replays': len(steps), 'step_wall_us': sum(wall) / max(len(wall), 1),
            'main_stream_idle_us': sum(idle) / max(len(idle), 1),
            'kernel_us_per_stream': {k: round(v, 1) for k, v in sorted(per_stream.items(), key=lambda kv: -kv[1])},
            'rulebook_kernel_us_total': round(rb_total, 1),
            'rulebook_kernels_us_by_occurrence': {k: [round(x, 1) for x in v] for k, v in sorted(rb_names.items())}}


def median_ms(fn, reps):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def isolated(det, reps):
    """rebuild each sparse conv's rulebook of one eager step in isolation, both paths"""
    seen, calls = set(), []
    orig = sp._SparseConv._rule

    def spy(self, x, schedule=True):
        if self.indice_key not in seen and self._wants_schedule():
            seen.add(self.indice_key)
            calls.append((self, x))
        return orig(self, x, schedule)
    sp._SparseConv._rule = spy
    try:
        with torch.no_grad():
            det.model.forward_device(det.batch_dict(0, det.dev_pts[0]))
        torch.cuda.synchronize()
    finally:
        sp._SparseConv._rule = orig
    out = []
    for conv, x in calls:
        ks, B, K = conv.kernel_size, x.batch_size, conv.kshape[0]
        idx, cnt, cap, gi = x._idx, x._count, x._cap, x.grid_index()
        rec = {'key': conv.indice_key, 'subm': conv.subm, 'rows_in': int(cnt.item())}
        if conv.subm:
            sws = ops.new_sched_ws(cap, idx.device)
            box = {}

            def table1():
                box['tab'] = ops.rulebook_subm(idx, cnt, cap, gi, ks, layout='row', sched_ws=sws)

            def table2():
                ops.rulebook_schedule(box['tab'], cnt, sws, B, False, K=K)

            def masks(walk):
                return lambda: ops.rulebook_subm_masks(idx, cnt, cap, gi, ks, sws, perm_walk=walk)

            def direct2():
                ops.rulebook_schedule_direct(idx, cnt, cap, gi, ks, [1, 1, 1], [0, 0, 0], True, sws, B)
            # the schedule consumes what the rulebook pass left in sched_ws, so it is timed as (pass + schedule) - pass
            rec['table_pass_ms'] = median_ms(table1, reps)
            rec['table_total_ms'] = median_ms(lambda: (table1(), table2()), reps)
            rec['mask_pass_ms'] = median_ms(masks(True), reps)
            rec['mask_pass_row_order_ms'] = median_ms(masks(False), reps)
            rec['direct_total_ms'] = median_ms(lambda: (masks(True)(), direct2()), reps)
        else:
            out_cap = conv._rule(x, schedule=False).out_cap
            sws = ops.new_sched_ws(out_cap, idx.device)
            box = {}

            def table1():
                box['r'] = ops.rulebook_conv(idx, cnt, cap, gi, ks, conv.stride, conv.padding, out_cap, layout='row', sched_ws=sws)

            def table2():
                ops.rulebook_schedule(box['r'][3], box['r'][1], sws, B, False, K=K)

            def mask1():
                box['m'] = ops.rulebook_conv_masks(idx, cnt, cap, gi, ks, conv.stride, conv.padding, out_cap, sws)

            def direct2():
                ops.rulebook_schedule_direct(box['m'][0], box['m'][1], out_cap, gi, ks, conv.stride, conv.padding, False, sws, B)
            rec['table_pass_ms'] = median_ms(table1, reps)
            rec['table_total_ms'] = median_ms(lambda: (table1(), table2()), reps)
            rec['mask_pass_ms'] = median_ms(mask1, reps)
            rec['direct_total_ms'] = median_ms(lambda: (mask1(), direct2()), reps)
            rec['rows_out'] = int(box['m'][1].item())
        rec['table_schedule_ms'] = rec['table_total_ms'] - rec['table_pass_ms']
        rec['direct_schedule_ms'] = rec['direct_total_ms'] - rec['mask_pass_ms']
        out.append({k: (round(v, 4) if isinstance(v, float) else v) for k, v in rec.items()})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--replays', type=int, default=5)
    ap.add_argument('--reps', type=int, default=15)
    ap.add_argument('--table', action='store_true', help='run the step on the table path (DIRECT_TILES off)')
    ap.add_argument('--timeline-only', action='store_true', help='skip the isolated rebuilds')
    ap.add_argument('--backbone', default='VoxelBackBone8x')
    ap.add_argument('--batch', type=int, default=8)
    a = ap.parse_args()
    sp._SparseConv.DIRECT_TILES = not a.table
    env = bench.Env()
    ds, batches = bench.build_inputs(a.batch)
    det = bench.Detector(env, ds, batches, a.backbone, 'tf32', synthetic.DEFAULT_SP_MODE)
    det.settle()
    det.capture()
    res = {'gpu': gpu_info(), 'workload': bench.workload_name(a.backbone, a.batch), 'sparse_conv_mode': synthetic.DEFAULT_SP_MODE,
           'rulebook_path': 'table' if a.table else 'direct', 'timeline': timeline(det, a.replays)}
    sp._SparseConv.DIRECT_TILES = True
    res['isolated'] = [] if a.timeline_only else isolated(det, a.reps)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    t = res['timeline']
    print('%s | %s path: step %.0f us, main stream idle %.0f us, rulebook kernels %.0f us, per stream %s' % (
        res['gpu'], res['rulebook_path'], t['step_wall_us'], t['main_stream_idle_us'], t['rulebook_kernel_us_total'], t['kernel_us_per_stream']))
    for r in res['isolated']:
        print('  %-10s subm=%d  table %.3f ms  direct %.3f ms  %s' % (r['key'], r['subm'], r['table_total_ms'], r['direct_total_ms'],
                                                                    {k: v for k, v in r.items() if k.endswith('_ms')}))


if __name__ == '__main__':
    main()
