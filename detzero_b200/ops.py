"""torch-facing wrappers over the C ABI.  torch is plumbing only: device memory, the current stream.

Every function enqueues on ``torch.cuda.current_stream()`` and never synchronises the host."""
import ctypes

import torch

from . import _lib
from ._lib import check, farr, iarr, lib


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


_launches = 0
_trace = None


def _count(n):
    """bookkeeping of how many of OUR kernels were enqueued (bench.py reports it as gpu_launches)"""
    global _launches
    _launches += n


def reset_launch_count():
    global _launches
    _launches = 0


def launch_count():
    return _launches


def enable_spconv_trace(on):
    """bench.py roofline: record a CUDA-event pair + shapes for every sparse-conv launch"""
    global _trace
    _trace = [] if on else None
    return _trace


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError('detzero_b200 ops need CUDA tensors (no CPU fallback); got a %s tensor' % t.device)


def _f32c(t):
    assert t.dtype == torch.float32 and t.is_contiguous(), (t.dtype, t.is_contiguous())
    return t


class GridIndex:
    """bitmap + popcount prefix (+perm) over a (B, D, H, W) lattice; rank order == ascending (b,z,y,x)."""

    def __init__(self, B, dhw, device, with_perm_cap=None):
        self.B, self.dhw = int(B), [int(v) for v in dhw]
        self.words = lib().dz_grid_index_words(self.B, *self.dhw)
        self.bitmap = torch.zeros(self.words, dtype=torch.int32, device=device)
        self.prefix = torch.empty(self.words, dtype=torch.int32, device=device)
        self.perm = torch.empty(with_perm_cap, dtype=torch.int32, device=device) if with_perm_cap else None

    def clear(self):
        self.bitmap.zero_()


_ws_cache = {}


def workspace(nbytes, device, tag='ws'):
    """a grow-only scratch buffer per (device, tag) -- stream-ordered reuse on the current stream"""
    key = (str(device), tag)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


def scan_ws_bytes(words):
    return lib().dz_scan_ws_bytes(words)


def grid_index_from_coords(coords, d_n, cap, B, dhw, with_perm=True):
    _need_cuda(coords)
    gi = GridIndex(B, dhw, coords.device, with_perm_cap=cap if with_perm else None)
    total = torch.zeros(1, dtype=torch.int32, device=coords.device)
    ws = workspace(scan_ws_bytes(gi.words), coords.device, 'rulebook')
    check(lib().dz_grid_index_from_coords(_p(coords), _p(d_n), cap, gi.B, *gi.dhw, _p(gi.bitmap), _p(gi.prefix),
                                          _p(gi.perm), _p(total), _p(ws), ws.numel(), _stream()), 'grid_index_from_coords')
    _count(5)
    return gi


def voxelize_hard(points, xyz_off, c, pc_range, voxel_size, grid_zyx, max_pts, max_voxels, batch_idx,
                  voxels, coords, num, mean, counters, index):
    """one cloud -> rows appended at counters[0]; see include/detzero_b200.h dz_voxelize_hard"""
    _need_cuda(points, voxels)
    _f32c(points)
    n, stride = points.shape
    cap = voxels.shape[0]
    nbytes = lib().dz_voxelize_hard_ws_bytes(n, max_pts, max_voxels, *index.dhw)
    ws = workspace(nbytes, points.device)
    check(lib().dz_voxelize_hard(_p(points), n, stride, xyz_off, c, farr(pc_range), farr(voxel_size), iarr(grid_zyx),
                                 max_pts, max_voxels, batch_idx, _p(voxels), _p(coords), _p(num), _p(mean), cap,
                                 _p(counters), index.B, *index.dhw, _p(index.bitmap), _p(index.prefix), _p(index.perm),
                                 _p(ws), ws.numel(), _stream()), 'voxelize_hard')
    _count(11)


def voxelize_hard_batch(clouds, xyz_off, c, pc_range, voxel_size, grid_zyx, max_pts, max_voxels, voxels, coords, num, mean, counters, index):
    """all frames of a batch in one call (internal streams overlap the frames); see dz_voxelize_hard_batch"""
    _need_cuda(voxels, *clouds)
    B = len(clouds)
    stride = clouds[0].shape[1]
    for p in clouds:
        _f32c(p)
        assert p.shape[1] == stride
    n_max = max(int(p.shape[0]) for p in clouds)
    nbytes = lib().dz_voxelize_hard_batch_ws_bytes(n_max, B, max_pts, max_voxels, *index.dhw)
    ws = workspace(nbytes, voxels.device, 'voxelize_batch')
    ptrs = (ctypes.c_void_p * B)(*[p.data_ptr() if p.shape[0] else None for p in clouds])
    ns = (ctypes.c_int * B)(*[int(p.shape[0]) for p in clouds])
    check(lib().dz_voxelize_hard_batch(ptrs, ns, B, stride, xyz_off, c, farr(pc_range), farr(voxel_size), iarr(grid_zyx), max_pts, max_voxels,
                                       _p(voxels), _p(coords), _p(num), _p(mean), voxels.shape[0], _p(counters), *index.dhw,
                                       _p(index.bitmap), _p(index.prefix), _p(index.perm), _p(ws), ws.numel(), _stream()),
          'voxelize_hard_batch')
    _count(13 * B)


def mean_vfe(voxels, num_i32):
    _need_cuda(voxels, num_i32)
    m, p, c = voxels.shape
    out = torch.empty((m, c), dtype=torch.float32, device=voxels.device)
    check(lib().dz_mean_vfe(_p(_f32c(voxels)), _p(num_i32), m, p, c, _p(out), _stream()), 'mean_vfe')
    _count(1)
    return out


def voxelize_dynamic_mean(points, c, B, pc_range, voxel_size, grid_xyz, cap):
    _need_cuda(points)
    _f32c(points)
    n = points.shape[0]
    assert points.shape[1] == 1 + c
    feats = torch.empty((cap, c), dtype=torch.float32, device=points.device)
    coords = torch.zeros((cap, 4), dtype=torch.int32, device=points.device)
    d_m = torch.zeros(1, dtype=torch.int32, device=points.device)
    nbytes = lib().dz_voxelize_dynamic_ws_bytes(n, cap, B, *[int(g) for g in grid_xyz])
    ws = workspace(nbytes, points.device, 'dyn')
    check(lib().dz_voxelize_dynamic_mean(_p(points), n, c, B, farr(pc_range), farr(voxel_size), iarr(grid_xyz),
                                         _p(feats), _p(coords), cap, _p(d_m), _p(ws), ws.numel(), _stream()),
          'voxelize_dynamic_mean')
    _count(6)
    return feats, coords, d_m


def new_sched_ws(cap, device):
    """scratch a rulebook kernel fills with the mask digests + scanned histogram its tile schedule is built from (one per
    rulebook: the schedule is built later, on another stream)"""
    return torch.empty(int(lib().dz_rulebook_schedule_ws_bytes(cap)), dtype=torch.uint8, device=device)


def rulebook_subm(coords, d_n, cap, index, ksize, layout='k', sched_ws=None, frame_major=False):
    """layout 'k': k-major (K, cap) table (exact-fp32 kernel, parity tests); 'row': row-major (cap, 32) table for the
    tensor-core kernels; 'both': (nbr, tab).  sched_ws (row/both only): also leave the tile-schedule digests there."""
    K = ksize[0] * ksize[1] * ksize[2]
    nbr = torch.empty((K, cap), dtype=torch.int32, device=coords.device) if layout in ('k', 'both') else None
    tab = torch.empty((cap, 32), dtype=torch.int32, device=coords.device) if layout in ('row', 'both') else None
    check(lib().dz_rulebook_subm(_p(coords), _p(d_n), cap, index.B, *index.dhw, iarr(ksize), _p(index.bitmap),
                                 _p(index.prefix), _p(index.perm), _p(nbr), _p(tab), _p(sched_ws), int(bool(frame_major)), _stream()),
          'rulebook_subm')
    _count(1 if sched_ws is None else 2)
    return nbr if layout == 'k' else tab if layout == 'row' else (nbr, tab)


def rulebook_schedule(tab, d_n, sched_ws, B=1, frame_major=False, K=None):
    """tile schedule for the tensor-core conv from the scratch the rulebook call filled: returns `order`
    (cap + ceil(cap/128),) = row order | tile launch order; see dz_rulebook_schedule.  frame_major (same value as in the
    rulebook call): rows sorted by (frame, mask), tiles ordered frame by frame"""
    _need_cuda(tab)
    cap = tab.shape[0]
    tiles = (cap + 127) // 128
    if K is None:                                       # row order | tile order
        order = torch.empty(cap + tiles, dtype=torch.int32, device=tab.device)
        check(lib().dz_rulebook_schedule(_p(tab), cap, _p(d_n), _p(order), _p(sched_ws), sched_ws.numel(), int(B), int(bool(frame_major)),
                                         0, None, _stream()), 'rulebook_schedule')
        _count(1)
        return order
    # K given: also the TILE-major table (tiles, K+1, 128) for the persistent bf16-plane conv; order gets the tile masks appended
    order = torch.empty(cap + 2 * tiles, dtype=torch.int32, device=tab.device)
    tab_tiles = torch.empty((tiles, int(K) + 1, 128), dtype=torch.int32, device=tab.device)
    check(lib().dz_rulebook_schedule(_p(tab), cap, _p(d_n), _p(order), _p(sched_ws), sched_ws.numel(), int(B), int(bool(frame_major)),
                                     int(K), _p(tab_tiles), _stream()), 'rulebook_schedule')
    _count(2)
    return order, tab_tiles


def rulebook_subm_masks(coords, d_n, cap, index, ksize, sched_ws, frame_major=False, perm_walk=True):
    """direct path (bf16-plane layers with a schedule), mask pass of a submanifold rulebook: fills sched_ws as rulebook_subm
    does and writes no table; rulebook_schedule_direct then builds the tile-major table.  perm_walk: visit the rows in lattice
    order through the index's perm (ignored without one)"""
    _need_cuda(coords)
    walk = bool(perm_walk) and index.perm is not None
    check(lib().dz_rulebook_subm_masks(_p(coords), _p(d_n), cap, index.B, *index.dhw, iarr(ksize), _p(index.bitmap), _p(index.prefix),
                                       _p(index.perm), _p(sched_ws), int(bool(frame_major)), int(walk), _stream()), 'rulebook_subm_masks')
    _count(2)


def rulebook_conv_masks(coords, d_n, in_cap, in_index, ksize, stride, pad, out_cap, sched_ws, frame_major=False):
    """direct path, mask pass of a strided-conv rulebook: the output sites, their count and grid index as rulebook_conv, and
    sched_ws filled as rulebook_conv fills it; no table.  Returns (out_coords, d_n_out, out_index, out_dhw)"""
    _need_cuda(coords)
    dev = coords.device
    out_dhw = conv_out_dhw(in_index.dhw, ksize, stride, pad)
    out_index = GridIndex(in_index.B, out_dhw, dev)
    out_coords = torch.empty((out_cap, 4), dtype=torch.int32, device=dev)
    d_n_out = torch.empty(1, dtype=torch.int32, device=dev)
    ws = workspace(scan_ws_bytes(out_index.words), dev, 'rulebook')
    check(lib().dz_rulebook_conv_masks(_p(coords), _p(d_n), in_cap, in_index.B, iarr(in_index.dhw), iarr(ksize), iarr(stride), iarr(pad),
                                       _p(in_index.bitmap), _p(in_index.prefix), _p(in_index.perm), _p(out_coords), _p(d_n_out), out_cap,
                                       _p(out_index.bitmap), _p(out_index.prefix), _p(ws), ws.numel(), _p(sched_ws), int(bool(frame_major)),
                                       _stream()), 'rulebook_conv_masks')
    _count(7)
    return out_coords, d_n_out, out_index, out_dhw


def rulebook_schedule_direct(coords, d_n, cap, in_index, ksize, stride, pad, subm, sched_ws, B=1, frame_major=False):
    """direct path: schedule + tile-major table of a rulebook whose mask pass filled sched_ws.  coords / d_n / cap: the rulebook's
    rows (output sites); in_index: the grid index of the conv's input.  Returns (order, tab_tiles) as rulebook_schedule(K=...)"""
    _need_cuda(coords)
    K = ksize[0] * ksize[1] * ksize[2]
    tiles = (cap + 127) // 128
    order = torch.empty(cap + 2 * tiles, dtype=torch.int32, device=coords.device)
    tab_tiles = torch.empty((tiles, K + 1, 128), dtype=torch.int32, device=coords.device)
    check(lib().dz_rulebook_schedule_direct(_p(coords), cap, _p(d_n), int(B), iarr(in_index.dhw), iarr(ksize), iarr(stride), iarr(pad),
                                            int(bool(subm)), _p(in_index.bitmap), _p(in_index.prefix), _p(in_index.perm), _p(order),
                                            _p(sched_ws), sched_ws.numel(), int(bool(frame_major)), _p(tab_tiles), _stream()),
          'rulebook_schedule_direct')
    _count(2)
    return order, tab_tiles


def tiles_to_rows(tab_tiles, order, d_n, cap):
    """tile-major table + its schedule -> the row-major (cap, 32) table in canonical row order (rows beyond the count: -1,
    mask 0).  For callers that need the row form of a direct-path rulebook; no host read of the count"""
    tiles, K1, _ = tab_tiles.shape
    K = K1 - 1
    dev = tab_tiles.device
    flat = tab_tiles.permute(0, 2, 1).reshape(tiles * 128, K1)
    pos = torch.arange(tiles * 128, device=dev)
    live = (pos < d_n.long()) & (pos < cap)
    dst = torch.where(live, flat[:, K].long(), torch.full_like(pos, cap))       # positions beyond the count go to a spare row
    tab = torch.full((cap + 1, 32), -1, dtype=torch.int32, device=dev)
    tab[dst, :K] = flat[:, :K]
    tab = tab[:cap]
    tab[:, 27] = ((tab[:, :K] >= 0).to(torch.int64) << torch.arange(K, device=dev)[None, :]).sum(1).to(torch.int32)
    tab[:, 28:] = 0
    return tab


def table_to_rows(nbr):
    """k-major (K, cap) table -> the row-major (cap, 32) layout of the tensor-core kernels (host-side helper for callers that
    only hold the k-major form; the rulebook kernels write either layout directly)"""
    K, cap = nbr.shape
    tab = torch.full((cap, 32), -1, dtype=torch.int32, device=nbr.device)
    tab[:, :K] = nbr.t()
    tab[:, 27] = ((nbr >= 0).to(torch.int64) << torch.arange(K, device=nbr.device)[:, None]).sum(0).to(torch.int32)
    tab[:, 28:] = 0
    return tab


def conv_out_dhw(in_dhw, ksize, stride, pad):
    return [(in_dhw[d] + 2 * pad[d] - (ksize[d] - 1) - 1) // stride[d] + 1 for d in range(3)]


def rulebook_conv(coords, d_n, in_cap, in_index, ksize, stride, pad, out_cap, layout='k', sched_ws=None, frame_major=False):
    dev = coords.device
    out_dhw = conv_out_dhw(in_index.dhw, ksize, stride, pad)
    out_index = GridIndex(in_index.B, out_dhw, dev)
    K = ksize[0] * ksize[1] * ksize[2]
    out_coords = torch.empty((out_cap, 4), dtype=torch.int32, device=dev)      # rows >= the count are never read
    d_n_out = torch.empty(1, dtype=torch.int32, device=dev)                    # written by the rank scan
    nbr = torch.empty((K, out_cap), dtype=torch.int32, device=dev) if layout in ('k', 'both') else None
    tab = torch.empty((out_cap, 32), dtype=torch.int32, device=dev) if layout in ('row', 'both') else None
    ws = workspace(scan_ws_bytes(out_index.words), dev, 'rulebook')      # own scratch: rulebooks run on a side stream
    check(lib().dz_rulebook_conv(_p(coords), _p(d_n), in_cap, in_index.B, iarr(in_index.dhw), iarr(ksize), iarr(stride),
                                 iarr(pad), _p(in_index.bitmap), _p(in_index.prefix), _p(in_index.perm), _p(out_coords),
                                 _p(d_n_out), out_cap, _p(out_index.bitmap), _p(out_index.prefix), _p(nbr), _p(tab), _p(ws),
                                 ws.numel(), _p(sched_ws), int(bool(frame_major)), _stream()), 'rulebook_conv')
    _count(6 if sched_ws is None else 7)
    return out_coords, d_n_out, out_index, (nbr if layout == 'k' else tab if layout == 'row' else (nbr, tab)), out_dhw


def pack_spconv_weight(w, mode):
    """spconv-2.x parameter (Cout, KD, KH, KW, Cin) -> kernel layout: DZ_F32 (K, Cin, Cout); DZ_TF32 (Cout, K*cin_pad)
    with cin_pad = 8 for Cin <= 8 (the reduction dim is the concatenation (offset, channel), 128-byte blocks)"""
    cout, cin = w.shape[0], w.shape[-1]
    w = w.detach().reshape(cout, -1, cin).float()
    if mode == _lib.DZ_F32:
        return w.permute(1, 2, 0).contiguous()
    cin_pad = 8 if cin <= 8 else cin
    if cin_pad != cin:
        w = torch.nn.functional.pad(w, (0, cin_pad - cin))
    w = w.reshape(cout, -1).contiguous()
    if mode in _lib.PLANES:                           # bf16 planes: rows [w0 ; w1], w0 = RN_bf16(W), w1 = RN_bf16(W - w0)
        w0 = w.to(torch.bfloat16)
        if _lib.PLANES[mode] == 1:
            return w0.contiguous()
        return torch.cat([w0, (w - w0.float()).to(torch.bfloat16)], dim=0).contiguous()
    if mode == _lib.DZ_TF32X3:                        # (2, Cout, K*cin_pad): hi = RN_tf32(W), lo = RN_tf32(W - hi)
        hi = round_tf32(w)
        return torch.stack([hi, round_tf32(w - hi)]).contiguous()
    return round_tf32(w)


def round_tf32(t):
    """round-to-nearest-even to TF32 precision (10 explicit mantissa bits) so the tensor core's truncating read of the
    fp32 container is exact: removes the systematic toward-zero bias of truncation"""
    i = t.contiguous().view(torch.int32)
    lsb = (i >> 13) & 1
    return ((i + 0xFFF + lsb) & ~0x1FFF).view(torch.float32)


def spconv_fwd(feats, nbr, d_n_out, out_cap, weight_packed, scale, shift, residual, relu, mode=_lib.DZ_F32, out=None,
               d_n_in=None, kshape=None, row_order=None, layout=None, tab_tiles=None):
    """feats (in_cap, cin); weight_packed per pack_spconv_weight; kshape = (K, cin, cout).
    nbr: k-major (K, cap) table for DZ_F32; row-major (cap, 32) table for the tensor-core modes (a k-major table is
    converted on the fly); layout: 'k' | 'row' says which one `nbr` is (None: inferred from the shape, ambiguous only for
    cap == K or cap == 32 -- callers that know pass it); row_order: tile schedule from rulebook_schedule (tensor-core modes).
    nbr may be None for the bf16-plane modes when tab_tiles and row_order are given (direct-path rulebook: no row-major table)"""
    _need_cuda(feats, nbr, weight_packed)
    K, cin, cout = kshape if kshape is not None else weight_packed.shape
    if nbr is None:
        if not (_lib.PLANES.get(mode) and tab_tiles is not None and row_order is not None):
            raise RuntimeError('spconv_fwd without a row-major table needs a bf16-plane mode, tab_tiles and row_order')
        assert row_order.numel() == out_cap + 2 * tab_tiles.shape[0] and tab_tiles.shape[1] == K + 1
    elif layout is None:
        layout = 'row' if (nbr.shape[1] == 32 and nbr.shape[0] != K) else 'k'
    if nbr is not None:
        assert layout in ('k', 'row')
        if mode != _lib.DZ_F32 and layout == 'k':
            nbr = table_to_rows(nbr)
        elif mode == _lib.DZ_F32 and layout == 'row':
            raise RuntimeError('the exact-fp32 kernel needs the k-major (K, cap) table')
        assert nbr.shape[0] == K if mode == _lib.DZ_F32 else nbr.shape[1] == 32
    planes = _lib.PLANES.get(mode, 0)
    if planes:
        cin_pad = 8 if cin <= 8 else cin
        assert feats.dtype == torch.bfloat16 and feats.is_contiguous() and feats.shape[1] == planes * cin_pad, (feats.dtype, feats.shape)
        assert weight_packed.dtype == torch.bfloat16 and tuple(weight_packed.shape) == (planes * cout, K * cin_pad)
        assert residual is None or (residual.dtype == torch.bfloat16 and residual.shape[1] == planes * cout)
        if out is None:
            out = torch.empty((out_cap, planes * cout), dtype=torch.bfloat16, device=feats.device)
    else:
        assert feats.shape[1] == cin
    if out is None:
        out = torch.empty((out_cap, cout), dtype=torch.float32, device=feats.device)
    if _trace is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    if planes:
        check(lib().dz_spconv_fwd_planes(_p(feats), cin, feats.shape[0], _p(nbr), K, out_cap if nbr is None else nbr.shape[0], _p(row_order),
                                         _p(d_n_out), out_cap,
                                         _p(weight_packed), _p(scale), _p(shift), _p(residual), int(relu), _p(out), cout, planes,
                                         _p(tab_tiles if row_order is not None else None), _stream()), 'spconv_fwd_planes')
    else:
        check(lib().dz_spconv_fwd(_p(_f32c(feats)), cin, feats.shape[0], _p(nbr), K, nbr.shape[1] if mode == _lib.DZ_F32 else nbr.shape[0],
                                  _p(row_order), _p(d_n_out), out_cap,
                                  _p(_f32c(weight_packed)), _p(scale), _p(shift), _p(residual), int(relu), _p(out), cout,
                                  mode, _stream()), 'spconv_fwd')
    _count(1)
    if _trace is not None:
        ev1.record()
        torch.cuda.synchronize()
        n_out = min(int(d_n_out.item()), out_cap)
        n_in = min(int(d_n_in.item()), feats.shape[0]) if d_n_in is not None else n_out
        if nbr is None:                                 # direct-path rulebook: the trace records the row-major form (outside the events)
            nbr = tiles_to_rows(tab_tiles, row_order, d_n_out, out_cap)
        _trace.append(dict(start=ev0, end=ev1, K=K, cin=cin, cout=cout, n_in=n_in, n_out=n_out, nbr=nbr, row_order=row_order,
                           residual=residual is not None))
    return out


def rulebook_transpose(nbr, d_n_out, cap_in):
    """k-major (K, cap_out) table -> (K, cap_in) table of the transposed pairs: nbrT[k][j] = o (dgrad / SparseInverseConv3d)"""
    _need_cuda(nbr)
    K, cap_out = nbr.shape
    nbrT = torch.empty((K, int(cap_in)), dtype=torch.int32, device=nbr.device)
    check(lib().dz_rulebook_transpose(_p(nbr), K, cap_out, _p(d_n_out), _p(nbrT), int(cap_in), _stream()), 'rulebook_transpose')
    _count(2)
    return nbrT


def spconv_wgrad(feats, nbr, d_n_out, out_cap, dout):
    """dW (K, cin, cout) = sum over the pairs of in[nbr[k][o]]^T (x) dout[o]; k-major table, exact fp32"""
    _need_cuda(feats, nbr, dout)
    K, cin, cout = nbr.shape[0], feats.shape[1], dout.shape[1]
    dW = torch.empty((K, cin, cout), dtype=torch.float32, device=feats.device)
    check(lib().dz_spconv_wgrad(_p(_f32c(feats)), cin, _p(nbr), K, nbr.shape[1], _p(d_n_out), out_cap, _p(_f32c(dout)), cout, _p(dW),
                                _stream()), 'spconv_wgrad')
    _count(1)
    return dW


def to_planes(x, d_n, planes, c_pad=None):
    """fp32 (rows, c) -> bf16 operand planes (rows, planes * c_pad): row = [p0 | p1], p0 = RN_bf16(x), p1 = RN_bf16(x - p0)
    (channels zero-padded to c_pad); rows >= *d_n are left untouched"""
    _need_cuda(x)
    rows, c = x.shape
    c_pad = c if c_pad is None else int(c_pad)
    out = torch.empty((rows, planes * c_pad), dtype=torch.bfloat16, device=x.device)
    if rows:
        check(lib().dz_to_planes(_p(_f32c(x)), _p(d_n), rows, c, c_pad, planes, _p(out), _stream()), 'to_planes')
        _count(1)
    return out


def from_planes(x, d_n, planes):
    """bf16 operand planes (rows, planes * c) -> fp32 (rows, c) = p0 (+ p1)"""
    _need_cuda(x)
    rows, c = x.shape[0], x.shape[1] // planes
    out = torch.empty((rows, c), dtype=torch.float32, device=x.device)
    if rows:
        assert x.dtype == torch.bfloat16 and x.is_contiguous()
        check(lib().dz_from_planes(_p(x), _p(d_n), rows, c, planes, _p(out), _stream()), 'from_planes')
        _count(1)
    return out


def sparse_to_bev(feats, coords, d_n, cap, B, D, H, W, out=None, planes=0):
    """planes = 0: fp32 (rows, c) features; 1 / 2: bf16 operand planes (rows, planes * c) -- always an fp32 NHWC map"""
    c = feats.shape[1] // max(planes, 1)
    if out is None:
        out = torch.zeros((B, H, W, c * D), dtype=torch.float32, device=feats.device)
    else:
        out.zero_()
    if planes:
        assert feats.dtype == torch.bfloat16 and feats.is_contiguous()
        check(lib().dz_sparse_to_bev_planes(_p(feats), _p(coords), _p(d_n), cap, c, planes, B, D, H, W, _p(out), _stream()),
              'sparse_to_bev_planes')
    else:
        check(lib().dz_sparse_to_bev(_p(_f32c(feats)), _p(coords), _p(d_n), cap, c, B, D, H, W, _p(out), _stream()),
              'sparse_to_bev')
    _count(1)
    return out


def conv2d(x, weight_packed, kshape, stride, pad, scale, shift, relu, out=None, out_coff=0, mode=_lib.DZ_F32):
    """x (B,H,W,cin) NHWC; kshape = (KH, KW, cin, cout); weight_packed layout depends on mode:
    DZ_F32 -> (KH,KW,cin,cout) ; DZ_TF32 -> (cout,KH,KW,cin)   (see pack_conv_weight)"""
    _need_cuda(x, weight_packed)
    B, H, W, cstride = x.shape
    KH, KW, cin, cout = kshape
    assert cin == cstride and weight_packed.numel() == KH * KW * cin * cout
    Ho = (H + 2 * pad - KH) // stride + 1
    Wo = (W + 2 * pad - KW) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, cout), dtype=torch.float32, device=x.device)
    assert out.shape[:3] == (B, Ho, Wo)
    check(lib().dz_conv2d_fwd(_p(_f32c(x)), B, H, W, cin, cstride, _p(_f32c(weight_packed)), KH, KW, stride, pad,
                              _p(scale), _p(shift), int(relu), _p(out), Ho, Wo, cout, out_coff, out.shape[3], mode,
                              _stream()), 'conv2d_fwd')
    _count(1)
    return out


def deconv2d(x, weight_packed, kshape, scale, shift, relu, out=None, out_coff=0, mode=_lib.DZ_F32):
    """ConvTranspose2d with kernel == stride; kshape = (s, cin, cout); weight layout DZ_F32 -> (s,s,cin,cout),
    DZ_TF32 -> (s,s,cout,cin)"""
    B, H, W, cin = x.shape
    s, cin2, cout = kshape
    assert cin2 == cin and weight_packed.numel() == s * s * cin * cout
    if out is None:
        out = torch.empty((B, H * s, W * s, cout), dtype=torch.float32, device=x.device)
    check(lib().dz_deconv2d_fwd(_p(_f32c(x)), B, H, W, cin, _p(_f32c(weight_packed)), s, _p(scale), _p(shift),
                                int(relu), _p(out), cout, out_coff, out.shape[3], mode, _stream()), 'deconv2d_fwd')
    _count(s * s)
    return out


def pack_conv_weight(w_oihw, mode):
    """torch (Cout,Cin,KH,KW) -> kernel layout for `mode`"""
    if mode == _lib.DZ_F32:
        return w_oihw.detach().permute(2, 3, 1, 0).contiguous().float()       # (KH,KW,Cin,Cout)
    return round_tf32(w_oihw.detach().permute(0, 2, 3, 1).contiguous().float())   # (Cout,KH,KW,Cin): K-major rows for TMA


def pack_deconv_weight(w_iohw, mode):
    """torch ConvTranspose2d (Cin,Cout,s,s) -> kernel layout for `mode`"""
    if mode == _lib.DZ_F32:
        return w_iohw.detach().permute(2, 3, 0, 1).contiguous().float()       # (s,s,Cin,Cout)
    return round_tf32(w_iohw.detach().permute(2, 3, 1, 0).contiguous().float())   # (s,s,Cout,Cin)


def centerhead_decode(head, ch_layout, num_class, K, pc_range, voxel_size, fmap_stride, post_limit, score_thresh,
                      use_iou):
    """head (B,H,W,ch) NHWC; ch_layout dict of channel offsets: center, center_z, dim, rot, iou, hm"""
    B, H, W, ch = head.shape
    dev = head.device
    boxes = torch.zeros((B, K, 7), dtype=torch.float32, device=dev)
    scores = torch.zeros((B, K), dtype=torch.float32, device=dev)
    labels = torch.zeros((B, K), dtype=torch.int32, device=dev)
    d_n = torch.zeros(B, dtype=torch.int32, device=dev)
    nbytes = lib().dz_centerhead_decode_ws_bytes(B, H, W, num_class, K)
    ws = workspace(nbytes, dev, 'decode')
    check(lib().dz_centerhead_decode(_p(_f32c(head)), B, H, W, ch, ch_layout['center'], ch_layout['center_z'],
                                     ch_layout['dim'], ch_layout['rot'], ch_layout.get('iou', 0), ch_layout['hm'],
                                     num_class, K, farr(pc_range), farr(voxel_size), int(fmap_stride), farr(post_limit),
                                     float(score_thresh), int(use_iou), _p(boxes), _p(scores), _p(labels), _p(d_n),
                                     _p(ws), ws.numel(), _stream()), 'centerhead_decode')
    _count(2)
    return boxes, scores, labels, d_n


def nms_bev(boxes, scores, labels, d_n, thresh, post_max, label_offset=1, out=None, d_out_n=None):
    """boxes (B,cap,7) in descending score order; returns out (B,post_max,9), d_out_n (B).  out / d_out_n may be views into a
    caller-owned buffer -- e.g. the send buffer of the per-sequence box gather (dist.SequenceGather), so the NMS output needs
    no staging copy before the collective"""
    B, cap, _ = boxes.shape
    dev = boxes.device
    if out is None:
        out = torch.empty((B, post_max, 9), dtype=torch.float32, device=dev)
    else:
        assert out.shape == (B, post_max, 9) and out.dtype == torch.float32 and out.is_contiguous()
    if d_out_n is None:
        d_out_n = torch.zeros(B, dtype=torch.int32, device=dev)
    else:
        assert d_out_n.shape == (B,) and d_out_n.dtype == torch.int32 and d_out_n.is_contiguous()
        d_out_n.zero_()
    ws = workspace(lib().dz_nms_bev_ws_bytes(B, cap), dev, 'nms')
    check(lib().dz_nms_bev(_p(_f32c(boxes)), _p(_f32c(scores)), _p(labels), _p(d_n), B, cap, float(thresh), post_max,
                           label_offset, _p(out), _p(d_out_n), _p(ws), ws.numel(), _stream()), 'nms_bev')
    _count(2)
    return out, d_out_n


def boxes_iou_bev(a, b):
    _need_cuda(a, b)
    a = a[:, :7].contiguous().float()
    b = b[:, :7].contiguous().float()
    out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.float32, device=a.device)
    check(lib().dz_boxes_iou_bev(_p(a), a.shape[0], _p(b), b.shape[0], _p(out), _stream()), 'boxes_iou_bev')
    _count(1)
    return out


def linear(x, w, scale=None, shift=None, relu=False, out=None, mode=_lib.DZ_F32):
    """y = act((x @ w.T) * scale + shift); x (M,K), w (N,K)"""
    _need_cuda(x, w)
    M, K = x.shape
    N = w.shape[0]
    assert w.shape[1] == K
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=x.device)
    ldy = out.stride(0)
    check(lib().dz_linear_fwd(_p(_f32c(x)), M, K, _p(_f32c(w)), N, _p(scale), _p(shift), int(relu), _p(out), ldy, mode,
                              _stream()), 'linear_fwd')
    _count(1)
    return out


def linear_grouped(x, w, gshift, gsize, scale=None, shift=None, relu=False, mode=_lib.DZ_F32):
    """y[m] = act((x[m] @ w.T) * scale + shift + gshift[m // gsize]); gshift (M // gsize, N) -- the fused form of
    Linear(cat([global.expand, x])) (see dz_linear_fwd_grouped)"""
    _need_cuda(x, w, gshift)
    M, K = x.shape
    N = w.shape[0]
    assert w.shape[1] == K and gshift.shape == (M // gsize, N) and M % gsize == 0
    out = torch.empty((M, N), dtype=torch.float32, device=x.device)
    check(lib().dz_linear_fwd_grouped(_p(_f32c(x)), M, K, _p(_f32c(w)), N, _p(scale), _p(shift), _p(_f32c(gshift)), int(gsize), int(relu),
                                      _p(out), N, mode, _stream()), 'linear_fwd_grouped')
    _count(1)
    return out


def linear_max(x, w, group, scale=None, shift=None, relu=False, mode=_lib.DZ_TF32):
    """max over groups of `group` rows of act((x @ w.T) * scale + shift) -> (M // group, N); see dz_linear_max_fwd"""
    _need_cuda(x, w)
    M, K = x.shape
    N = w.shape[0]
    y = torch.empty((M // group, N), dtype=torch.float32, device=x.device)
    check(lib().dz_linear_max_fwd(_p(_f32c(x)), M, K, _p(_f32c(w)), N, _p(scale), _p(shift), int(relu), int(group), _p(y), mode, _stream()),
          'linear_max_fwd')
    _count(2)
    return y


def group_max(x, G, group):
    C = x.shape[1]
    assert x.shape[0] == G * group
    y = torch.empty((G, C), dtype=torch.float32, device=x.device)
    check(lib().dz_group_max(_p(_f32c(x)), G, group, C, _p(y), _stream()), 'group_max')
    _count(1)
    return y


def attention(q, k, v, key_padding_mask, H, mode=_lib.DZ_F32):
    """q (B,Pq,E) pre-scaled, k/v (B,Pk,E) -- may be strided views with contiguous last dim; mask (B,Pk) uint8"""
    _need_cuda(q, k, v)
    B, Pq, E = q.shape
    Pk = k.shape[1]
    dh = E // H
    for t in (q, k, v):
        assert t.stride(2) == 1 and t.stride(0) == t.shape[1] * t.stride(1)
    out = torch.empty((B, Pq, E), dtype=torch.float32, device=q.device)
    check(lib().dz_attention_fwd(_p(q), q.stride(1), _p(k), k.stride(1), _p(v), v.stride(1), _p(key_padding_mask), B, Pq,
                                 Pk, H, dh, _p(out), E, mode, _stream()), 'attention_fwd')
    _count(1)
    return out


def layernorm_residual(x, r, gamma, beta, eps=1e-5):
    M, C = x.shape
    y = torch.empty_like(x)
    check(lib().dz_layernorm_residual(_p(_f32c(x)), _p(r), _p(gamma), _p(beta), float(eps), M, C, _p(y), _stream()),
          'layernorm_residual')
    _count(1)
    return y


def add(a, b):
    assert a.shape == b.shape and a.is_contiguous() and b.is_contiguous()
    out = torch.empty_like(a)
    check(lib().dz_add(_p(a), _p(b), a.numel(), _p(out), _stream()), 'add')
    _count(1)
    return out
