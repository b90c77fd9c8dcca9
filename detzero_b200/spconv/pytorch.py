"""``spconv.pytorch``-shaped API on top of libdetzero_b200 (sm_100a).

Mirrors exactly the surface the reference touches (SURVEY.md §8b): ``SparseConvTensor(features=, indices=,
spatial_shape=, batch_size=)`` with ``.features .indices .spatial_shape .batch_size .indice_dict
.replace_feature() .dense()``; ``SubMConv3d`` / ``SparseConv3d(in, out, k, stride=, padding=, bias=, indice_key=)``
with spconv-2.x weight layout ``(Cout, KD, KH, KW, Cin)`` (state-dict compatible, SURVEY Appendix A.3);
``SparseSequential``; ``SparseModule``; ``SparseInverseConv3d`` (never constructed by the shipped configs).
Reference call sites: detection/detzero_det/models/centerpoint_modules/backbone3d.py:68-73,93-100,135-195.

B200-native differences (behaviour-preserving):
  * tensors carry a *capacity* and a device-side row count, so a whole backbone runs without a host sync;
    ``.features`` / ``.indices`` slice to the true row count lazily (one D2H only if the caller asks)
  * the rulebook is a neighbour table built from an L2-resident grid index (no hash table, no sort);
    strided-conv output sites are emitted sorted by (b,z,y,x) (spconv's order is implementation-defined)
  * in eval mode ``SparseSequential`` fuses conv + BatchNorm1d + ReLU (+ residual) into one launch.
"""
import os

import torch
import torch.nn as nn

from .. import _lib, ops


def _triple(v):
    if isinstance(v, (list, tuple)):
        assert len(v) == 3
        return [int(x) for x in v]
    return [int(v)] * 3


class SparseConvTensor:
    def __init__(self, features, indices, spatial_shape, batch_size, grid=None, voxel_num=None, indice_dict=None,
                 benchmark=False, *, count=None, n_host=None, index=None):
        if not features.is_cuda:
            raise RuntimeError('detzero_b200.spconv needs CUDA tensors (there is no CPU fallback)')
        self._feat = features
        self._idx = indices if indices.dtype == torch.int32 else indices.int()
        if not self._idx.is_contiguous():
            self._idx = self._idx.contiguous()
        self.spatial_shape = [int(s) for s in spatial_shape]
        self.batch_size = int(batch_size)
        self.indice_dict = indice_dict if indice_dict is not None else {}
        self._cap = int(features.shape[0])
        if count is None:
            n_host = self._cap
            count = torch.full((1,), self._cap, dtype=torch.int32, device=features.device)
        self._count = count
        self._n = n_host
        self._index = index
        self._planes = 0            # 0: fp32 (rows, C) features; 1 / 2: bf16 operand planes (rows, planes*C), csrc/spconv_bf16.cu

    # ---- spconv-visible surface ---------------------------------------------------------------------------
    def num(self):
        """true number of rows (host int); one device->host read the first time if it is not known yet"""
        if self._n is None:
            self.set_num(int(self._count.item()))
        return self._n

    def set_num(self, n):
        """record the true row count (read back by the caller); feeds the producing layer's capacity hint"""
        prod = getattr(self, '_producer', None)
        if prod is not None:
            prod._cap_hint = max(n, int(getattr(prod, '_cap_hint', 0) or 0))
        if n > self._cap:
            raise RuntimeError('sparse tensor overflow: %d sites > capacity %d (capacity hint raised; re-run the frame)' % (n, self._cap))
        self._n = n

    @property
    def features(self):
        """(N, C) float32 features (spconv contract).  A tensor produced by a bf16-plane layer is converted on demand."""
        if self._planes:
            return ops.from_planes(self._feat, self._count, self._planes)[:self.num()]
        return self._feat[:self.num()]

    @features.setter
    def features(self, v):          # spconv 1.x style assignment (backbone3d.py:59-62 else-branch)
        self._feat = v

    @property
    def indices(self):
        return self._idx[:self.num()]

    def replace_feature(self, new_features):
        t = SparseConvTensor.__new__(SparseConvTensor)
        t.__dict__.update(self.__dict__)
        if new_features.shape[0] != self._cap:               # caller sliced to the true size
            t._cap = int(new_features.shape[0])
            t._idx = self._idx[:t._cap]
            t._n = t._cap
            t._count = torch.full((1,), t._cap, dtype=torch.int32, device=new_features.device)
        t._feat = new_features
        t._planes = 0
        return t

    def dense(self, channels_first=True):
        """(B, C, D, H, W) like spconv's .dense() (height_compression.py:21)"""
        D, H, W = self.spatial_shape
        c = self._feat.shape[1] // max(self._planes, 1)
        nhwc = ops.sparse_to_bev(self._feat, self._idx, self._count, self._cap, self.batch_size, D, H, W, planes=self._planes)  # (B,H,W,c*D)
        x = nhwc.view(self.batch_size, H, W, c, D)
        return x.permute(0, 3, 4, 1, 2).contiguous() if channels_first else x

    # ---- internal ------------------------------------------------------------------------------------------
    def grid_index(self):
        if self._index is None:
            self._index = ops.grid_index_from_coords(self._idx, self._count, self._cap, self.batch_size,
                                                     self.spatial_shape, with_perm=True)
        return self._index

    def _like(self, feat, planes=0):
        t = SparseConvTensor.__new__(SparseConvTensor)
        t.__dict__.update(self.__dict__)
        t._feat = feat
        t._planes = planes
        return t

    def _as_planes(self, planes, c_pad):
        """this tensor's features as bf16 operand planes (converted once per tensor if they are fp32)"""
        if self._planes == planes:
            return self._feat
        if self._planes:
            raise RuntimeError('a %d-plane tensor cannot feed a %d-plane layer: use one COMPUTE_MODE per backbone' % (self._planes, planes))
        key = ('_as_planes', planes, c_pad)
        if self.__dict__.get('_planes_cache', (None,))[0] != key:
            self._planes_cache = (key, ops.to_planes(self._feat, self._count, planes, c_pad))
        return self._planes_cache[1]


class SparseModule(nn.Module):
    pass


def _tensor_state(ts):
    """identity + in-place version of every involved tensor (load_state_dict bumps ``_version``; ``.to()`` swaps data_ptr)"""
    return tuple((t._version, t.data_ptr(), t.device) for t in ts)


def fold_bn(bn, conv_bias, device=None):
    """eval-mode BatchNorm folded to (scale, shift): y = conv*scale + shift.  Cached ON THE MODULE (never in a global keyed
    by id(): ids and allocator addresses are recycled after a model is freed); refreshed when any involved tensor changes."""
    ts = [t for t in (bn.weight, bn.bias, bn.running_mean, bn.running_var, conv_bias) if t is not None]
    ver = _tensor_state(ts)
    hit = bn.__dict__.get('_dz_fold')
    if hit is not None and hit[0] == ver:
        return hit[1], hit[2]
    with torch.no_grad():
        scale = torch.rsqrt(bn.running_var.detach().float() + bn.eps)
        if bn.affine:
            scale = scale * bn.weight.detach().float()
        shift = -bn.running_mean.detach().float() * scale
        if bn.affine:
            shift = shift + bn.bias.detach().float()
        if conv_bias is not None:
            shift = shift + conv_bias.detach().float() * scale
        scale, shift = scale.contiguous(), shift.contiguous()
    bn.__dict__['_dz_fold'] = (ver, scale, shift)
    return scale, shift


class _SparseConvFn(torch.autograd.Function):
    """training path (SURVEY.md §8f row 1): exact-fp32 forward on the k-major table; backward = dgrad (the forward kernel on the
    transposed table with W^T) + wgrad (gathered A^T B per offset) + bias grad.  Tensors are exact-size here (count == capacity)."""

    @staticmethod
    def forward(ctx, feats, weight, bias, nbr, d_n_out, out_cap, d_n_in, kshape):
        wp = ops.pack_spconv_weight(weight, _lib.DZ_F32)                       # (K, cin, cout)
        out = ops.spconv_fwd(feats.contiguous(), nbr, d_n_out, out_cap, wp, None, None if bias is None else bias.detach().float(), None,
                             False, _lib.DZ_F32, kshape=kshape, layout='k')
        ctx.save_for_backward(feats, weight, nbr, d_n_out, d_n_in)
        ctx.out_cap, ctx.kshape, ctx.has_bias = out_cap, kshape, bias is not None
        return out

    @staticmethod
    def backward(ctx, dout):
        feats, weight, nbr, d_n_out, d_n_in = ctx.saved_tensors
        K, cin, cout = ctx.kshape
        dout = dout.contiguous().float()
        dfeat = dweight = dbias = None
        if ctx.needs_input_grad[0]:
            if cin not in (16, 32, 64, 128):
                raise NotImplementedError('dgrad for cin=%d (only the raw-voxel input layer has such a width; its input needs no gradient)' % cin)
            nbrT = ops.rulebook_transpose(nbr, d_n_out, feats.shape[0])
            wpT = ops.pack_spconv_weight(weight, _lib.DZ_F32).transpose(1, 2).contiguous()        # (K, cout, cin)
            dfeat = ops.spconv_fwd(dout, nbrT, d_n_in, feats.shape[0], wpT, None, None, None, False, _lib.DZ_F32, kshape=(K, cout, cin), layout='k')
        if ctx.needs_input_grad[1]:
            dwp = ops.spconv_wgrad(feats.contiguous(), nbr, d_n_out, ctx.out_cap, dout)            # (K, cin, cout)
            dweight = dwp.permute(2, 0, 1).reshape(weight.shape)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            dbias = dout.sum(0)
        return dfeat, dweight, dbias, None, None, None, None, None


class _RuleSubm:
    def __init__(self, nbr, tab):
        self.nbr = nbr             # k-major table (exact-fp32 kernel) or None
        self.tab = tab             # row-major table (tensor-core kernels) or None
        self.order = None          # tile schedule (tensor-core kernels)
        self.tab_tiles = None      # tile-major scheduled table (persistent bf16-plane kernel)
        self.sched_ws = None       # mask digests + histogram left by the rulebook kernel


class _RuleConv:
    def __init__(self, out_idx, d_n_out, out_index, tables, out_dhw, out_cap):
        self.out_idx, self.d_n_out, self.out_index, self.out_dhw, self.out_cap = out_idx, d_n_out, out_index, out_dhw, out_cap
        self.nbr, self.tab = tables
        self.order = None
        self.tab_tiles = None
        self.sched_ws = None


class _SparseConv(SparseModule):
    #: capacity of a strided conv's output relative to its input capacity the FIRST time a layer runs (k3 s2 sites grow
    #: by <= ~1.8x in practice, 8x in theory).  Afterwards the capacity follows the largest count this layer has produced
    #: (x CAP_HEADROOM), so buffers and launch grids track the real sparsity without a per-frame host sync.  Overflow
    #: is detected (device count > capacity), raised, and the hint grows -- never silently truncated.
    OUT_CAP_FACTOR = 3.0
    CAP_HEADROOM = 1.3
    #: build a tile schedule (rows grouped by neighbour mask) with every rulebook used by a tensor-core layer
    SCHEDULE_TILES = True
    #: batches: sort the schedule by (frame, mask) so that the tiles in flight gather from ONE frame's (L2-resident) feature map
    FRAME_MAJOR = bool(int(os.environ.get('DZ_FRAME_MAJOR', '0')))      # measured (profiles/r02_spconv_notes.md): the 3 digest bits it costs outweigh the L2 gain
    #: bf16-plane layers with a schedule: build the tile-major table directly from the grid index (mask pass -> scatter -> tile
    #: pass) instead of writing a row-major table and transposing it; the tables are identical row for row
    DIRECT_TILES = True
    #: direct path, submanifold mask pass: visit rows in lattice order (neighbouring lanes share bitmap lines)
    MASK_PERM_WALK = True

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1, bias=True,
                 indice_key=None, subm=False, algo=None, mode='fp32'):
        super().__init__()
        assert groups == 1 and _triple(dilation) == [1, 1, 1], 'only what backbone3d.py uses'
        self.in_channels, self.out_channels = int(in_channels), int(out_channels)
        self.kernel_size, self.stride, self.padding = _triple(kernel_size), _triple(stride), _triple(padding)
        self.subm = subm
        self.indice_key = indice_key
        self.mode = mode
        self.weight = nn.Parameter(torch.empty(out_channels, *self.kernel_size, in_channels))
        nn.init.kaiming_uniform_(self.weight, a=5 ** 0.5)
        self.bias = nn.Parameter(torch.zeros(out_channels)) if bias else None
        self._packed = None
        self._packed_ver = None

    def packed_weight(self, mode=_lib.DZ_F32):
        """kernel-layout copy of the spconv-layout parameter (refreshed when the parameter changes)"""
        ver = (self.weight._version, self.weight.data_ptr(), mode)
        if self._packed is None or self._packed_ver != ver:
            self._packed = ops.pack_spconv_weight(self.weight, mode)
            self._packed_ver = ver
        return self._packed

    @property
    def kshape(self):
        return (self.kernel_size[0] * self.kernel_size[1] * self.kernel_size[2], self.in_channels, self.out_channels)

    def _rule(self, x, schedule=True):
        key = self.indice_key
        rule = x.indice_dict.get(key) if key is not None else None
        if rule is None:
            tc = _lib.MODES[self.mode] != _lib.DZ_F32
            layout = 'row' if tc else 'k'
            want = self._wants_schedule()
            direct = want and self.DIRECT_TILES and _lib.MODES[self.mode] in _lib.PLANES
            fm = self.FRAME_MAJOR and x.batch_size > 1
            if self.subm:
                sws = ops.new_sched_ws(x._cap, x._idx.device) if want else None
                if direct:
                    ops.rulebook_subm_masks(x._idx, x._count, x._cap, x.grid_index(), self.kernel_size, sws, frame_major=fm,
                                            perm_walk=self.MASK_PERM_WALK)
                    rule = _RuleSubm(None, None)
                else:
                    t = ops.rulebook_subm(x._idx, x._count, x._cap, x.grid_index(), self.kernel_size, layout=layout, sched_ws=sws,
                                          frame_major=fm)
                    rule = _RuleSubm(None if tc else t, t if tc else None)
                rule.rows = (x._idx, x._count, x._cap)
            else:
                in_index = x.grid_index()
                out_dhw = ops.conv_out_dhw(x.spatial_shape, self.kernel_size, self.stride, self.padding)
                cells = x.batch_size * out_dhw[0] * out_dhw[1] * out_dhw[2]
                # one input site reaches prod_d ceil(k_d / s_d) output sites at most (8 for k3 s2, 2 for conv_out's (3,1,1)/(2,1,1));
                # in practice k3 s2 grows the site count by <= ~1.8x, hence the smaller first-run factor
                worst = 1
                for kd, sd_ in zip(self.kernel_size, self.stride):
                    worst *= -(-kd // sd_)
                grow = min(float(worst), self.OUT_CAP_FACTOR)
                out_cap = int(min(cells, max(64, int(x._cap * grow))))
                hint = getattr(self, '_cap_hint', None)
                if hint is not None:
                    out_cap = int(min(cells, max(128, (int(hint * self.CAP_HEADROOM) + 127) // 128 * 128)))
                sws = ops.new_sched_ws(out_cap, x._idx.device) if want else None
                if direct:
                    oc, d_n_out, out_index, odhw = ops.rulebook_conv_masks(x._idx, x._count, x._cap, in_index, self.kernel_size, self.stride,
                                                                           self.padding, out_cap, sws, frame_major=fm)
                    rule = _RuleConv(oc, d_n_out, out_index, (None, None), odhw, out_cap)
                else:
                    oc, d_n_out, out_index, t, odhw = ops.rulebook_conv(x._idx, x._count, x._cap, in_index, self.kernel_size, self.stride,
                                                                        self.padding, out_cap, layout=layout, sched_ws=sws, frame_major=fm)
                    rule = _RuleConv(oc, d_n_out, out_index, (None, t) if tc else (t, None), odhw, out_cap)
                rule.rows = (oc, d_n_out, out_cap)
            rule.sched_ws = sws
            rule.frame_major = fm
            rule.direct = direct
            rule.in_idx, rule.in_count, rule.in_cap, rule.in_dhw, rule.in_index = x._idx, x._count, x._cap, x.spatial_shape, x._index
            if key is not None:
                x.indice_dict[key] = rule
        if schedule:
            self._schedule(rule, x)
        return rule

    def _wants_schedule(self):
        K = self.kernel_size[0] * self.kernel_size[1] * self.kernel_size[2]
        return self.SCHEDULE_TILES and _lib.MODES[self.mode] != _lib.DZ_F32 and K > 1

    def _schedule(self, rule, x):
        """tile schedule of a rulebook (once per rulebook; only the tensor-core kernels use it)"""
        if rule.order is None and rule.sched_ws is not None:
            d_n = x._count if self.subm else rule.d_n_out
            fm = getattr(rule, 'frame_major', False)
            if getattr(rule, 'direct', False):             # tile-major table straight from the masks and the input grid index
                rows, d_n, cap = rule.rows
                stride, pad = ([1, 1, 1], [0, 0, 0]) if self.subm else (self.stride, self.padding)
                rule.order, rule.tab_tiles = ops.rulebook_schedule_direct(rows, d_n, cap, rule.in_index, self.kernel_size, stride, pad,
                                                                          self.subm, rule.sched_ws, x.batch_size, fm)
            elif _lib.MODES[self.mode] in _lib.PLANES:        # persistent kernel: also the tile-major table (one bulk copy per tile)
                rule.order, rule.tab_tiles = ops.rulebook_schedule(rule.tab, d_n, rule.sched_ws, x.batch_size, fm, K=self.kshape[0])
            else:
                rule.order = ops.rulebook_schedule(rule.tab, d_n, rule.sched_ws, x.batch_size, fm)

    def _table(self, rule):
        """(table, row_order) for this layer's kernel; the table is None for a direct-path rulebook on a bf16-plane layer"""
        if _lib.MODES[self.mode] != _lib.DZ_F32:
            if rule.tab is None and rule.nbr is None:     # direct path: only the tile-major table exists
                if _lib.MODES[self.mode] in _lib.PLANES:
                    return None, rule.order
                _, d_n, cap = rule.rows
                rule.tab = ops.tiles_to_rows(rule.tab_tiles, rule.order, d_n, cap)
            if rule.tab is None:                      # rulebook shared with an exact-fp32 layer: convert once
                rule.tab = ops.table_to_rows(rule.nbr)
            return rule.tab, rule.order
        if rule.nbr is None:
            raise RuntimeError('rulebook %r was built for a tensor-core layer; an exact-fp32 layer cannot share it' % self.indice_key)
        return rule.nbr, None

    def forward_fused(self, x, scale=None, shift=None, residual=None, relu=False):
        rule = self._rule(x)
        evs = x.indice_dict.get('__events__')
        if evs is not None and self.indice_key in evs:               # rulebook was built on the side stream
            torch.cuda.current_stream().wait_event(evs[self.indice_key])
        mode = _lib.MODES[self.mode]
        nbr, order = self._table(rule)
        lay = 'k' if mode == _lib.DZ_F32 else 'row'
        planes = _lib.PLANES.get(mode, 0)
        if planes:                                       # bf16 operand planes: inputs converted once, outputs stay in planes
            feat = x._as_planes(planes, 8 if self.in_channels <= 8 else self.in_channels)
            res = None if residual is None else residual._as_planes(planes, self.out_channels)
        else:
            if x._planes or (residual is not None and residual._planes):
                raise RuntimeError('a bf16-plane tensor cannot feed a %s layer: use one COMPUTE_MODE per backbone' % self.mode)
            feat, res = x._feat, (None if residual is None else residual._feat)
        if self.subm:
            out = ops.spconv_fwd(feat, nbr, x._count, x._cap, self.packed_weight(mode), scale, shift, res, relu, mode,
                                 kshape=self.kshape, row_order=order, layout=lay, tab_tiles=rule.tab_tiles)
            return x._like(out, planes)
        out = ops.spconv_fwd(feat, nbr, rule.d_n_out, rule.out_cap, self.packed_weight(mode), scale, shift, None,
                             relu, mode, d_n_in=x._count, kshape=self.kshape, row_order=order, layout=lay, tab_tiles=rule.tab_tiles)
        t = SparseConvTensor(out, rule.out_idx, rule.out_dhw, x.batch_size, indice_dict=x.indice_dict,
                             count=rule.d_n_out, n_host=None, index=rule.out_index)
        t._planes = planes
        t._producer = self
        return t

    def _rule_train(self, x):
        """exact-size k-major rulebook for the autograd path (one host read of the output-site count per strided conv)"""
        key = ('train', self.indice_key)
        rule = x.indice_dict.get(key) if self.indice_key is not None else None
        if rule is None:
            n_in = x.num()
            if self.subm:
                nbr = ops.rulebook_subm(x._idx, x._count, x._cap, x.grid_index(), self.kernel_size, layout='k')
                rule = _RuleSubm(nbr, None)
            else:
                out_dhw = ops.conv_out_dhw(x.spatial_shape, self.kernel_size, self.stride, self.padding)
                worst = 1
                for kd, sd_ in zip(self.kernel_size, self.stride):
                    worst *= -(-kd // sd_)
                cells = x.batch_size * out_dhw[0] * out_dhw[1] * out_dhw[2]
                cap = int(min(cells, max(64, n_in * worst)))
                oc, d_n_out, out_index, nbr, odhw = ops.rulebook_conv(x._idx, x._count, x._cap, x.grid_index(), self.kernel_size, self.stride,
                                                                      self.padding, cap, layout='k')
                n_out = int(d_n_out.item())
                rule = _RuleConv(oc[:n_out].contiguous(), d_n_out, out_index, (nbr[:, :n_out].contiguous(), None), odhw, n_out)
            rule.in_idx, rule.in_count, rule.in_cap, rule.in_dhw, rule.in_index = x._idx, x._count, x._cap, x.spatial_shape, x._index
            if self.indice_key is not None:
                x.indice_dict[key] = rule
        return rule

    def forward_train(self, x):
        if x._planes:
            raise RuntimeError('the training path works on fp32 features')
        if x._cap != x.num():
            x = x.replace_feature(x.features)                    # exact-size tensor (count == capacity)
            x._index = None
        rule = self._rule_train(x)
        if self.subm:
            out = _SparseConvFn.apply(x._feat, self.weight, self.bias, rule.nbr, x._count, x._cap, x._count, self.kshape)
            return x._like(out)
        out = _SparseConvFn.apply(x._feat, self.weight, self.bias, rule.nbr, rule.d_n_out, rule.out_cap, x._count, self.kshape)
        return SparseConvTensor(out, rule.out_idx, rule.out_dhw, x.batch_size, indice_dict=x.indice_dict, index=rule.out_index)

    def forward(self, x):
        if self.training:
            return self.forward_train(x)
        shift = None if self.bias is None else self.bias.detach().float()
        return self.forward_fused(x, None, shift, None, False)


class SubMConv3d(_SparseConv):
    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1, bias=True,
                 indice_key=None, algo=None, **kw):
        super().__init__(in_channels, out_channels, kernel_size, 1, padding, dilation, groups, bias, indice_key, True,
                         algo, kw.get('mode', 'fp32'))


class SparseConv3d(_SparseConv):
    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1, bias=True,
                 indice_key=None, algo=None, **kw):
        super().__init__(in_channels, out_channels, kernel_size, stride, padding, dilation, groups, bias, indice_key,
                         False, algo, kw.get('mode', 'fp32'))


class _InverseConvFn(torch.autograd.Function):
    """out[j] = sum over the pairs (k, j, o) of the matching SparseConv3d of W[k] in[o]: the forward kernel on the transposed table"""

    @staticmethod
    def forward(ctx, feats, weight, bias, nbrT, nbr, d_n_in_sites, in_cap, d_n_out_sites, kshape):
        wp = ops.pack_spconv_weight(weight, _lib.DZ_F32)
        out = ops.spconv_fwd(feats.contiguous(), nbrT, d_n_in_sites, in_cap, wp, None, None if bias is None else bias.detach().float(), None,
                             False, _lib.DZ_F32, kshape=kshape, layout='k')
        ctx.save_for_backward(feats, weight, nbrT, nbr, d_n_in_sites, d_n_out_sites)
        ctx.in_cap, ctx.kshape, ctx.has_bias = in_cap, kshape, bias is not None
        return out

    @staticmethod
    def backward(ctx, dout):
        feats, weight, nbrT, nbr, d_a, d_b = ctx.saved_tensors
        K, cin, cout = ctx.kshape
        dout = dout.contiguous().float()
        dfeat = dweight = dbias = None
        if ctx.needs_input_grad[0]:
            wpT = ops.pack_spconv_weight(weight, _lib.DZ_F32).transpose(1, 2).contiguous()
            dfeat = ops.spconv_fwd(dout, nbr, d_b, feats.shape[0], wpT, None, None, None, False, _lib.DZ_F32, kshape=(K, cout, cin), layout='k')
        if ctx.needs_input_grad[1]:
            dweight = ops.spconv_wgrad(feats.contiguous(), nbrT, d_a, ctx.in_cap, dout).permute(2, 0, 1).reshape(weight.shape)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            dbias = dout.sum(0)
        return dfeat, dweight, dbias, None, None, None, None, None, None


class SparseInverseConv3d(SparseModule):
    """spconv.SparseInverseConv3d(in, out, kernel_size, indice_key=, bias=) (post_act_block 'inverseconv', backbone3d.py:72-73):
    undoes the sparsity pattern of the SparseConv3d that shares its ``indice_key`` -- output sites = that conv's INPUT sites,
    ``out[j] = sum W[k] in[o]`` over that conv's pairs (k, j, o).  Exact fp32, differentiable."""

    def __init__(self, in_channels, out_channels, kernel_size, indice_key=None, bias=True, **kw):
        super().__init__()
        assert indice_key is not None, 'SparseInverseConv3d needs the indice_key of the SparseConv3d it inverts'
        self.in_channels, self.out_channels = int(in_channels), int(out_channels)
        self.kernel_size = _triple(kernel_size)
        self.indice_key = indice_key
        self.weight = nn.Parameter(torch.empty(out_channels, *self.kernel_size, in_channels))
        nn.init.kaiming_uniform_(self.weight, a=5 ** 0.5)
        self.bias = nn.Parameter(torch.zeros(out_channels)) if bias else None

    def forward(self, x):
        rule = x.indice_dict.get(('train', self.indice_key)) or x.indice_dict.get(self.indice_key)
        if rule is None or not isinstance(rule, _RuleConv):
            raise RuntimeError('SparseInverseConv3d(%r): no SparseConv3d with this indice_key has run on this tensor' % self.indice_key)
        K = self.kernel_size[0] * self.kernel_size[1] * self.kernel_size[2]
        if rule.nbr is None:                                    # rulebook built for a tensor-core layer: k-major copy of the row-major table
            if rule.tab is None:                                # direct path: row-major form of the tile-major table first
                rule.tab = ops.tiles_to_rows(rule.tab_tiles, rule.order, rule.d_n_out, rule.out_cap)
            rule.nbr = rule.tab[:, :K].t().contiguous()
        if not hasattr(rule, 'in_idx'):
            raise RuntimeError('rulebook %r does not remember its input sites' % self.indice_key)
        if x._planes:
            x = x.replace_feature(x.features)
        if getattr(rule, 'nbrT', None) is None:
            rule.nbrT = ops.rulebook_transpose(rule.nbr, rule.d_n_out, rule.in_cap)
        out = _InverseConvFn.apply(x._feat, self.weight, self.bias, rule.nbrT, rule.nbr, rule.in_count, rule.in_cap, rule.d_n_out,
                                   (K, self.in_channels, self.out_channels))
        return SparseConvTensor(out, rule.in_idx, rule.in_dhw, x.batch_size, indice_dict=x.indice_dict, count=rule.in_count, n_host=None,
                                index=rule.in_index)


class SparseSequential(SparseModule):
    """Applies SparseModules to the tensor and plain nn.Modules to ``.features`` (spconv semantics).  In eval mode
    the pattern conv -> BatchNorm1d [-> ReLU] is executed as ONE fused launch."""

    def __init__(self, *mods):
        super().__init__()
        for i, m in enumerate(mods):
            self.add_module(str(i), m)

    def forward(self, x):
        mods = list(self._modules.values())
        i = 0
        while i < len(mods):
            m = mods[i]
            if isinstance(m, _SparseConv) and not self.training and i + 1 < len(mods) and \
                    isinstance(mods[i + 1], nn.BatchNorm1d) and not mods[i + 1].training:
                bn = mods[i + 1]
                relu = i + 2 < len(mods) and isinstance(mods[i + 2], nn.ReLU)
                scale, shift = fold_bn(bn, m.bias, x._feat.device)
                x = m.forward_fused(x, scale, shift, None, relu)
                i += 3 if relu else 2
            elif isinstance(m, SparseModule):
                x = m(x)                       # training: _SparseConv.forward -> the autograd path, BatchNorm1d / ReLU follow unfused
                i += 1
            else:
                if x._planes:
                    raise RuntimeError('plain nn.Modules cannot act on a bf16-plane tensor (only the fused eval path supports the bf16 modes)')
                x = x._like(m(x._feat))        # acts on all capacity rows; rows beyond the count are never read
                i += 1
        return x
