"""ctypes binding of libdetzero_b200.so (the C ABI in include/detzero_b200.h).

There is no CPU fallback: if the library is missing, or a call fails, this raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libdetzero_b200.so')

DZ_F32, DZ_TF32, DZ_BF16, DZ_TF32X3, DZ_BF16X2 = 0, 1, 2, 3, 4
MODES = {'fp32': DZ_F32, 'f32': DZ_F32, 'tf32': DZ_TF32, 'bf16': DZ_BF16, 'tf32x3': DZ_TF32X3, 'fp32_tc': DZ_TF32X3,
         'bf16x2': DZ_BF16X2}
#: bf16 operand planes per mode (sparse conv, csrc/spconv_bf16.cu)
PLANES = {DZ_BF16: 1, DZ_BF16X2: 2}

_lib = None

vp = ctypes.c_void_p
ci = ctypes.c_int
cf = ctypes.c_float
sz = ctypes.c_size_t

_SIGS = {
    'dz_version': (ci, []),
    'dz_sm_arch': (ci, []),
    'dz_last_error_string': (ctypes.c_char_p, []),
    'dz_grid_index_words': (sz, [ci, ci, ci, ci]),
    'dz_scan_ws_bytes': (sz, [sz]),
    'dz_grid_index_scan': (ci, [vp, vp, sz, vp, vp, vp, sz, vp]),
    'dz_grid_index_from_coords': (ci, [vp, vp, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp, sz, vp]),
    'dz_voxelize_hard_ws_bytes': (sz, [ci, ci, ci, ci, ci, ci]),
    'dz_voxelize_hard': (ci, [vp, ci, ci, ci, ci, vp, vp, vp, ci, ci, ci, vp, vp, vp, vp, ci, vp,
                              ci, ci, ci, ci, vp, vp, vp, vp, sz, vp]),
    'dz_voxelize_hard_batch_ws_bytes': (sz, [ci, ci, ci, ci, ci, ci, ci]),
    'dz_voxelize_hard_batch': (ci, [vp, vp, ci, ci, ci, ci, vp, vp, vp, ci, ci, vp, vp, vp, vp, ci, vp,
                                    ci, ci, ci, vp, vp, vp, vp, sz, vp]),
    'dz_mean_vfe': (ci, [vp, vp, ci, ci, ci, vp, vp]),
    'dz_voxelize_dynamic_ws_bytes': (sz, [ci, ci, ci, ci, ci, ci]),
    'dz_voxelize_dynamic_mean': (ci, [vp, ci, ci, ci, vp, vp, vp, vp, vp, ci, vp, vp, sz, vp]),
    'dz_rulebook_subm': (ci, [vp, vp, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp, vp, vp, ci, vp]),
    'dz_rulebook_conv': (ci, [vp, vp, ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci, vp, vp, vp, vp, vp, sz, vp, ci, vp]),
    'dz_rulebook_schedule_ws_bytes': (sz, [ci]),
    'dz_rulebook_schedule': (ci, [vp, ci, vp, vp, vp, sz, ci, ci, ci, vp, vp]),
    'dz_rulebook_subm_masks': (ci, [vp, vp, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp, ci, ci, vp]),
    'dz_rulebook_conv_masks': (ci, [vp, vp, ci, ci, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci, vp, vp, vp, sz, vp, ci, vp]),
    'dz_rulebook_schedule_direct': (ci, [vp, ci, vp, ci, vp, vp, vp, vp, ci, vp, vp, vp, vp, vp, sz, ci, vp, vp]),
    'dz_spconv_fwd': (ci, [vp, ci, ci, vp, ci, ci, vp, vp, ci, vp, vp, vp, vp, ci, vp, ci, ci, vp]),
    'dz_rulebook_transpose': (ci, [vp, ci, ci, vp, vp, ci, vp]),
    'dz_spconv_wgrad': (ci, [vp, ci, vp, ci, ci, vp, ci, vp, ci, vp, vp]),
    'dz_spconv_fwd_planes': (ci, [vp, ci, ci, vp, ci, ci, vp, vp, ci, vp, vp, vp, vp, ci, vp, ci, ci, vp, vp]),
    'dz_to_planes': (ci, [vp, vp, ci, ci, ci, ci, vp, vp]),
    'dz_from_planes': (ci, [vp, vp, ci, ci, ci, vp, vp]),
    'dz_sparse_to_bev': (ci, [vp, vp, vp, ci, ci, ci, ci, ci, ci, vp, vp]),
    'dz_sparse_to_bev_planes': (ci, [vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, vp, vp]),
    'dz_conv2d_fwd': (ci, [vp, ci, ci, ci, ci, ci, vp, ci, ci, ci, ci, vp, vp, ci, vp, ci, ci, ci, ci, ci, ci, vp]),
    'dz_deconv2d_fwd': (ci, [vp, ci, ci, ci, ci, vp, ci, vp, vp, ci, vp, ci, ci, ci, ci, vp]),
    'dz_centerhead_decode_ws_bytes': (sz, [ci, ci, ci, ci, ci]),
    'dz_centerhead_decode': (ci, [vp, ci, ci, ci, ci, ci, ci, ci, ci, ci, ci, ci, ci, vp, vp, ci, vp, cf, ci,
                                  vp, vp, vp, vp, vp, sz, vp]),
    'dz_nms_bev_ws_bytes': (sz, [ci, ci]),
    'dz_nms_bev': (ci, [vp, vp, vp, vp, ci, ci, cf, ci, ci, vp, vp, vp, sz, vp]),
    'dz_boxes_iou_bev': (ci, [vp, ci, vp, ci, vp, vp]),
    'dz_prepare_points_ws_bytes': (sz, [ci]),
    'dz_prepare_points': (ci, [vp, ci, vp, cf, ci, ci, vp, ci, vp, vp, sz, vp]),
    'dz_boxes_pairwise': (ci, [vp, ci, ci, vp, ci, ci, ci, vp, vp]),
    'dz_crop_points_ws_bytes': (sz, [ci, ci]),
    'dz_crop_points_in_boxes': (ci, [vp, ci, ci, vp, ci, ci, vp, ci, vp, vp, sz, vp]),
    'dz_points_in_boxes_mask': (ci, [vp, ci, ci, vp, ci, ci, vp, vp]),
    'dz_linear_fwd': (ci, [vp, ci, ci, vp, ci, vp, vp, ci, vp, ci, ci, vp]),
    'dz_linear_fwd_grouped': (ci, [vp, ci, ci, vp, ci, vp, vp, vp, ci, ci, vp, ci, ci, vp]),
    'dz_linear_max_fwd': (ci, [vp, ci, ci, vp, ci, vp, vp, ci, ci, vp, ci, vp]),
    'dz_group_max': (ci, [vp, ci, ci, ci, vp, vp]),
    'dz_attention_fwd': (ci, [vp, ci, vp, ci, vp, ci, vp, ci, ci, ci, ci, ci, vp, ci, ci, vp]),
    'dz_layernorm_residual': (ci, [vp, vp, vp, vp, cf, ci, ci, vp, vp]),
    'dz_add': (ci, [vp, vp, sz, vp, vp]),
}


def lib():
    """Load the library (once).  Raises if it has not been built -- the product path never falls back to CPU."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                'detzero_b200: %s is missing. Build it with `python -c "import __graft_entry__ as g; g.build()"` '
                '(nvcc, sm_100a). There is no CPU fallback.' % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)            # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def exported_symbols():
    return sorted(_SIGS.keys())


def check(rc, what=''):
    if rc != 0:
        msg = lib().dz_last_error_string()
        raise RuntimeError('detzero_b200 %s failed (rc=%d): %s' % (what, rc, msg.decode() if msg else ''))


def farr(vals):
    return (ctypes.c_float * len(vals))(*[float(v) for v in vals])


def iarr(vals):
    return (ctypes.c_int * len(vals))(*[int(v) for v in vals])
