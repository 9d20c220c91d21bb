"""ctypes loader for libyolo2_b200.so.  No fallback: a missing library is an ImportError with build
instructions, a non-zero return code is a RuntimeError carrying yb_last_error()."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# YB_LIB_PATH: A/B a differently-compiled build of the same library (tools/ only)
LIB_PATH = os.environ.get('YB_LIB_PATH') or os.path.join(os.path.dirname(_HERE), 'libyolo2_b200.so')

c_int, c_float, c_void_p, c_longlong = ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_longlong
P = c_void_p

# name -> argument ctypes (every function returns int); mirrors include/yolo2_b200.h
SIGNATURES = {
    'yb_version': [],
    'yb_debug_read': [ctypes.POINTER(c_int * 4)],
    'yb_conv_set_trace': [P],
    'yb_pack_weight_f16': [P, P, c_int, c_int, c_int, c_int, P],
    'yb_bn_fold': [P, P, P, P, c_float, P, P, c_int, P],
    'yb_conv0_bn_leaky_pool_fwd': [P, P, P, P, c_float, P, c_int, c_int, c_int, c_int, P],
    'yb_conv0_u8_bn_leaky_pool_fwd': [P, P, P, P, c_float, P, c_int, c_int, c_int, c_int, P],
    'yb_conv_bn_act_fwd': [P, P, P, P, c_float, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_longlong, c_int, c_int, c_int, P],
    'yb_conv_bn_act_stats_fwd': [P, P, P, P, c_float, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_longlong, c_int, c_int, P, P],
    'yb_conv_workspace_bytes': [],
    'yb_conv_bn_act_fwd_ws': [P, P, P, P, c_float, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_longlong, c_int, c_int, c_int, P,
                              c_longlong, P],
    'yb_conv_bn_act_split_fwd': [P, P, P, P, c_float, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_longlong, c_int, c_int, c_int,
                                 c_int, P, c_longlong, P],
    'yb_pack_weight_split_f16': [P, P, c_int, c_int, c_int, c_int, c_int, P],
    'yb_maxpool2x2_split_f16': [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P],
    'yb_conv_ref_fwd': [P, P, P, P, c_float, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_longlong, c_int, c_int, P],
    'yb_maxpool2x2_f16': [P, P, c_int, c_int, c_int, c_int, c_int, P],
    'yb_maxpool2x2_s1_f16': [P, P, c_int, c_int, c_int, c_int, c_int, P],
    'yb_maxpool2x2_s1_bwd_f16': [P, P, P, c_int, c_int, c_int, c_int, P],
    'yb_reorg_f16': [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P],
    'yb_reorg_f32_nchw': [P, P, c_int, c_int, c_int, c_int, c_int, c_int, P],
    'yb_decode_fwd': [P, P, P, P, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, P],
    'yb_filter_nms': [P, P, P, P, c_int, c_int, c_int, c_int, c_float, c_float, c_float, c_int, P, P, P, P, P, P, P, P, c_int, P, P, P, P],
    'yb_iou_matrix': [P, P, P, P, P, c_int, c_int, c_int, c_float, P],
    'yb_region_loss_fwd': [P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_int, P, P, P, P, P, P, P, P, P],
    'yb_region_loss_bwd': [P, P, P, P, c_int, c_int, c_int, c_int, c_int, P],
    'yb_conv0_raw_fwd': [P, P, P, c_int, c_int, c_int, c_int, P],
    'yb_conv0_raw_stats_fwd': [P, P, P, P, c_int, c_int, c_int, c_int, P],
    'yb_pack_weight_dgrad_f16': [P, P, c_int, c_int, c_int, c_int, P],
    'yb_pack_weights_batch': [P, c_int, c_int, P],
    'yb_bn_stats': [P, c_longlong, c_longlong, c_int, P, P],
    'yb_bn_finalize': [P, c_longlong, c_int, c_float, c_float, P, P, P, P, P],
    'yb_bn_act_apply': [P, c_longlong, P, P, P, P, c_float, P, c_longlong, c_int, c_int, c_int, c_int, c_int, c_int, P],
    'yb_bn_act_bwd': [c_int, P, c_longlong, P, P, P, P, c_float, P, c_longlong, c_int, P, c_longlong, c_int, c_int, c_int, c_int, c_int, c_int,
                      P, P, c_longlong, c_int, P],
    'yb_bn_param_grad': [P, c_int, P, P, c_int, c_float, P],
    'yb_reorg_bwd_f16': [P, c_longlong, c_int, P, c_int, c_int, c_int, c_int, P],
    'yb_head_grad_prepare': [P, P, P, c_int, c_int, c_int, c_int, P],
    'yb_conv0_wgrad': [P, P, P, c_int, c_int, c_int, P],
    'yb_conv0_wgrad_bn': [P, P, P, c_longlong, c_int, P, P, P, P, c_float, P, P, c_int, c_int, c_int, P],
    'yb_conv_wgrad': [P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P],
    'yb_unpack_wgrad': [P, P, c_int, c_int, c_int, c_float, P],
    'yb_grad_guard': [P, c_longlong, P, c_int, P],
    'yb_resize_batch_u8': [P, P, P, P, c_int, c_int, c_int, c_int, P, P, c_int, P],
    'yb_resize_aug_batch_u8': [P, P, P, P, P, P, P, c_int, c_int, c_int, c_int, P, P, c_int, P],
    'yb_warp_affine_u8': [P, c_int, c_int, P, c_int, c_int, ctypes.POINTER(ctypes.c_double * 6), ctypes.POINTER(c_int * 3), P],
    'yb_totensor_u8': [P, P, c_int, c_int, c_int, P],
    'yb_photometric_u8': [P, P, c_int, c_int, c_int, P, c_int, P, c_int, P, P],
    'yb_eval_match': [P, P, P, P, P, P, P, P, c_int, c_int, c_int, c_float, c_float, P, P],
    'yb_mb_conv0_raw_fwd': [P, P, P, c_int, c_int, c_int, P],
    'yb_mb_conv0_split_fwd': [P, P, P, P, P, c_int, c_int, c_int, P],
    'yb_dwconv3x3_split_fwd': [P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, P],
    'yb_mb_conv0_wgrad': [P, P, P, c_int, c_int, c_int, P],
    'yb_dwconv3x3_raw_fwd': [P, P, P, c_int, c_int, c_int, c_int, c_int, P],
    'yb_dwconv3x3_dgrad': [P, P, P, c_int, c_int, c_int, c_int, c_int, P],
    'yb_dwconv3x3_wgrad': [P, P, P, c_int, c_int, c_int, c_int, c_int, P],
    'yb_stem7x7_bn_relu_fwd': [P, P, P, P, P, c_int, c_int, c_int, P],
    'yb_maxpool3x3_s2_f16': [P, P, c_int, c_int, c_int, c_int, P],
    'yb_subsample2_f16': [P, P, c_int, c_int, c_int, c_int, P],
    'yb_add_relu_f16': [P, P, P, c_longlong, P],
    'yb_comm_version': [ctypes.POINTER(c_int)],
    'yb_comm_unique_id': [P],
    'yb_comm_init': [ctypes.POINTER(P), c_int, P, c_int],
    'yb_comm_destroy': [P],
    'yb_allreduce_bucket': [P, P, c_longlong, c_int, P],
    'yb_broadcast_buffer': [P, P, c_longlong, c_int, c_int, P],
    'yb_mb_conv0_bn_relu_fwd': [P, P, P, P, P, c_int, c_int, c_int, P],
    'yb_dwconv3x3_bn_relu_fwd': [P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, P],
}

_lib = None


def load():
    """Load (once) and return the ctypes handle."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            'libyolo2_b200.so not found at %s -- build it with `python yolo2-pytorch_b200/build.py` '
            '(nvcc, sm_100a).  There is no CPU or PyTorch fallback for this path.' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.argtypes = argtypes
        fn.restype = c_longlong if name == 'yb_conv_workspace_bytes' else c_int
    lib.yb_last_error.argtypes = []
    lib.yb_last_error.restype = ctypes.c_char_p
    _lib = lib
    return lib


def last_error():
    return load().yb_last_error().decode('utf-8', 'replace')


def debug_read():
    buf = (c_int * 4)()
    load().yb_debug_read(ctypes.byref(buf))
    return list(buf)


def check(rc, what):
    if rc != 0:
        raise RuntimeError('%s failed (code %d): %s' % (what, rc, last_error()))
