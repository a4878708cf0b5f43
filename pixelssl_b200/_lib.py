"""ctypes binding of libpixelssl_b200.so (the C ABI declared in include/pixelssl_b200.h).

There is NO fallback: if the shared library is missing or a symbol is absent, importing / calling
raises.  The binding below is exactly the stub shown in INTEGRATION.md."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libpixelssl_b200.so')

c_void_p, c_int, c_int64, c_float, c_double = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                               ctypes.c_float, ctypes.c_double)


class ConvGeom(ctypes.Structure):
    """mirror of pxl_conv_geom"""
    _fields_ = [('N', c_int), ('H', c_int), ('W', c_int), ('Cin', c_int),
                ('OH', c_int), ('OW', c_int), ('Cout', c_int), ('ldo', c_int),
                ('mul', c_int), ('div', c_int), ('ntaps', c_int), ('precision', c_int)]


class ConvTcExt(ctypes.Structure):
    """mirror of pxl_conv_tc_ext"""
    _fields_ = [('w_ntaps', c_int), ('widx_host', ctypes.POINTER(c_int)), ('out_mul', c_int),
                ('out_offy', c_int), ('out_offx', c_int), ('out_H', c_int), ('out_W', c_int),
                ('bn_stats', c_void_p), ('out_scale', c_float), ('out_scale_dev', c_void_p), ('out_accumulate', c_int)]


P = c_void_p
# name -> (restype, argtypes); must list every symbol of include/pixelssl_b200.h
SIGNATURES = {
    'pxl_abi_version': (c_int, []),
    'pxl_launch_count': (c_int64, []),
    'pxl_reset_launch_count': (None, []),
    'pxl_mse_workspace_bytes': (c_int64, []),
    'pxl_mse_consistency': (c_int, [P, P, c_int64, c_float, P, P, P, P]),
    'pxl_mse_consistency_bwd': (c_int, [P, P, c_int64, c_float, P, P, P]),
    'pxl_ce2d': (c_int, [P, P, c_int, c_int, c_int64, c_int, P, P, P, c_float, P]),
    'pxl_softmax_planar': (c_int, [P, P, c_int, c_int, c_int64, P]),
    'pxl_softmax_planar_bwd': (c_int, [P, P, P, c_int, c_int, c_int64, P]),
    'pxl_softmax_mse': (c_int, [P, P, c_int, c_int, c_int64, c_float, P, P, P, P, P]),
    'pxl_bilinear_fwd': (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_bilinear_bwd': (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_cutmix_mix': (c_int, [P, P, P, P, c_int, c_int, c_int64, P]),
    'pxl_cutmix_confidence': (c_int, [P, c_int, c_int, c_int64, c_float, P, P]),
    'pxl_bn_stats': (c_int, [P, c_int64, c_int, P, P]),
    'pxl_bn_finalize': (c_int, [P, c_double, c_int, P, P, P, P, c_float, c_float, c_int, P, P, P, P, P]),
    'pxl_bn_eval_coeffs': (c_int, [c_int, P, P, P, P, c_float, P, P, P]),
    'pxl_bn_apply': (c_int, [P, P, P, P, c_int, P, c_int64, c_int, P]),
    'pxl_bn_bwd_reduce': (c_int, [P, P, P, P, P, c_int, c_int64, c_int, P, P, P, P]),
    'pxl_bn_bwd_dx': (c_int, [P, P, P, P, P, P, P, c_double, c_int, P, P, c_int64, c_int, P, P, P, P, P]),
    'pxl_bn_finalize_apply': (c_int, [P, P, c_double, P, P, P, P, c_float, c_float, c_int, P, P, P, P, P, c_int, P, c_int64,
                                      c_int, P]),
    'pxl_bn_bwd_params': (c_int, [P, c_int, P, P, c_int, P]),
    'pxl_bn_apply_h16': (c_int, [P, P, P, P, c_int, P, c_int64, c_int, P, P, c_float, P, P]),
    'pxl_bn_finalize_apply_h16': (c_int, [P, P, c_double, P, P, P, P, c_float, c_float, c_int, P, P, P, P, P, c_int, P, c_int64,
                                          c_int, P, P, c_float, P, P]),
    'pxl_bn_bwd_reduce_h16': (c_int, [P, P, P, P, P, c_int, c_int64, c_int, P, P, P, P, P, P]),
    'pxl_bn_bwd_dx_h16': (c_int, [P, P, P, P, P, P, P, c_double, c_int, P, P, c_int64, c_int, P, P, P, P, P, P, P, c_int, P, P]),
    'pxl_maxpool3x3s2_fwd': (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_maxpool3x3s2_bwd': (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_conv_nhwc': (c_int, [ctypes.POINTER(ConvGeom), ctypes.POINTER(c_int), P, P, P, P, P]),
    'pxl_conv_wgrad_nhwc': (c_int, [ctypes.POINTER(ConvGeom), ctypes.POINTER(c_int), P, P, P, P]),
    'pxl_conv_tc_launch': (c_int, [ctypes.POINTER(ConvGeom), ctypes.POINTER(c_int), P, P, P, P, P, P, P]),
    'pxl_conv_tc_launch_ex': (c_int, [ctypes.POINTER(ConvGeom), ctypes.POINTER(c_int), ctypes.POINTER(ConvTcExt), P, P, P, P, P, P, P]),
    'pxl_conv_wgrad_workspace_floats': (c_int64, [ctypes.POINTER(ConvGeom), ctypes.POINTER(c_int)]),
    'pxl_conv_wgrad_tc_launch': (c_int, [ctypes.POINTER(ConvGeom), ctypes.POINTER(c_int), P, P, P, P, P, P, c_int64, P]),
    'pxl_conv_h16_launch': (c_int, [ctypes.POINTER(ConvGeom), ctypes.POINTER(c_int), ctypes.POINTER(ConvTcExt), P, P, P, P, P, P, P]),
    'pxl_conv_wgrad_h16_launch': (c_int, [ctypes.POINTER(ConvGeom), ctypes.POINTER(c_int), P, P, P, P, P, c_float, P, P, c_int64,
                                          P]),
    'pxl_h16_split': (c_int, [P, P, P, c_int64, c_float, P, c_int, P]),
    'pxl_h16_absmax': (c_int, [P, c_int64, P, P]),
    'pxl_h16_sat_counter': (c_void_p, []),
    'pxl_h16_status': (c_int, []),
    'pxl_h16_status_sites': (c_int, [P]),
    'pxl_h16_reset_status': (c_int, []),
    'pxl_split_tf32': (c_int, [P, P, P, c_int64, P]),
    'pxl_conv_tc_status': (c_int, []),
    'pxl_conv_transpose_weights': (c_int, [P, P, c_int, c_int, c_int, P]),
    'pxl_conv_transpose_weights_batched': (c_int, [P, P, P, c_int, c_int64, P]),
    'pxl_bias_grad': (c_int, [P, c_int64, c_int, c_int, P, c_int, P]),
    'pxl_stem_conv7x7s2': (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_stem_conv7x7s2_wgrad': (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_stem_im2col': (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_planar_to_nhwc': (c_int, [P, P, c_int, c_int, c_int64, c_int, c_int, P]),
    'pxl_nhwc_to_planar': (c_int, [P, P, c_int, c_int, c_int64, c_int, c_int, P]),
    'pxl_onehot_nhwc': (c_int, [P, P, c_int64, c_int, c_int, c_int, P]),
    'pxl_leaky_relu_fwd': (c_int, [P, P, c_int64, c_float, P]),
    'pxl_leaky_relu_bwd': (c_int, [P, P, P, c_int64, c_float, P]),
    'pxl_bce_logits_masked': (c_int, [P, P, c_float, c_int, c_int, c_int64, P, P, P, c_float, P]),
    'pxl_adam': (c_int, [P, P, P, P, c_int64, c_float, c_float, c_float, c_float, c_float, c_int, P]),
    'pxl_gauss_blur_sep': (c_int, [P, P, P, c_int, c_int, c_int, c_int, P, c_float, P]),
    'pxl_dilate3x3_reflect': (c_int, [P, P, c_int, c_int, c_int, P]),
    'pxl_minmax_norm': (c_int, [P, P, c_int, c_int64, c_float, c_float, c_float, P]),
    'pxl_gct_dcgt': (c_int, [P, P, P, P, c_float, c_int, c_int, c_int64, P, P, P, P]),
    'pxl_fdgt_absdiff': (c_int, [P, P, c_float, c_int, c_int, c_int64, P, P]),
    'pxl_pixel_shuffle2_nhwc': (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_perturb_nhwc': (c_int, [P, P, P, P, P, c_int, c_int64, c_int, P]),
    'pxl_channel_mean_nhwc': (c_int, [P, P, c_int64, c_int, P]),
    'pxl_argmax_nonzero_mask': (c_int, [P, P, c_int, c_int, c_int64, P]),
    'pxl_adaptive_avgpool_nhwc': (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_bilinear_nhwc': (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_copy_lanes_nhwc': (c_int, [P, P, c_int64, c_int, c_int, c_int, c_int, P]),
    'pxl_confusion_matrix': (c_int, [P, P, c_int, c_int, c_int64, P, P]),
    'pxl_gaussian_noise_workspace_bytes': (c_int64, [c_int]),
    'pxl_gaussian_noise': (c_int, [P, P, c_int, c_int64, P, P]),
    'pxl_peer_mailbox_bytes': (c_int64, []),
    'pxl_peer_alloc': (c_int, [P]),
    'pxl_peer_free': (c_int, [P]),
    'pxl_peer_export': (c_int, [P, P]),
    'pxl_peer_open': (c_int, [P, P]),
    'pxl_peer_close': (c_int, [P]),
    'pxl_peer_allreduce_bn': (c_int, [P, c_int, P, c_int, c_int, c_int64, c_double, c_int, P, P, P, P, c_float, c_float,
                                      c_int, P, P, P, P, P, P, P]),
    'pxl_peer_status': (c_int, []),
    'pxl_stem_im2col_h16': (c_int, [P, P, P, c_float, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_aspp_gather': (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_int), c_int, P]),
    'pxl_aspp_scatter_h16': (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_int), c_int, P]),
    'pxl_s4l_rotate_batch': (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, P]),
    'pxl_input_prehandle': (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, P, P, c_int, P, P, c_int, P, P, c_int, c_int, c_int, c_int,
                                    c_int, c_float, c_float, P, P, P, P, P]),
    'pxl_sgd_ema': (c_int, [P, P, P, P, c_int64, c_float, c_float, c_float, c_float, c_int, P]),
    'pxl_ema': (c_int, [P, P, c_int64, c_float, P]),
}

PXL_ERR_BAD_ARG = -1
PXL_ERR_UNSUPPORTED = -2

_lib = None


class PxlError(RuntimeError):
    def __init__(self, fn, code):
        self.fn, self.code = fn, code
        what = {PXL_ERR_BAD_ARG: 'bad argument', PXL_ERR_UNSUPPORTED: 'unsupported configuration'}.get(
            code, 'cudaError_t %d' % code)
        super().__init__('%s failed: %s' % (fn, what))


def load():
    """Load (once) and type the library.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            'pixelssl_b200: %s not found. Build it with `python -c "import __graft_entry__ as g; '
            'g.build()"` (nvcc, sm_100a). There is no CPU/PyTorch fallback.' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing: loud by design
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


_bound = {}


def call(name, *args):
    """Call an int-returning entry point and raise PxlError on a non-zero return."""
    fn = _bound.get(name)
    if fn is None:
        fn = _bound[name] = getattr(load(), name)
    rc = fn(*args)
    if rc != 0:
        raise PxlError(name, rc)
    return rc
