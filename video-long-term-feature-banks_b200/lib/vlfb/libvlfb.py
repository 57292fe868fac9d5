"""ctypes binding of libvlfb.so (the C ABI declared in include/vlfb.h).

There is deliberately NO fallback: if the shared library is missing or a CUDA
device is absent the import of the kernels fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('VLFB_LIB') or os.path.normpath(os.path.join(_HERE, '..', '..', 'csrc', 'libvlfb.so'))   # VLFB_LIB: kernel-variant experiments (scripts/)

OP_DENSE_K, OP_DENSE_MN, OP_CONV_K, OP_DGRAD_K, OP_CONV_MN, OP_STEM_K, OP_STEM_MN = range(7)
EPI_RELU, EPI_ACCUM, EPI_ATOMIC, EPI_TF32 = 1, 2, 4, 8


class ConvGeom(C.Structure):
    _fields_ = [(n, C.c_int) for n in
                ('N', 'T', 'H', 'W', 'C', 'To', 'Ho', 'Wo', 'Co', 'kT', 'kH', 'kW',
                 'sT', 'sH', 'sW', 'pT', 'pH', 'pW', 'dT', 'dH', 'dW')]


class Operand(C.Structure):
    _fields_ = [('ptr', C.c_void_p), ('kind', C.c_int), ('ld', C.c_int64), ('batch_stride', C.c_int64)]


class GemmParams(C.Structure):
    _fields_ = [('a', Operand), ('b', Operand), ('g', ConvGeom),
                ('M', C.c_int), ('N', C.c_int), ('K', C.c_int),
                ('batch', C.c_int), ('taps', C.c_int), ('split_k', C.c_int),
                ('d', C.c_void_p), ('ldd', C.c_int64), ('d_batch_stride', C.c_int64),
                ('d_tap_stride', C.c_int64), ('alpha', C.c_float),
                ('col_scale', C.c_void_p), ('col_bias', C.c_void_p), ('row_scale', C.c_void_p),
                ('residual', C.c_void_p), ('relu_mask', C.c_void_p), ('flags', C.c_int),
                ('workspace', C.c_void_p), ('workspace_bytes', C.c_size_t),
                ('engine', C.c_int), ('tile_n', C.c_int), ('pair', C.c_int), ('stream_k', C.c_int),
                ('relu_mask_bits', C.c_void_p), ('relu_bits_out', C.c_void_p)]


class GemmPlan(C.Structure):
    _fields_ = [(n, C.c_int) for n in ('tile_n', 'split_k', 'pair', 'stream_k', 'tiles', 'units')]


ENGINE_TCGEN05, ENGINE_SIMT = 0, 1
DT_F32, DT_BF16 = 0, 1              # vlfb_dtype_t


class FboLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ('w_theta', 'b_theta', 'w_phi', 'b_phi', 'w_g', 'b_g', 'w_out', 'b_out',
                 'gw_theta', 'gb_theta', 'gw_phi', 'gb_phi', 'gw_g', 'gb_g', 'gw_out', 'gb_out',
                 'theta', 'prob', 's', 't', 'xhat', 'ln_mean', 'ln_std', 'out', 'a_out')] + [('drop_offset', C.c_uint64)]


class FboCfg(C.Structure):
    _fields_ = [('R', C.c_int), ('L', C.c_int), ('dA', C.c_int), ('d', C.c_int), ('dB', C.c_int), ('layers', C.c_int),
                ('scale', C.c_float), ('pre_act', C.c_int), ('pre_act_ln', C.c_int), ('ln_eps', C.c_float),
                ('drop_ratio', C.c_float), ('seed', C.c_uint64), ('step', C.c_void_p)]


_P, _I, _L, _F, _U = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint64
_GP = C.POINTER(ConvGeom)

# name -> argtypes (restype int unless noted).  Mirrors include/vlfb.h one to one.
SIGNATURES = {
    'vlfb_version': [],
    'vlfb_last_error': [],
    'vlfb_gemm': [C.POINTER(GemmParams), _P],
    'vlfb_gemm_plan': [C.POINTER(GemmParams), _I, C.POINTER(GemmPlan)],
    'vlfb_gemm_workspace_bytes': [],
    'vlfb_affine_nd_fwd': [_P, _P, _P, _P, _L, _I, _P],
    'vlfb_affine_nd_bwd': [_P, _P, _P, _L, _I, _P],
    'vlfb_spatial_bn_workspace_bytes': [_I],
    'vlfb_spatial_bn_fwd': [_P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _F, _F, _P, C.c_size_t, _P],
    'vlfb_spatial_bn_infer': [_P, _P, _P, _P, _P, _P, _L, _I, _F, _P, C.c_size_t, _P],
    'vlfb_spatial_bn_bwd': [_P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _P, C.c_size_t, _P],
    'vlfb_maxpool3d_fwd': [_P, _P, _P, _GP, _P],
    'vlfb_maxpool3d_bwd': [_P, _P, _P, _GP, _P],
    'vlfb_maxpool3d_bwd_gather': [_P, _P, _P, _P, _GP, _I, _P],
    'vlfb_avgpool3d_fwd': [_P, _P, _GP, _P],
    'vlfb_avgpool3d_bwd': [_P, _P, _GP, _I, _P],
    'vlfb_roi_align_fwd': [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _P],
    'vlfb_roi_align_bwd': [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _P],
    'vlfb_roi_align_table': [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _I, _P],
    'vlfb_softmax_fwd': [_P, _P, _L, _I, _F, _I, _P],
    'vlfb_softmax_bwd': [_P, _P, _P, _L, _I, _F, _I, _P],
    'vlfb_layernorm_fwd': [_P, _P, _P, _P, _L, _I, _F, _P],
    'vlfb_layernorm_bwd': [_P, _P, _P, _P, _L, _I, _P],
    'vlfb_relu_fwd': [_P, _P, _L, _P],
    'vlfb_relu_bwd': [_P, _P, _P, _L, _P],
    'vlfb_axpby': [_P, _F, _P, _F, _P, _L, _P],
    'vlfb_fill': [_P, _F, _L, _P],
    'vlfb_round_tf32': [_P, _P, _L, _P],
    'vlfb_add_tf32': [_P, _P, _P, _L, _P],
    'vlfb_relu_tf32': [_P, _P, _L, _P],
    'vlfb_relu_bits': [_P, _P, _L, _P],
    'vlfb_relu_bwd_tf32': [_P, _P, _P, _L, _P],
    'vlfb_add_relu_bwd_tf32': [_P, _P, _P, _P, _L, _P],
    'vlfb_colsum_workspace_bytes': [_L, _I],
    'vlfb_colsum': [_P, _L, _P, _L, _I, _I, _P, C.c_size_t, _P],
    'vlfb_sigmoid_fwd': [_P, _P, _L, _P],
    'vlfb_dropout_fwd': [_P, _P, _L, _F, _U, _U, _P, _P],
    'vlfb_copy2d': [_P, _L, _P, _L, _L, _I, _I, _P],
    'vlfb_nc_to_cl': [_P, _P, _I, _I, _L, _I, _P],
    'vlfb_nc_to_cl_round': [_P, _P, _I, _I, _L, _I, _I, _P],
    'vlfb_nc_to_cl_pitched': [_P, _P, _I, _I, _L, _I, _I, _I, _I, _I, _P],
    'vlfb_cl_to_nc': [_P, _P, _I, _I, _L, _I, _P],
    'vlfb_weight_transpose': [_P, _P, _P, _I, _I, _I, _P],
    'vlfb_weight_transpose_multi': [_P, _I, _I, _P],
    'vlfb_sigmoid_ce_fwd': [_P, _P, _P, _L, _F, _P],
    'vlfb_sigmoid_ce_bwd': [_P, _P, _P, _P, _L, _F, _P],
    'vlfb_softmax_ce_fwd': [_P, _P, _P, _P, _I, _I, _F, _P],
    'vlfb_softmax_ce_bwd': [_P, _P, _P, _I, _I, _F, _P],
    'vlfb_sgd_nesterov': [_P, _P, _P, _P, _L, _P, _F, _F, _I, _P],
    'vlfb_fbo_nl_scratch_floats': [C.POINTER(FboCfg)],
    'vlfb_fbo_nl_fwd': [C.POINTER(FboCfg), C.POINTER(FboLayer), _P, _P, _P],
    'vlfb_fbo_nl_bwd': [C.POINTER(FboCfg), C.POINTER(FboLayer), _P, _P, _P, _P, _P, _P, C.c_size_t, _P],
    'vlfb_fbo_bank_scan_splits': [_I, _I, _I],
    'vlfb_fbo_bank_scan_workspace': [_I, _I, _I],
    'vlfb_fbo_bank_scan': [_P, _P, _F, _P, _P, _I, _I, _I, _I, _P, C.c_size_t, _P],
    'vlfb_fbo_bank_scan_splits_dt': [_I, _I, _I, _I],
    'vlfb_fbo_bank_scan_workspace_dt': [_I, _I, _I, _I],
    'vlfb_fbo_bank_scan_dt': [_P, _I, _P, _F, _P, _P, _I, _I, _I, _I, _P, C.c_size_t, _P],
    'vlfb_cast_f32_to_bf16': [_P, _P, _L, _P],
    'vlfb_lfb_gather': [_P, _L, _P, _P, _L, _I, _I, _P],
}
RESTYPES = {'vlfb_last_error': C.c_char_p, 'vlfb_fbo_bank_scan_workspace': C.c_size_t,
            'vlfb_fbo_bank_scan_workspace_dt': C.c_size_t,
            'vlfb_fbo_nl_scratch_floats': C.c_size_t,
            'vlfb_gemm_workspace_bytes': C.c_size_t, 'vlfb_colsum_workspace_bytes': C.c_size_t, 'vlfb_spatial_bn_workspace_bytes': C.c_size_t}

_lib = None


def load():
    """Load libvlfb.so and declare every prototype.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            'libvlfb.so not found at %s -- build it first (python -c "import __graft_entry__ as g; '
            'g.build()" or make -C csrc).  There is no CPU fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError if the symbol is missing
        fn.argtypes = argtypes
        fn.restype = RESTYPES.get(name, C.c_int)
    _lib = lib
    return lib


class VlfbError(RuntimeError):
    pass


def check(rc, what):
    if rc != 0:
        msg = load().vlfb_last_error()
        raise VlfbError('%s failed (%d): %s' % (what, rc, msg.decode() if msg else ''))
