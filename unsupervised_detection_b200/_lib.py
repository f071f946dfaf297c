"""ctypes binding of libcis_b200.so (C ABI in include/cis_b200.h).

The product path has NO fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CIS_LIB_NAME: developer switch to the trace build (make -C csrc trace); the default is the product library
LIB_PATH = os.path.join(_HERE, os.environ.get('CIS_LIB_NAME', 'libcis_b200.so'))

MAX_TAPS, MAX_SRC = 49, 4
ACT_NONE, ACT_ELU, ACT_LEAKY = 0, 1, 2


class CisSrc(C.Structure):
    _fields_ = [('ptr', C.c_void_p), ('pitch', C.c_int32), ('c_off', C.c_int32), ('chunks', C.c_int32), ('n_mod', C.c_int32)]


class CisParamJob(C.Structure):
    _fields_ = [('kind', C.c_int32), ('i', C.c_int32 * 8), ('n', C.c_int64), ('p', C.c_void_p * 8)]


JOB_PACK, JOB_PACK_TILED, JOB_UNPACK, JOB_BN_FOLD, JOB_BN_CHAIN = range(5)


class CisSub(C.Structure):
    _fields_ = [('tap0', C.c_int32), ('ntaps', C.c_int32), ('hoy', C.c_int32), ('hox', C.c_int32), ('OH', C.c_int32), ('OW', C.c_int32),
                ('oa', C.c_int32), ('ob', C.c_int32), ('wpack', C.c_void_p)]


class CisConv(C.Structure):
    _fields_ = [('N', C.c_int32), ('H', C.c_int32), ('W', C.c_int32), ('OH', C.c_int32), ('OW', C.c_int32),
                ('sh', C.c_int32), ('sw', C.c_int32), ('ntaps', C.c_int32),
                ('dh', C.c_int16 * MAX_TAPS), ('dw', C.c_int16 * MAX_TAPS),
                ('nsrc', C.c_int32), ('src', CisSrc * MAX_SRC),
                ('wpack', C.c_void_p), ('K_pad', C.c_int32), ('BN', C.c_int32), ('n_tiles', C.c_int32),
                ('bias', C.c_void_p), ('act', C.c_int32), ('alpha', C.c_float),
                ('DH', C.c_int32), ('DW', C.c_int32), ('osh', C.c_int32), ('osw', C.c_int32), ('oa', C.c_int32), ('ob', C.c_int32),
                ('out', C.c_void_p), ('out_pitch', C.c_int32), ('out_coff', C.c_int32), ('out_ch', C.c_int32),
                ('outf', C.c_void_p), ('outf_pitch', C.c_int32), ('outf_coff', C.c_int32), ('outf_ch', C.c_int32),
                ('add_pre', C.c_void_p), ('add_pre_pitch', C.c_int32), ('add_pre_coff', C.c_int32),
                ('addf_pre', C.c_void_p), ('addf_pitch', C.c_int32), ('addf_coff', C.c_int32),
                ('add_post', C.c_void_p), ('add_post_pitch', C.c_int32), ('add_post_coff', C.c_int32),
                ('mode', C.c_int32),
                ('halo', C.c_int32), ('dil', C.c_int32), ('MT', C.c_int32), ('hoy', C.c_int32), ('hox', C.c_int32),
                ('ey', C.c_int32), ('ex', C.c_int32),
                ('splits', C.c_int32), ('sk_scratch', C.c_void_p), ('sk_counters', C.c_void_p),
                ('nph', C.c_int32), ('ph_tap', C.c_int32 * 5), ('sk_cluster', C.c_int32),
                ('nsub', C.c_int32), ('sub', CisSub * 4), ('thin', C.c_int32)]


class CisWgrad(C.Structure):
    _fields_ = [('N', C.c_int32), ('H', C.c_int32), ('W', C.c_int32), ('OH', C.c_int32), ('OW', C.c_int32),
                ('sh', C.c_int32), ('sw', C.c_int32), ('ntaps', C.c_int32),
                ('dh', C.c_int16 * MAX_TAPS), ('dw', C.c_int16 * MAX_TAPS),
                ('nsrc', C.c_int32), ('src', CisSrc * MAX_SRC),
                ('g', C.c_void_p), ('g_pitch', C.c_int32), ('g_coff', C.c_int32), ('g_chunks', C.c_int32),
                ('dwp', C.c_void_p), ('Cout', C.c_int32), ('K_pad', C.c_int32), ('splits', C.c_int32), ('tma', C.c_int32)]


_i32, _i64, _f32, _p, _u64 = C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_uint64

# name -> argtypes (the trailing stream argument is appended automatically)
_PROTOS = {
    'cis_conv_igemm': [C.POINTER(CisConv)],
    'cis_conv_wgrad': [C.POINTER(CisWgrad)],
    'cis_pack_weights': [_p, _p, _i32, _i32, _i32, _i32, _p, _p],
    'cis_pack_weights_tiled': [_p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _i32],
    'cis_unpack_wgrad': [_p, _p, _i32, _i32, _i32, _p, _p, _i32, _i32, _p, _i32],
    'cis_bn_fold': [_p, _p, _p, _p, _i64, _i32, _p, _p],
    'cis_param_multi': [_p, _i32, _i32],
    'cis_bn_chain': [_p, _p, _p, _p, _p, _i64, _i32, _p, _p, _p],
    'cis_dact_mul': [_p, _i32, _i32, _p, _i32, _i32, _p, _i32, _i32, _i64, _i32, _i32, _f32],
    'cis_add_slice': [_p, _i32, _i32, _p, _i32, _i32, _i64, _i32, _i32, _i32],
    'cis_colsum': [_p, _i32, _i32, _i64, _i32, _p, _i32],
    'cis_zero': [_p, _i64],
    'cis_dact_colsum': [_p, _i32, _i32, _p, _i32, _i32, _p, _i32, _i32, _i64, _i32, _i32, _f32, _p, _i32],
    'cis_resize_bilinear_bf16': [_p, _i32, _i32, _i32, _i32, _i32, _p, _i32, _i32, _i32, _i32, _i32],
    'cis_resize_concat_bf16': [C.POINTER(CisSrc), _i32, _i32, _i32, _i32, _p, _i32, _i32, _i32, _i32],
    'cis_resize_concat_bf16_bwd': [_p, _i32, _i32, _i32, _i32, _i32, C.POINTER(CisSrc), C.POINTER(C.c_int32), C.POINTER(C.c_int32), _i32, _i32, _i32],
    'cis_resize_bilinear_bf16_bwd': [_p, _i32, _i32, _i32, _i32, _i32, _p, _i32, _i32, _i32, _i32, _i32, _i32],
    'cis_resize_bilinear_f32': [_p, _i32, _i32, _i32, _i32, _p, _i32, _i32, _f32],
    'cis_upsample_nn2x': [_p, _i32, _i32, _i32, _i32, _p],
    'cis_upsample_nn2x_bwd': [_p, _i32, _i32, _i32, _i32, _p, _i32],
    'cis_crop_resize_bilinear_f32': [_p, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _p, _i32, _i32],
    'cis_resize_nn_f32': [_p, _i32, _i32, _i32, _i32, _p, _i32, _i32],
    'cis_warp_costvol': [_p, _i32, _i32, _p, _i32, _i32, _p, _f32, _i32, _i32, _i32, _i32, _p, _i32, _i32],
    'cis_dense_image_warp': [_p, _i32, _i32, _p, _f32, _i32, _i32, _i32, _i32, _p, _i32],
    'cis_pack_f32_to_bf16': [_p, _i64, _i32, _f32, _p, _i32, _i32],
    'cis_flow_stats': [_p, _i32, _i64, _p],
    'cis_pack_generator_input': [_p, _p, _p, _i32, _i64, _p],
    'cis_mask_apply': [_p, _p, _i32, _i64, _p],
    'cis_charbonnier_sum': [_p, _p, _p, _i32, _i64, _i32, _i32, _f32, _p],
    'cis_cis_loss_fwd': [_p, _p, _p, _i32, _i32, _i32, _i32, _i32, _f32, _p, _p],
    'cis_cis_loss_reduce': [_p, _i32, _i32, _i64, _f32, _p, _p],
    'cis_cis_loss_bwd': [_p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _f32, _i32, _p, _p],
    'cis_resize_f32_bwd_to_bf16': [_p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _i32],
    'cis_mask_bwd': [_p, _p, _p, _p, _i32, _i64, _p],
    'cis_abs_sum': [_p, _i64, _p],
    'cis_grad_avg_abs': [_p, _p, _i32, _p],
    'cis_clip_adam': [_p, _p, _p, _p, _i64, _f32, _f32, _f32, _f32, _f32, _f32, _p, _p, _i32, _u64],
    'cis_cast_f32_to_bf16': [_p, _i64, _p],
    'cis_cast_bf16_to_f32': [_p, _i64, _i32, _i32, _i32, _p],
}
EXPORTS = sorted(list(_PROTOS) + ['cis_last_error', 'cis_version', 'cis_set_persist_mode', 'cis_crc32c', 'cis_host_resize_bilinear_legacy',
                                  'cis_host_bgr8_to_rgb_resized'])

_lib = None


def load():
    """Load the shared library (once).  Fails loudly when it has not been built (`__graft_entry__.build()`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError('libcis_b200.so not built: run `python -c "import __graft_entry__ as g; g.build()"` '
                               '(no CPU fallback exists for the product path)')
        lib = C.CDLL(LIB_PATH)
        lib.cis_last_error.restype = C.c_char_p
        lib.cis_version.restype = C.c_int
        lib.cis_set_persist_mode.argtypes = [C.c_int]
        lib.cis_set_persist_mode.restype = C.c_int
        lib.cis_crc32c.argtypes = [C.c_uint32, C.c_void_p, C.c_size_t]
        lib.cis_crc32c.restype = C.c_uint32
        lib.cis_host_resize_bilinear_legacy.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32]
        lib.cis_host_resize_bilinear_legacy.restype = C.c_int
        lib.cis_host_bgr8_to_rgb_resized.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32]
        lib.cis_host_bgr8_to_rgb_resized.restype = C.c_int
        for name, args in _PROTOS.items():
            fn = getattr(lib, name)
            fn.argtypes = list(args) + [C.c_void_p]
            fn.restype = C.c_int
        _lib = lib
    return _lib


def check(rc, what=''):
    if rc != 0:
        raise RuntimeError('libcis_b200 %s failed (code %d): %s' % (what, rc, load().cis_last_error().decode()))


def call(name, *args):
    """Call an entry point; the last positional argument must be the cudaStream_t handle (int)."""
    check(getattr(load(), name)(*args), name)
