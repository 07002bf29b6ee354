"""ctypes binding of ``include/cae_b200.h`` (the C ABI of the hot path).

The library is built in-tree (``cnn_autoencoder_b200/lib/libcae_b200.so``) by
``cnn_autoencoder_b200/csrc/Makefile`` for sm_100a only.  There is no CPU
fallback: if the library is missing, :func:`lib` raises.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libcae_b200.so')
CSRC = os.path.join(_HERE, 'csrc')

FMT_NONE, FMT_U8_HWC, FMT_F32_NCHW, FMT_F16_PLANAR, FMT_F16_SPLIT = 0, 1, 2, 3, 4
HALO_KEEP, HALO_REFLECT = 0, 1
ACT_NONE, ACT_LEAKY_RELU, ACT_RELU = 0, 1, 2
ABI_VERSION = 4
CONV_S1, CONV_S2, CONVT_S1, CONVT_S2 = 0, 1, 2, 3
PAD_ZERO, PAD_REFLECT = 0, 1

SYMBOLS = ['cae_abi_version', 'cae_last_error', 'cae_device_info', 'cae_launch_count',
           'cae_packed_weight_bytes', 'cae_pack_weights', 'cae_conv_igemm', 'cae_conv_direct',
           'cae_conv_head', 'cae_proj_weight_bytes', 'cae_proj_bytes', 'cae_pack_proj_weights',
           'cae_image_from_proj',
           'cae_nchw_to_planar', 'cae_planar_to_nchw', 'cae_eb_quantize', 'cae_eb_dequantize_planar',
           'cae_eb_train_blob_size', 'cae_eb_train_fwd', 'cae_eb_train_bwd', 'cae_gdn',
           'cae_act_grad', 'cae_conv_wgrad', 'cae_conv_wgrad_workspace_bytes',
           'cae_pmf_to_quantized_cdf', 'cae_rans_encode', 'cae_rans_decode',
           'cae_rans_enc_table_bytes', 'cae_rans_build_enc_table',
           'cae_rans_encode_batch', 'cae_rans_scan', 'cae_rans_compact', 'cae_rans_decode_batch',
           'cae_tiles_upload_u8', 'cae_tiles_download_u8', 'cae_tiles_upload_u8_banded',
           'cae_tiles_download_u8_banded', 'cae_sse_u8', 'cae_ssim_u8', 'cae_delta_e_u8', 'cae_u8_to_planes_f32',
           'cae_avgpool2_planes_f32', 'cae_ssim_gauss_planes_f32', 'cae_tiles_gather_u8', 'cae_files_write', 'cae_files_stat', 'cae_files_read',
           'cae_files_remove', 'cae_tiles_crop_u8', 'cae_tiles_paste_u8',
           'cae_tiles_crop_reduce_u8', 'cae_tiles_pyramid_u8']


class Tensor(ctypes.Structure):
    _fields_ = [('ptr', ctypes.c_void_p), ('fmt', ctypes.c_int32), ('planes', ctypes.c_int32),
                ('halo', ctypes.c_int32), ('reserved', ctypes.c_int32)]


class ConvDesc(ctypes.Structure):
    _fields_ = [('kind', ctypes.c_int32), ('n', ctypes.c_int32), ('h_in', ctypes.c_int32),
                ('w_in', ctypes.c_int32), ('c_in', ctypes.c_int32), ('c_out', ctypes.c_int32),
                ('inp', Tensor), ('out', Tensor), ('skip', Tensor),
                ('weights', ctypes.c_void_p), ('bias', ctypes.c_void_p),
                ('pre_act', ctypes.c_int32), ('post_act', ctypes.c_int32),
                ('pad_mode', ctypes.c_int32), ('ck', ctypes.c_int32), ('mt', ctypes.c_int32),
                ('grid', ctypes.c_int32), ('aux_out', ctypes.c_void_p),
                ('quant', ctypes.c_void_p), ('groups', ctypes.c_int32),
                ('reserved', ctypes.c_int32), ('proj', ctypes.c_void_p)]


class ActGradDesc(ctypes.Structure):
    _fields_ = [('n', ctypes.c_int32), ('h', ctypes.c_int32), ('w', ctypes.c_int32), ('c', ctypes.c_int32),
                ('g', Tensor), ('g_h', ctypes.c_int32), ('g_w', ctypes.c_int32),
                ('g_oy', ctypes.c_int32), ('g_ox', ctypes.c_int32),
                ('fold', ctypes.c_int32), ('fold_shift', ctypes.c_int32),
                ('out', Tensor), ('out_h', ctypes.c_int32), ('out_w', ctypes.c_int32),
                ('act', ctypes.c_int32), ('post_act', ctypes.c_int32),
                ('dz', Tensor), ('dz_h', ctypes.c_int32), ('dz_w', ctypes.c_int32),
                ('dz_oy', ctypes.c_int32), ('dz_ox', ctypes.c_int32),
                ('skip', Tensor), ('gsum', Tensor), ('g2', Tensor),
                ('scale', ctypes.c_void_p), ('db', ctypes.c_void_p)]


class ProjFuse(ctypes.Structure):
    _fields_ = [('weights', ctypes.c_void_p), ('proj', ctypes.c_void_p)]


class HeadDesc(ctypes.Structure):
    _fields_ = [('n', ctypes.c_int32), ('h_in', ctypes.c_int32), ('w_in', ctypes.c_int32),
                ('c_in', ctypes.c_int32), ('c_out', ctypes.c_int32),
                ('inp', Tensor), ('out', Tensor),
                ('w_stem', ctypes.c_void_p), ('b_stem', ctypes.c_void_p),
                ('w_down', ctypes.c_void_p), ('b_down', ctypes.c_void_p),
                ('act_stem', ctypes.c_int32), ('act_down', ctypes.c_int32),
                ('pad_mode', ctypes.c_int32), ('residual', ctypes.c_int32),
                ('w_stem2', ctypes.c_void_p), ('b_stem2', ctypes.c_void_p),
                ('act_mid', ctypes.c_int32), ('reserved', ctypes.c_int32)]


class EbTables(ctypes.Structure):
    _fields_ = [('medians', ctypes.c_void_p), ('lut', ctypes.c_void_p),
                ('lut_min', ctypes.c_int32), ('lut_len', ctypes.c_int32),
                ('mlp', ctypes.c_void_p), ('n_layers', ctypes.c_int32),
                ('mlp_stride', ctypes.c_int32), ('dims', ctypes.c_int32 * 10),
                ('hist_min', ctypes.c_int32), ('hist_bins', ctypes.c_int32),
                ('tail_lik', ctypes.c_float), ('lik_bound', ctypes.c_float)]


class QuantFuse(ctypes.Structure):
    _fields_ = [('tables', EbTables), ('y_q', ctypes.c_void_p), ('symbols', ctypes.c_void_p),
                ('y_q_planar', Tensor), ('hist', ctypes.c_void_p), ('rate_bits', ctypes.c_void_p),
                ('status', ctypes.c_void_p)]


class CaeError(RuntimeError):
    pass


_lib = None


def build(verbose=False):
    """Compile the shared library in-tree with nvcc (sm_100a)."""
    out = subprocess.run(['make', '-C', CSRC, '-j8'], capture_output=True, text=True)
    if out.returncode != 0:
        raise CaeError('building libcae_b200.so failed:\n' + out.stdout + out.stderr)
    if verbose:
        print(out.stdout + out.stderr)
    return LIB_PATH


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CaeError(f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; '
                       f'g.build()"` (there is no CPU fallback for the hot path)')
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_size_t
    L.cae_abi_version.restype = ctypes.c_int
    L.cae_last_error.restype = ctypes.c_char_p
    L.cae_device_info.argtypes = [ctypes.POINTER(ctypes.c_int)] * 3
    L.cae_launch_count.restype = ctypes.c_uint64
    L.cae_packed_weight_bytes.restype = sz
    L.cae_packed_weight_bytes.argtypes = [ctypes.c_int] * 4
    L.cae_pack_weights.argtypes = [ctypes.c_int] * 4 + [vp, vp, vp, vp]
    L.cae_conv_igemm.argtypes = [ctypes.POINTER(ConvDesc), vp]
    L.cae_conv_direct.argtypes = [ctypes.POINTER(ConvDesc), vp]
    L.cae_conv_head.argtypes = [ctypes.POINTER(HeadDesc), vp]
    L.cae_proj_weight_bytes.restype = sz
    L.cae_proj_weight_bytes.argtypes = []
    L.cae_proj_bytes.restype = sz
    L.cae_proj_bytes.argtypes = [ctypes.c_int] * 3
    L.cae_pack_proj_weights.argtypes = [ctypes.c_int, ctypes.c_int, vp, vp, vp, vp]
    L.cae_image_from_proj.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp,
                                      ctypes.c_int, ctypes.c_int, vp, vp, vp]
    L.cae_nchw_to_planar.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     Tensor, vp]
    L.cae_planar_to_nchw.argtypes = [Tensor, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_int, vp, vp]
    L.cae_gdn.argtypes = [Tensor, Tensor, Tensor, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                          ctypes.c_int, vp, vp, ctypes.c_int, vp]
    L.cae_eb_quantize.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                  ctypes.POINTER(EbTables), vp, vp, vp, vp, vp, vp, vp]
    L.cae_pmf_to_quantized_cdf.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp]
    L.cae_rans_encode.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int, vp, vp, vp,
                                  sz, ctypes.POINTER(sz)]
    L.cae_rans_decode.argtypes = [vp, sz, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int, vp, vp,
                                  vp]
    L.cae_rans_enc_table_bytes.restype = sz
    L.cae_rans_enc_table_bytes.argtypes = [ctypes.c_int, ctypes.c_int]
    L.cae_rans_build_enc_table.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp]
    L.cae_rans_encode_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp,
                                        ctypes.c_int, vp, vp, vp, vp, ctypes.c_int, vp, vp, vp]
    L.cae_rans_scan.argtypes = [vp, ctypes.c_int, vp, vp]
    L.cae_rans_compact.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp]
    L.cae_rans_decode_batch.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp,
                                        ctypes.c_int, vp, vp, vp, vp, vp]
    i64 = ctypes.c_int64
    L.cae_eb_dequantize_planar.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, Tensor, vp]
    L.cae_eb_train_blob_size.argtypes = []
    L.cae_eb_train_fwd.argtypes = [vp, vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                   ctypes.c_float, vp, vp, vp]
    L.cae_eb_train_bwd.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                   vp, vp, vp, vp, vp]
    ci = ctypes.c_int
    L.cae_act_grad.argtypes = [ctypes.POINTER(ActGradDesc), vp]
    L.cae_conv_wgrad.argtypes = [ci, ci, ci, ci, ci, ci, Tensor, Tensor, ci, vp, vp, vp, sz, vp]
    L.cae_conv_wgrad_workspace_bytes.restype = sz
    L.cae_conv_wgrad_workspace_bytes.argtypes = []
    L.cae_tiles_upload_u8.argtypes = [vp, i64, i64, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int,
                                      vp, vp]
    L.cae_tiles_download_u8.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, i64,
                                        i64, vp]
    L.cae_tiles_upload_u8_banded.argtypes = [vp, i64, i64, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int,
                                             vp, vp, vp]
    L.cae_tiles_download_u8_banded.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, i64,
                                               i64, vp, vp]
    L.cae_sse_u8.argtypes = [vp, vp, ctypes.c_int, i64, vp, vp]
    L.cae_ssim_u8.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp]
    L.cae_delta_e_u8.argtypes = [vp, vp, ctypes.c_int, i64, vp, vp]
    L.cae_u8_to_planes_f32.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp]
    L.cae_avgpool2_planes_f32.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp]
    L.cae_ssim_gauss_planes_f32.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                            vp, vp, vp]
    L.cae_tiles_gather_u8.argtypes = [vp, i64, i64, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int, vp,
                                      ctypes.c_int]
    L.cae_files_write.argtypes = [ctypes.c_char_p, ctypes.c_int, vp, ctypes.c_int, vp, vp, ctypes.c_int]
    L.cae_files_stat.argtypes = [ctypes.c_char_p, ctypes.c_int, vp, ctypes.c_int]
    L.cae_files_remove.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int]
    L.cae_files_read.argtypes = [ctypes.c_char_p, ctypes.c_int, vp, ctypes.c_int, vp, vp, ctypes.c_int]
    L.cae_tiles_crop_u8.argtypes = [vp, ci, ci, ci, vp, ci, vp, vp, ci, ci, ci, vp]
    L.cae_tiles_paste_u8.argtypes = [vp, ci, ci, ci, vp, ci, vp, vp, ci, ci, ci, vp]
    L.cae_tiles_crop_reduce_u8.argtypes = [vp, ci, ci, ci, ci, vp, ci, vp, vp, ci, ci, ci, vp]
    L.cae_tiles_pyramid_u8.argtypes = [vp, ci, ci, ci, ci, vp, vp, ci, ci, vp, vp]
    for name in SYMBOLS:
        if name not in ('cae_abi_version', 'cae_last_error', 'cae_launch_count',
                        'cae_packed_weight_bytes', 'cae_rans_enc_table_bytes',
                        'cae_proj_weight_bytes', 'cae_proj_bytes',
                        'cae_conv_wgrad_workspace_bytes'):
            getattr(L, name).restype = ctypes.c_int
    if L.cae_abi_version() != ABI_VERSION:
        raise CaeError('libcae_b200.so ABI version mismatch')
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise CaeError(f'[{rc}] ' + lib().cae_last_error().decode())


_replayed = 0


def note_graph_replay(kernels):
    """Kernels of this library launched by replaying a CUDA graph (the library's own counter
    only sees them once, when the graph is captured)."""
    global _replayed
    _replayed += int(kernels)


def launch_count():
    return int(lib().cae_launch_count()) + _replayed
