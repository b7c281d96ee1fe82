"""ctypes binding of libctb200.so (the C ABI declared in include/ctb200.h).

The product path has NO CPU fallback: if the library cannot be loaded, or a call fails, a
RuntimeError is raised with ct_last_error().
"""
import ctypes as C
import glob
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libctb200.so')
CSRC = os.path.join(_HERE, 'csrc')
SOURCES = ['api.cu', 'conv_simt.cu', 'conv_tc.cu', 'conv_halo.cu', 'elementwise.cu', 'decode.cu', 'stream.cu']

# ---- enums (mirror include/ctb200.h) ----
CT_F32, CT_BF16 = 0, 1
CT_A_CONV, CT_A_DCN, CT_A_DCN_WIN = 0, 1, 2
CT_OUT_NHWC, CT_OUT_NHWC_F32, CT_OUT_NCHW_F32, CT_OUT_NHWC_S2D = 0, 1, 2, 3
CT_HEAD_NONE, CT_HEAD_SIGMOID, CT_HEAD_DEPTH = 0, 1, 2
CT_ENGINE_SIMT, CT_ENGINE_TCGEN05, CT_ENGINE_TCGEN05_HALO, CT_ENGINE_TCGEN05_X3 = 0, 1, 2, 3
CT_ROLE_RAW, CT_ROLE_REG, CT_ROLE_WH, CT_ROLE_LTRB, CT_ROLE_LTRB_AMODAL, CT_ROLE_HPS = range(6)
CT_DECODE_MAX_HEADS = 12
CT_REC_SCORE, CT_REC_CLS, CT_REC_XS, CT_REC_YS, CT_REC_BBOX, CT_REC_IND, CT_REC_HEADS = 0, 1, 2, 3, 4, 8, 9


class ConvDesc(C.Structure):
  _fields_ = [
      ('engine', C.c_int32), ('dtype', C.c_int32), ('a_mode', C.c_int32),
      ('B', C.c_int32), ('H', C.c_int32), ('W', C.c_int32),
      ('C_in', C.c_int32), ('ld_in', C.c_int32), ('C_out', C.c_int32),
      ('KH', C.c_int32), ('KW', C.c_int32), ('stride', C.c_int32), ('pad', C.c_int32),
      ('OH', C.c_int32), ('OW', C.c_int32), ('ld_out', C.c_int32), ('out_mode', C.c_int32),
      ('relu', C.c_int32), ('ld_res', C.c_int32), ('head_act', C.c_int32),
      ('sig_from', C.c_int32), ('depth_scale', C.c_float), ('ld_om', C.c_int32),
      ('n_tile', C.c_int32), ('epilogue_sum3', C.c_int32), ('pad_w1', C.c_int32),
      ('x', C.c_void_p), ('w', C.c_void_p), ('shift', C.c_void_p), ('residual', C.c_void_p),
      ('om', C.c_void_p), ('out', C.c_void_p),
  ]


class DecodeHead(C.Structure):
  _fields_ = [('map', C.c_void_p), ('channels', C.c_int32), ('role', C.c_int32),
              ('rec_offset', C.c_int32)]


class DecodeDesc(C.Structure):
  _fields_ = [
      ('B', C.c_int32), ('C', C.c_int32), ('H', C.c_int32), ('W', C.c_int32), ('K', C.c_int32),
      ('hm', C.c_void_p), ('n_heads', C.c_int32),
      ('heads', DecodeHead * CT_DECODE_MAX_HEADS),
      ('hm_hp', C.c_void_p), ('hp_offset', C.c_void_p), ('J', C.c_int32),
      ('rec_hps', C.c_int32), ('rec_kps_score', C.c_int32), ('rec_floats', C.c_int32),
      ('has_bbox', C.c_int32), ('records', C.c_void_p), ('workspace', C.c_void_p),
  ]


CT_TRK_SCORE, CT_TRK_CLASS, CT_TRK_CT, CT_TRK_TRACKING, CT_TRK_BBOX, CT_TRK_ID, CT_TRK_AGE, CT_TRK_ACTIVE = \
    0, 1, 2, 4, 6, 10, 11, 12
CT_TRK_FLOATS = 13


class TrackDesc(C.Structure):
  _fields_ = [
      ('B', C.c_int32), ('K', C.c_int32), ('F', C.c_int32), ('rec_tracking', C.c_int32),
      ('max_tracks', C.c_int32), ('out_thresh', C.c_float), ('new_thresh', C.c_float), ('pre_thresh', C.c_float),
      ('max_age', C.c_int32), ('inp_h', C.c_int32), ('inp_w', C.c_int32),
      ('records', C.c_void_p), ('trans_out_inv', C.c_void_p), ('trans_input', C.c_void_p),
      ('tracks', C.c_void_p), ('counts', C.c_void_p), ('boxes', C.c_void_p),
      ('assign', C.c_int32), ('public_det', C.c_void_p), ('public_count', C.c_void_p), ('max_public', C.c_int32),
  ]


CT_ASSIGN_GREEDY, CT_ASSIGN_HUNGARIAN = 0, 1


EXPORTS = ['ct_packed_weight_bytes', 'ct_pack_weights', 'ct_conv_forward', 'ct_stem_forward',
           'ct_pack_stem_input', 'ct_pack_stem_input_f32', 'ct_maxpool2', 'ct_maxpool2_s2d', 'ct_upsample_add', 'ct_decode_workspace_bytes', 'ct_decode',
           'ct_render_pre_hm', 'ct_track_smem_bytes', 'ct_track_step', 'ct_render_tracks', 'ct_flip_merge',
           'ct_warp_affine_normalize', 'ct_last_error', 'ct_abi_version', 'ct_launch_count',
           'ct_reset_launch_count', 'ct_debug_trace', 'ct_debug_watch']

NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-shared', '-Xcompiler', '-fPIC']


def build(force=False, verbose=False):
  """Compile libctb200.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
  srcs = [os.path.join(CSRC, s) for s in SOURCES]
  deps = srcs + glob.glob(os.path.join(CSRC, '*.cuh')) + [os.path.join(_HERE, '..', 'include', 'ctb200.h')]
  if not force and os.path.exists(LIB_PATH) and \
      all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps):
    return LIB_PATH
  cmd = ['nvcc'] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-o', LIB_PATH] + srcs
  r = subprocess.run(cmd, capture_output=True, text=True)
  if r.returncode != 0:
    raise RuntimeError('nvcc failed:\n' + r.stdout + r.stderr)
  if verbose:
    print(r.stderr)
  return LIB_PATH


_lib = None


def lib():
  """Load the shared library (raises if it is missing -- there is no fallback)."""
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.exists(LIB_PATH):
    raise RuntimeError(
        'centertrack_b200: %s not found. Build it with `python -c "import __graft_entry__ as g; '
        'g.build()"` (nvcc, sm_100a). There is no CPU fallback.' % LIB_PATH)
  L = C.CDLL(LIB_PATH)
  L.ct_last_error.restype = C.c_char_p
  L.ct_packed_weight_bytes.restype = C.c_int64
  L.ct_packed_weight_bytes.argtypes = [C.c_int32] * 6
  L.ct_pack_weights.argtypes = [C.c_int32, C.c_void_p] + [C.c_int32] * 5 + [C.c_void_p]
  L.ct_conv_forward.argtypes = [C.POINTER(ConvDesc), C.c_void_p]
  L.ct_stem_forward.argtypes = [C.c_void_p] * 6 + [C.c_int32] * 5 + [C.c_void_p]
  L.ct_pack_stem_input.argtypes = [C.c_void_p] * 4 + [C.c_int32] * 3 + [C.c_void_p]
  L.ct_pack_stem_input_f32.argtypes = [C.c_void_p] * 4 + [C.c_int32] * 3 + [C.c_void_p]
  L.ct_maxpool2.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int32] * 7 + [C.c_void_p]
  L.ct_maxpool2_s2d.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int32] * 7 + [C.c_void_p]
  L.ct_upsample_add.argtypes = [C.c_void_p] * 4 + [C.c_int32] * 9 + [C.c_void_p]
  L.ct_decode_workspace_bytes.restype = C.c_int64
  L.ct_decode_workspace_bytes.argtypes = [C.c_int32] * 4
  L.ct_decode.argtypes = [C.POINTER(DecodeDesc), C.c_void_p]
  L.ct_render_pre_hm.argtypes = [C.c_void_p, C.c_int32, C.c_void_p] + [C.c_int32] * 3 + [C.c_void_p]
  L.ct_track_smem_bytes.restype = C.c_int64
  L.ct_track_smem_bytes.argtypes = [C.c_int32] * 2
  L.ct_track_step.argtypes = [C.POINTER(TrackDesc), C.c_void_p]
  L.ct_render_tracks.argtypes = [C.c_void_p, C.c_int32, C.c_void_p] + [C.c_int32] * 3 + [C.c_void_p]
  L.ct_flip_merge.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int32] * 3 + [C.c_void_p, C.c_void_p, C.c_void_p]
  L.ct_warp_affine_normalize.argtypes = [C.c_void_p] + [C.c_int32] * 4 + [C.c_void_p] * 4 + [C.c_int32] * 2 + [C.c_void_p]
  L.ct_launch_count.restype = C.c_int64
  L.ct_reset_launch_count.restype = None
  L.ct_debug_trace.argtypes = [C.c_void_p]
  L.ct_debug_watch.argtypes = [C.c_void_p]
  if L.ct_abi_version() != 1:
    raise RuntimeError('libctb200 ABI mismatch')
  _lib = L
  return L


def check(status, what=''):
  if status != 0:
    raise RuntimeError('libctb200 %s failed (%d): %s' %
                       (what, status, lib().ct_last_error().decode('utf-8', 'replace')))


def stream_ptr():
  import torch
  return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
  return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)
