"""ctypes binding of libt2r_b200.so (the C-ABI declared in include/t2r_b200.h).

The library is the product: there is no CPU or PyTorch fallback.  `lib()` raises if the shared
object has not been built (`python -c "import __graft_entry__ as g; g.build()"`), and every
wrapper raises `T2RError` with the library's own message on a non-zero status.
"""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libt2r_b200.so')

T2R_EPI_BIAS, T2R_EPI_RESIDUAL, T2R_EPI_RELU, T2R_EPI_OUT_F32 = 1, 2, 4, 8
T2R_DT_FLOAT, T2R_DT_INT64, T2R_DT_BYTES = 1, 2, 3


class T2RError(RuntimeError):
  pass


class ConvDesc(C.Structure):
  _fields_ = [('struct_size', C.c_uint32), ('N', C.c_int32), ('H', C.c_int32), ('W', C.c_int32),
              ('Cin', C.c_int32), ('Cout', C.c_int32), ('KH', C.c_int32), ('KW', C.c_int32),
              ('stride', C.c_int32), ('pad_top', C.c_int32), ('pad_left', C.c_int32),
              ('Ho', C.c_int32), ('Wo', C.c_int32), ('flags', C.c_int32)]


class DistortParams(C.Structure):
  _fields_ = [('brightness_delta', C.c_float), ('saturation_scale', C.c_float),
              ('hue_delta', C.c_float), ('contrast_scale', C.c_float), ('noise_stddev', C.c_float),
              ('crop_y', C.c_int32), ('crop_x', C.c_int32), ('reserved', C.c_int32)]


class JpegInfo(C.Structure):
  """T2RJpegInfo (include/t2r_b200.h)."""
  _fields_ = [('struct_size', C.c_uint32), ('width', C.c_int32), ('height', C.c_int32), ('ncomp', C.c_int32),
              ('comp_id', C.c_int32 * 3), ('h', C.c_int32 * 3), ('v', C.c_int32 * 3), ('tq', C.c_int32 * 3),
              ('hmax', C.c_int32), ('vmax', C.c_int32), ('mcux', C.c_int32), ('mcuy', C.c_int32),
              ('restart_interval', C.c_int32), ('reserved', C.c_int32), ('coef_offset', C.c_int64 * 3),
              ('coef_count', C.c_int64), ('qt', (C.c_uint16 * 64) * 4)]


class LossSegment(C.Structure):
  """T2RLossSegment (include/t2r_b200.h)."""
  _fields_ = [('struct_size', C.c_uint32), ('kind', C.c_int32), ('predictions', C.c_void_p), ('labels', C.c_void_p),
              ('row_mask', C.c_void_p), ('dpredictions', C.c_void_p), ('sigmoid_out', C.c_void_p), ('n', C.c_int64),
              ('cols', C.c_int32), ('row_mod', C.c_int32), ('row_mask_is_complement', C.c_int32), ('in_total', C.c_int32),
              ('weight', C.c_float), ('delta', C.c_float), ('label_const', C.c_float), ('reserved', C.c_float)]


T2R_LOSS_HUBER, T2R_LOSS_MSE, T2R_LOSS_SIGMOID_LOG, T2R_MAX_LOSS_SEGMENTS = 0, 1, 2, 16


class FeaturePlan(C.Structure):
  _fields_ = [('key', C.c_char_p), ('dtype', C.c_int32), ('count', C.c_int32),
              ('required', C.c_int32), ('dst', C.c_void_p), ('dst_len', C.c_void_p),
              ('pad_float', C.c_float), ('pad_int64', C.c_int64)]


_P, _I32, _I64, _U64, _F = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float
_CD = C.POINTER(ConvDesc)

# name -> (restype, argtypes); status-returning functions have restype int32.
_PROTOS = {
    't2r_version': (_I32, []),
    't2r_last_error': (C.c_char_p, []),
    't2r_launch_count': (_I64, []),
    't2r_launch_count_reset': (None, []),
    't2r_conv_same_padding': (_I32, [_I32, _I32, _I32, C.POINTER(_I32), C.POINTER(_I32)]),
    't2r_conv2d_fprop': (_I32, [_CD, _P, _P, _P, _P, _P, _P]),
    't2r_conv2d_fprop_stats': (_I32, [_CD, _P, _P, _P, _P, _P, _P, _P]),
    't2r_conv2d_dgrad': (_I32, [_CD, _P, _P, _P, _I32, _P]),
    't2r_conv2d_wgrad': (_I32, [_CD, _P, _P, _P, _P]),
    't2r_conv2d_fprop_bnrelu': (_I32, [_CD, _P, _P, _P, _P, _P, _P, _P, _P]),
    't2r_conv2d_wgrad_bnrelu': (_I32, [_CD, _P, _P, _P, _P, _P, _P]),
    't2r_conv2d_dgrad_bnrelu': (_I32, [_CD, _P, _P, _P, _P, _P, _P, _I32, _P, _P]),
    't2r_conv2d_wgrad_bnsums': (_I32, [_CD, _P, _P, _P, _P, _P, _P, _P, _P]),
    't2r_conv2d_dgrad_bnapply_supported': (_I32, [_CD]),
    't2r_conv2d_dgrad_bnapply': (_I32, [_CD, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    't2r_bn_backward_gemm_finalize': (_I32, [_P, _I64, _I32, _P, _P, _P, _P, _P, _P, _P]),
    't2r_pack_weights': (_I32, [_P, _P, _P, _I32, _I32, _I32, _P]),
    't2r_hp_split3': (_I32, [_P, _P, _I64, _I32, _P]),
    't2r_hp_pack_weights3': (_I32, [_P, _P, _I32, _I32, _I32, _P]),
    't2r_maxpool_f32_fwd': (_I32, [_P, _P] + [_I32] * 10 + [_P]),
    't2r_global_mean_f32_fwd': (_I32, [_P, _P, _I32, _I32, _I32, _P]),
    't2r_add_context_f32_fwd': (_I32, [_P, _P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_add_f32': (_I32, [_P, _P, _P, _I64, _P]),
    't2r_im2col_small_cin': (_I32, [_CD, _P, _P, _I32, _P]),
    't2r_pad_nhwc3_c4': (_I32, [_P, _P] + [_I32] * 7 + [_P]),
    't2r_stem_conv_fprop': (_I32, [_CD, _P, _I32, _I32, _P, _P, _P, _P]),
    't2r_stem_conv_wgrad': (_I32, [_CD, _P, _I32, _I32, _P, _P, _P]),
    't2r_stem_mask_grad': (_I32, [_P, _I32, _I32, _I32, _I32, _P]),
    't2r_stem_k': (_I32, [_I32, _I32, _I32]),
    't2r_stem_pack_image': (_I32, [_P, _P] + [_I32] * 9 + [_P]),
    't2r_sgemm': (_I32, [_I32, _I32, _I32, _I32, _I32, _F, _P, _I32, _P, _I32, _F, _P, _I32, _P]),
    't2r_bias_add_f32': (_I32, [_P, _P, _I64, _I32, _P]),
    't2r_colsum_f32': (_I32, [_P, _P, _I64, _I32, _P]),
    't2r_sumsq_f32': (_I32, [_P, _P, _I64, _F, _P]),
    't2r_cast_f32_to_bf16': (_I32, [_P, _P, _I64, _P]),
    't2r_add_context_affine_fwd': (_I32, [_P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _P]),
    't2r_npairs_loss': (_I32, [_P, _P, _I32, _I32, C.c_float, _P, _P, _P, _P, _P, _P]),
    't2r_triplet_semihard_loss': (_I32, [_P, _P, _I32, _I32, C.c_float, _P, _P, _P, _P]),
    't2r_relu_fwd_bf16': (_I32, [_P, _P, _I64, _P]),
    't2r_fold_bn_weights': (_I32, [_P, _P, _P, _I32, _I64, _P]),
    't2r_cast_bf16_to_f32': (_I32, [_P, _P, _I64, _P]),
    't2r_bn_stats': (_I32, [_P, _I64, _I32, _P, _P]),
    't2r_colsum_bf16': (_I32, [_P, _I64, _I32, _P, _P, _P]),
    't2r_bn_finalize': (_I32, [_P, _I64, _I32, _P, _P, _F, _F, _P, _P, _P, _P, _P, _P, _P]),
    't2r_bn_infer_params': (_I32, [_I32, _P, _P, _P, _P, _F, _P, _P, _P]),
    't2r_bn_apply': (_I32, [_P, _P, _I64, _I32, _P, _P, _P, _I64, _I32, _P]),
    't2r_bn_backward': (_I32, [_P, _P, _P, _P, _I64, _I32, _P, _P, _P, _P, _P, _I32, _P, _P, _P, _P]),
    't2r_bn_backward_presummed': (_I32, [_P, _P, _P, _P, _I64, _I32, _P, _P, _P, _P, _I32, _P, _P, _P, _P]),
    't2r_spatial_softmax_fwd': (_I32, [_P, _P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_spatial_softmax_bwd': (_I32, [_P, _P, _P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_bn_film_backward': (_I32, [_P, _P, _P, _P, _P, _P, _I64, _I32, _I64, _P, _P, _P, _P, _I32, _P, _P, _P, _P]),
    't2r_maxpool_fwd': (_I32, [_P, _P, _P] + [_I32] * 10 + [_P]),
    't2r_maxpool_bwd': (_I32, [_P, _P, _P] + [_I32] * 10 + [_P]),
    't2r_global_mean_fwd': (_I32, [_P, _P, _I32, _I32, _I32, _P]),
    't2r_global_mean_bwd': (_I32, [_P, _P, _I32, _I32, _I32, _P]),
    't2r_add_context_fwd': (_I32, [_P, _P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_add_context_bwd': (_I32, [_P, _P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_add_bf16': (_I32, [_P, _P, _P, _I64, _P]),
    't2r_add_relu_bf16': (_I32, [_P, _P, _P, _I64, _P]),
    't2r_relu_bwd_bf16': (_I32, [_P, _P, _P, _I64, _P]),
    't2r_crop_convert_distort': (_I32, [_P, _P, _P, _P] + [_I32] * 7 + [_U64, _U64, _P]),
    't2r_distort_f32': (_I32, [_P, _P, _P, _P] + [_I32] * 4 + [_U64, _U64, _P]),
    't2r_channel_gamma_f32': (_I32, [_P, _P, _I64, _I32, _F, _F, _F, _F, _P]),
    't2r_depth_distort_f32': (_I32, [_P, _P, _I64, _F, _F, _F, _F, _U64, _U64, _P]),
    't2r_resize_bilinear_legacy': (_I32, [_P, _P] + [_I32] * 6 + [_P]),
    't2r_sigmoid_logloss': (_I32, [_P, _P, _P, _P, _P, _I64, _P]),
    't2r_sigmoid_f32': (_I32, [_P, _P, _I64, _P]),
    't2r_cem_sample': (_I32, [_P, _P, _P, _I32, _I32, _I32, _U64, _U64, _P]),
    't2r_cem_refit': (_I32, [_P, _P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_bellman_target': (_I32, [_P, _P, _P, _F, _P, _I64, _P]),
    't2r_momentum_step': (_I32, [_P, _P, _P, _P, _P, _I64, _I64, _F, _F, _F, _F, _F, _P]),
    't2r_adam_step': (_I32, [_P, _P, _P, _P, _P, _P, _I64, _I64, _F, _F, _F, _F, _I64, _F, _F, _F, _P]),
    't2r_rmsprop_step': (_I32, [_P, _P, _P, _P, _P, _P, _I64, _I64, _F, _F, _F, _F, _F, _F, _F, _P]),
    't2r_mixup_reverse_f32': (_I32, [_P, _P, _I32, _I64, _F, _P]),
    't2r_weighted_losses': (_I32, [C.POINTER(LossSegment), _I32, _P, _P]),
    't2r_crc32c': (C.c_uint32, [_P, _U64]),
    't2r_masked_crc32c': (C.c_uint32, [_P, _U64]),
    't2r_tfrecord_index': (_I64, [_P, _U64, _P, _P, _I64, _I32]),
    't2r_example_parse_batch': (_I32, [_P, _P, _I32, C.POINTER(FeaturePlan), _I32]),
    't2r_jpeg_parse': (_I32, [_P, C.c_uint64, C.POINTER(JpegInfo)]),
    't2r_jpeg_entropy_decode_batch': (_I32, [_P, _P, _I32, C.POINTER(JpegInfo), _P, _I64]),
    't2r_jpeg_decode_host_batch': (_I32, [_P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_jpeg_idct_color': (_I32, [_P, _P, C.POINTER(JpegInfo), _P, _P, _I32, _I64, _I32, _P]),
    't2r_conv2d_direct_f32_fwd': (_I32, [_P, _P, _P, _P] + [_I32] * 12 + [_P]),
    't2r_conv2d_direct_f32_dgrad': (_I32, [_P, _P, _P] + [_I32] * 12 + [_P]),
    't2r_conv2d_direct_f32_wgrad': (_I32, [_P, _P, _P] + [_I32] * 12 + [_P]),
    't2r_layer_norm_f32_fwd': (_I32, [_P, _P, _P, _P, _P, _P, _I32, _I32, _I32, _F, _I32, _P]),
    't2r_layer_norm_f32_bwd': (_I32, [_P] * 9 + [_I32, _I32, _I32, _I32, _P]),
    't2r_spatial_softmax_f32_fwd': (_I32, [_P, _P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_spatial_softmax_f32_bwd': (_I32, [_P, _P, _P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_tile_add_context_f32_fwd': (_I32, [_P, _P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_tile_add_context_f32_bwd': (_I32, [_P, _P, _P, _I32, _I32, _I32, _I32, _P]),
    't2r_pcgrad_project': (_I32, [_P, _I32, _I64, _P, _P, _P, _I32, _F, _P, _P, _P, _P]),
    't2r_elu_f32_fwd': (_I32, [_P, _P, _I64, _P]),
    't2r_elu_f32_bwd': (_I32, [_P, _P, _P, _I64, _P]),
    't2r_bn_infer_f32_fwd': (_I32, [_P, _P, _P, _P, _P, _P, _I64, _I32, _F, _P]),
    't2r_bn_infer_f32_bwd': (_I32, [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _I32, _F, _P]),
    't2r_bn_train_f32_fwd': (_I32, [_P] * 8 + [_I64, _I32, _F, _F, _I32, _P]),
    't2r_bn_train_f32_bwd': (_I32, [_P] * 9 + [_I64, _I32, _I32, _P]),
    't2r_film_relu_f32_fwd': (_I32, [_P, _P, _P, _I32, _I32, _I32, _P]),
    't2r_film_relu_f32_bwd': (_I32, [_P, _P, _P, _P, _P, _I32, _I32, _I32, _P]),
    't2r_relu_f32_fwd': (_I32, [_P, _P, _I64, _P]),
    't2r_relu_f32_bwd': (_I32, [_P, _P, _P, _I64, _P]),
    't2r_sequence_example_parse_batch': (_I32, [_P, _P, _I32, C.POINTER(FeaturePlan), _I32, _I32, _P]),
}

# Functions whose int return value is a status code (checked by `call`).
_STATUS = {n for n, (r, _) in _PROTOS.items()
           if r is _I32 and n not in ('t2r_version', 't2r_stem_k', 't2r_conv2d_dgrad_bnapply_supported')}

EXPORTED_SYMBOLS = tuple(sorted(_PROTOS))

_lib = None
_lock = threading.Lock()


def lib():
  """Loads libt2r_b200.so (once).  Raises T2RError when it has not been built."""
  global _lib
  if _lib is not None:
    return _lib
  with _lock:
    if _lib is None:
      if not os.path.exists(LIB_PATH):
        raise T2RError(
            'libt2r_b200.so is missing at %s: build it with `python -c "import '
            '__graft_entry__ as g; g.build()"` (or `make -C tensor2robot_b200/csrc`). There is '
            'no CPU fallback.' % LIB_PATH)
      handle = C.CDLL(LIB_PATH)
      for name, (restype, argtypes) in _PROTOS.items():
        fn = getattr(handle, name)
        fn.restype = restype
        fn.argtypes = argtypes
      _lib = handle
  return _lib


def last_error():
  msg = lib().t2r_last_error()
  return msg.decode('utf-8', 'replace') if msg else ''


def call(name, *args):
  """Calls a status-returning entry point and raises T2RError on failure."""
  rc = getattr(lib(), name)(*args)
  if name in _STATUS and rc != 0:
    raise T2RError('%s failed (status %d): %s' % (name, rc, last_error()))
  return rc


def launch_count():
  return int(lib().t2r_launch_count())


def same_padding(size, k, stride):
  """TF SAME padding: returns (out, pad_before)."""
  out, pad = C.c_int32(), C.c_int32()
  call('t2r_conv_same_padding', size, k, stride, C.byref(out), C.byref(pad))
  return out.value, pad.value


def current_stream_ptr():
  """cudaStream_t of torch's current stream on the current device as a ctypes pointer.  torch.cuda.current_stream() builds
  a Python Stream object through several layers of device-index resolution (~16 us: 2.5 ms of a 13.5 ms BC-Z step with
  its ~150 kernel launches); the raw accessor behind it costs well under a microsecond."""
  import torch
  try:
    return C.c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))   # pylint: disable=protected-access
  except AttributeError:      # a torch build without the raw accessors
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
