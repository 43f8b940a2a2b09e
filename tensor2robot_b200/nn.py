"""Functional layer library of the B200 engine: torch tensors in, hand-written sm_100a kernels underneath.

This is the layer vocabulary the reference models are written in (slim.conv2d, slim.batch_norm,
slim.max_pool2d, slim.fully_connected, tf.layers.*; see research/qtopt/networks.py:343-615 and
layers/film_resnet_model.py:39-340), re-expressed over:

  * `VariableStore`  - TF-style named variables ("scope/conv1_1/weights") living in flat fp32
    buffers (parameters, gradients, optimizer slots, EMA) so the optimizer and the NCCL gradient
    all-reduce are each ONE pass over one contiguous buffer (SURVEY 8e, A-24).
  * `torch.autograd.Function`s whose forward/backward call the C-ABI (tensor2robot_b200/_lib.py).
    PyTorch supplies device memory, streams and the autograd tape only; parameter gradients are
    written by the kernels straight into the flat gradient buffer (wgrad accumulates with atomics),
    never through autograd.

Activations are NHWC bf16; the tiny action-context / logit layers run in fp32.
All functions fail loudly without a CUDA device or without libt2r_b200.so.
"""
import collections
import contextlib
import ctypes as C
import math
import os

import numpy as np
import torch

from tensor2robot_b200 import _lib

BF16 = torch.bfloat16
F32 = torch.float32


def _stream():
  return _lib.current_stream_ptr()


def _p(t):
  return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _require_cuda(t, what):
  if not torch.is_tensor(t):
    if hasattr(t, 'materialize'):
      raise _lib.T2RError('%s received a deferred inference op (%s): only batch_norm / conv2d consume those; '
                          'call .materialize() first' % (what, type(t).__name__))
    raise _lib.T2RError('%s expects a CUDA tensor, got %s' % (what, type(t).__name__))
  if not t.is_cuda:
    raise _lib.T2RError('%s: tensor is on %s; the B200 engine has no CPU path' % (what, t.device))


# ---------------------------------------------------------------------------------------------
# variables
# ---------------------------------------------------------------------------------------------
class Variable(object):
  """A named parameter.  `data`/`grad` are fp32 views into the store's flat buffers."""

  def __init__(self, name, shape, trainable, regularize, kind, tf_layout):
    self.name = name
    self.shape = tuple(int(s) for s in shape)
    self.trainable = trainable
    self.regularize = regularize  # receives the slim l2_regularizer gradient
    self.kind = kind              # 'conv' (OHWI weights), 'fc32', 'other'
    self.tf_layout = tf_layout    # how to_tf / from_tf permute: 'hwio', 'io', 'fcgrasp', None
    self.data = None
    self.grad = None
    self.bf16 = None    # bf16 copy in compute layout (conv: OHWI)
    self.dgrad = None   # bf16 [Cin][taps][Cout] for conv layers that need a data gradient
    self.needs_dgrad = False
    self.store = None   # the VariableStore that owns the variable

  def grad_ready(self):
    """Called by a backward kernel wrapper once this variable's gradient is complete in the flat buffer: lets the
    data-parallel reducer start the all-reduce of a finished bucket while the backward pass is still running, and
    catches a trainable variable used twice in one pass (the kernels OVERWRITE .grad, so the TF `reuse=True`
    pattern would silently drop a contribution)."""
    if self.store is not None:
      self.store.grad_ready(self)

  @property
  def numel(self):
    return int(np.prod(self.shape)) if self.shape else 1

  def to_tf(self):
    """numpy array in the reference's (TensorFlow) variable layout."""
    a = self.data.detach().float().cpu().numpy().reshape(self.shape)
    if self.tf_layout == 'hwio':      # ours [Cout,KH,KW,Cin] -> [KH,KW,Cin,Cout]
      return np.ascontiguousarray(a.transpose(1, 2, 3, 0))
    if self.tf_layout == 'io':        # ours [out,in] -> [in,out]
      return np.ascontiguousarray(a.T)
    if self.tf_layout == 'io_hwc':    # ours [out,1,1,in] -> [in,out]
      return np.ascontiguousarray(a.reshape(self.shape[0], -1).T)
    if len(self.shape) == 2 and self.shape[0] == 1 and self.name.endswith(('biases', 'bias')):
      return a[0].copy()            # stored [1, units], the reference has [units]
    return a.copy()

  def from_tf(self, a):
    a = np.asarray(a, dtype=np.float32)
    if self.tf_layout == 'hwio':
      a = a.transpose(3, 0, 1, 2)
    elif self.tf_layout == 'io':
      a = a.T
    elif self.tf_layout == 'io_hwc':
      a = a.T.reshape(self.shape)
    elif a.size == self.numel and len(self.shape) == 2 and self.shape[0] == 1:
      a = a.reshape(self.shape)
    if tuple(a.shape) != self.shape:
      raise ValueError('variable %s: expected shape %s (our layout), got %s' % (self.name, self.shape, a.shape))
    self.data.copy_(torch.from_numpy(np.ascontiguousarray(a)).to(self.data.device))


class VariableStore(object):
  """Named variables with TF-style scopes, consolidated into flat buffers by `finalize()`."""

  def __init__(self, device='cuda', seed=0):
    self.device = torch.device(device)
    self.vars = collections.OrderedDict()
    self._scope = []
    self._finalized = False
    self._rng = np.random.RandomState(seed)
    self.flat = None        # trainable fp32 params  [decay | no-decay]
    self.flat_grad = None
    self.flat_bf16 = None
    self.n_decay = 0
    self.state_flat = None  # non-trainable (moving statistics)
    self.workspace = {}
    # A leaf that requires grad: fed to the first layers so that autograd runs their backward
    # (parameters live outside autograd, and images / actions are constants).
    self.anchor = torch.zeros((), dtype=F32, device=self.device, requires_grad=True)

  # -- scopes ---------------------------------------------------------------------------------
  @contextlib.contextmanager
  def scope(self, name):
    if name:
      self._scope.append(name)
    try:
      yield
    finally:
      if name:
        self._scope.pop()

  def full_name(self, name):
    return '/'.join(self._scope + [name])

  # -- creation -------------------------------------------------------------------------------
  def get_variable(self, name, shape, init, trainable=True, regularize=False, kind='other',
                   tf_layout=None):
    full = self.full_name(name)
    if full in self.vars:
      v = self.vars[full]
      if v.shape != tuple(shape):
        raise ValueError('variable %s exists with shape %s, requested %s' % (full, v.shape, tuple(shape)))
      return v
    if self._finalized:
      raise ValueError('variable %s requested after finalize(); build the model first' % full)
    v = Variable(full, shape, trainable, regularize, kind, tf_layout)
    value = init(v.shape, self._rng) if callable(init) else np.full(v.shape, init, np.float32)
    v.data = torch.from_numpy(np.ascontiguousarray(value, dtype=np.float32)).to(self.device)
    v.store = self
    self.vars[full] = v
    return v

  @property
  def finalized(self):
    return self._finalized

  def trainable_variables(self):
    return [v for v in self.vars.values() if v.trainable]

  def finalize(self):
    """Moves every variable into flat buffers: trainable = [regularised | rest], state = rest."""
    if self._finalized:
      return
    train = [v for v in self.vars.values() if v.trainable]
    decay = [v for v in train if v.regularize]
    nodecay = [v for v in train if not v.regularize]
    state = [v for v in self.vars.values() if not v.trainable]
    align = 64  # elements: keeps every view 256-byte aligned (TMA needs 16 B)

    def layout(vs):
      off, table = 0, []
      for v in vs:
        table.append((v, off))
        off += (v.numel + align - 1) // align * align
      return table, off

    t1, n1 = layout(decay)
    t2, n2 = layout(nodecay)
    total = n1 + n2
    self.n_decay = n1
    self.flat = torch.zeros(max(total, align), dtype=F32, device=self.device)
    self.flat_grad = torch.zeros_like(self.flat)
    self.flat_bf16 = torch.zeros(self.flat.numel(), dtype=BF16, device=self.device)
    for table, base in ((t1, 0), (t2, n1)):
      for v, off in table:
        sl = slice(base + off, base + off + v.numel)
        self.flat[sl].copy_(v.data.reshape(-1))
        v.data = self.flat[sl].view(v.shape)
        v.grad = self.flat_grad[sl].view(v.shape)
        v.bf16 = self.flat_bf16[sl].view(v.shape)
        v.offset = base + off
    t3, n3 = layout(state)
    self.state_flat = torch.zeros(max(n3, align), dtype=F32, device=self.device)
    for v, off in t3:
      sl = slice(off, off + v.numel)
      self.state_flat[sl].copy_(v.data.reshape(-1))
      v.data = self.state_flat[sl].view(v.shape)
      v.offset = off
    self._finalized = True
    self.sync_compute_copies()

  def sync_compute_copies(self, after_optimizer=False):
    """Refreshes the bf16 compute copies of the weights from the fp32 masters.

    after_optimizer=True: the optimizer kernel already wrote the flat bf16 buffer, only the
    transposed data-gradient packs remain."""
    st = _stream()
    if not self._finalized:
      raise ValueError('finalize() first')
    self.compute_epoch = getattr(self, 'compute_epoch', 0) + 1   # invalidates weights derived from the masters
    if not after_optimizer:
      _lib.call('t2r_cast_f32_to_bf16', _p(self.flat), _p(self.flat_bf16), self.flat.numel(), st)
    for v in self.vars.values():
      if v.kind == 'conv' and not v.trainable:   # frozen weights live outside the flat buffer
        if v.bf16 is None:
          v.bf16 = torch.empty(v.shape, dtype=BF16, device=self.device)
        _lib.call('t2r_cast_f32_to_bf16', _p(v.data), _p(v.bf16), v.numel, st)
      if v.kind == 'conv' and v.needs_dgrad:
        cout, kh, kw, cin = v.shape
        if v.dgrad is None:
          v.dgrad = torch.empty(cin * kh * kw * cout, dtype=BF16, device=self.device)
        _lib.call('t2r_pack_weights', _p(v.data), None, _p(v.dgrad), cout, kh * kw, cin, st)

  def copy_values_from(self, other, trainable_flat=None):
    """Overwrites this (finalized, identically built) store's values with `other`'s: the trainable
    parameters from `trainable_flat` (e.g. the optimizer's EMA shadow) or other.flat, the moving
    statistics from other.state_flat; then refreshes the bf16 compute copies."""
    if not (self._finalized and other._finalized) or list(self.vars) != list(other.vars):
      raise ValueError('copy_values_from needs two finalized stores built by the same model')
    src = other.flat if trainable_flat is None else trainable_flat
    if src.numel() != self.flat.numel():
      raise ValueError('flat buffer sizes differ')
    self.flat.copy_(src)
    if self.state_flat is not None and other.state_flat is not None:
      self.state_flat.copy_(other.state_flat)
    self.sync_compute_copies()

  def zero_grad(self):
    self.flat_grad.zero_()
    self._grads_written = set()

  def grad_ready(self, var):
    written = self.__dict__.setdefault('_grads_written', set())
    if var.name in written:
      raise _lib.T2RError('variable %s received two gradients in one backward pass: the kernels overwrite .grad, '
                          'weight sharing (a layer applied twice) is not supported' % var.name)
    written.add(var.name)
    listener = getattr(self, 'grad_listener', None)
    if listener is not None:
      listener(var)

  def scratch(self, key, numel, dtype):
    """Persistent small workspaces (BN statistics etc.), keyed by use site."""
    t = self.workspace.get(key)
    if t is None or t.numel() < numel or t.dtype != dtype:
      t = torch.zeros(numel, dtype=dtype, device=self.device)
      self.workspace[key] = t
    return t

  # -- checkpoints in the reference's naming/layout ---------------------------------------------
  def export_tf_grads(self):
    """Gradients of the trainable variables, keyed and laid out like export_tf()."""
    saved = {}
    for n, v in self.vars.items():
      if v.trainable and v.grad is not None:
        saved[n] = v.data
        v.data = v.grad
    try:
      out = self.export_tf()
    finally:
      for n, d in saved.items():
        self.vars[n].data = d
    keep = set()
    for n in saved:
      parts = getattr(self.vars[n], 'tf_parts', None)
      keep.update([p[0] for p in parts] if parts else [n])
    return collections.OrderedDict((k, a) for k, a in out.items() if k in keep)

  def export_tf(self):
    """{reference variable name: numpy array in the reference (TF) layout}.

    A variable with `tf_parts = [(tf_name, row_start, row_stop, squeeze)]` is the row-wise
    concatenation of several reference variables (the fcgrasp_* blocks)."""
    out = collections.OrderedDict()
    for n, v in self.vars.items():
      parts = getattr(v, 'tf_parts', None)
      if parts is None:
        out[n] = v.to_tf()
        continue
      a = v.to_tf()
      for tf_name, r0, r1, squeeze in parts:
        out[tf_name] = a[r0] if squeeze else a[r0:r1]
    return out

  def import_tf(self, arrays, strict=True):
    for n, v in self.vars.items():
      parts = getattr(v, 'tf_parts', None)
      if parts is None:
        if n in arrays:
          v.from_tf(arrays[n])
        elif strict:
          raise ValueError('checkpoint lacks variable %s' % n)
        continue
      if not all(p[0] in arrays for p in parts):
        if strict:
          raise ValueError('checkpoint lacks parts of %s' % n)
        continue
      a = np.zeros(v.shape, np.float32)
      for tf_name, r0, r1, squeeze in parts:
        a[r0:r1] = np.asarray(arrays[tf_name], np.float32).reshape(a[r0:r1].shape)
      v.from_tf(a)
    if self._finalized:
      self.sync_compute_copies()


_STORE_STACK = []
# When a list is installed here every layer call appends (op, scope, output): used by the
# layer-by-layer parity tests (tests/parity_trace.py).  None in production.
TRACE = None


# When a list is installed here, every tensor-core kernel launch is bracketed by CUDA events on the
# launching stream and (kind, algorithmic_flops, start_event, end_event, algorithmic_bytes) is appended: bench.py's
# live roofline measurement.  None in production.
PROFILE = None


class _prof(object):
  """with _prof('fprop', flops): <one kernel launch>"""

  def __init__(self, kind, flops):
    nbytes = 0.0
    if not isinstance(flops, float):     # a ConvDesc: algorithmic flops + bytes (input + output once, bf16) + a shape tag
      d = flops
      flops = _conv_flops(d)
      nbytes = 2.0 * d.N * (d.H * d.W * d.Cin + d.Ho * d.Wo * d.Cout)
      kind = '%s|%dx%dx%dx%d->%d k%d s%d' % (kind, d.N, d.H, d.W, d.Cin, d.Cout, d.KH, d.stride)
    self.kind, self.flops, self.nbytes = kind, flops, nbytes

  def __enter__(self):
    if PROFILE is not None:
      self.start = torch.cuda.Event(enable_timing=True)
      self.end = torch.cuda.Event(enable_timing=True)
      self.start.record()
    return self

  def __exit__(self, *exc):
    if PROFILE is not None:
      self.end.record()
      PROFILE.append((self.kind, self.flops, self.start, self.end, self.nbytes))
    return False



# ---------------------------------------------------------------------------------------------
# high-precision PREDICT mode (csrc/hp.cu): fp32 activations, convolutions as bf16x3
# ---------------------------------------------------------------------------------------------
_HIGH_PRECISION = False


@contextlib.contextmanager
def high_precision():
  """Inference graphs built inside this context keep every activation in fp32 and evaluate convolutions /
  tensor-core dense layers as bf16x3 (x_hi*w_hi + x_lo*w_hi + x_hi*w_lo, fp32 accumulation) on the same
  tcgen05 kernels: q_predicted within 1e-4 of the fp32 restatement of the reference where bf16 activation
  storage is ~1e-2 off.  Meant for what consumes Q values - CEM arg-max, Bellman targets, serving; the
  training step stays bf16.  Images must be fed as fp32."""
  global _HIGH_PRECISION
  if torch.is_grad_enabled():
    raise _lib.T2RError('nn.high_precision() is an inference mode: wrap it in torch.no_grad()')
  old, _HIGH_PRECISION = _HIGH_PRECISION, True
  try:
    yield
  finally:
    _HIGH_PRECISION = old


def is_high_precision():
  return _HIGH_PRECISION


def _hp_f32(x):
  return to_f32(x).contiguous() if x.dtype != F32 else x.contiguous()


def _hp_cached(v, key, build):
  """Per-variable cache of derived weights, dropped whenever the store refreshes its compute copies."""
  vs = current_store()
  epoch = getattr(vs, 'compute_epoch', 0) if vs.finalized else None
  cache = v.__dict__.setdefault('_hp_cache', {})
  hit = cache.get(key)
  if hit is not None and epoch is not None and hit[0] == epoch:
    return hit[1]
  value = build()
  cache[key] = (epoch, value)
  return value


def _hp_conv(x, wv, bv, kh, kw, stride, ho, wo, pt, pl, residual, relu, small):
  st = _stream()
  x = _hp_f32(x)
  n, h, w, cin = x.shape
  cout = wv.shape[0]
  y = torch.empty((n, ho, wo, cout), dtype=F32, device=x.device)
  bias = bv.data if bv is not None else None
  if small:   # the 3-channel stem: direct fp32 convolution on the CUDA cores (2 % of the network's flops)
    w_hwio = _hp_cached(wv, 'hwio', lambda: torch.from_numpy(np.ascontiguousarray(wv.to_tf())).to(x.device))
    _lib.call('t2r_conv2d_direct_f32_fwd', _p(x), _p(w_hwio), _p(bias), _p(y), n, h, w, cin, cout, kh, kw, stride, pt,
              pl, ho, wo, st)
  else:
    def pack():
      w3 = torch.empty((cout, kh, kw, 3 * cin), dtype=BF16, device=x.device)
      _lib.call('t2r_hp_pack_weights3', _p(wv.data), _p(w3), cout, kh * kw, cin, st)
      return w3
    w3 = _hp_cached(wv, 'w3', pack)
    x3 = torch.empty((n, h, w, 3 * cin), dtype=BF16, device=x.device)
    _lib.call('t2r_hp_split3', _p(x), _p(x3), n * h * w, cin, st)
    flags = _lib.T2R_EPI_OUT_F32 | (_lib.T2R_EPI_BIAS if bias is not None else 0)
    d = _conv_desc(n, h, w, 3 * cin, cout, kh, kw, stride, pt, pl, ho, wo, flags)
    with _prof('fprop', d):
      _lib.call('t2r_conv2d_fprop', C.byref(d), _p(x3), _p(w3), _p(bias), None, _p(y), st)
  if residual is not None:
    _lib.call('t2r_add_f32', _p(y), _p(_hp_f32(residual)), _p(y), y.numel(), st)
  if relu:
    _lib.call('t2r_relu_f32_fwd', _p(y), _p(y), y.numel(), st)
  return y


def _hp_batch_norm(x, bn, relu):
  x = _hp_f32(x)
  c = x.shape[-1]
  st = _stream()
  gamma = bn['gamma'].data if bn['gamma'] is not None else torch.ones(c, dtype=F32, device=x.device)
  y = torch.empty_like(x)
  _lib.call('t2r_bn_infer_f32_fwd', _p(x), _p(gamma), _p(bn['beta'].data), _p(bn['moving_mean'].data),
            _p(bn['moving_variance'].data), _p(y), x.numel() // c, c, bn['eps'], st)
  if relu:
    _lib.call('t2r_relu_f32_fwd', _p(y), _p(y), y.numel(), st)
  return y


def _conv_flops(d):
  return 2.0 * d.N * d.Ho * d.Wo * d.Cout * d.KH * d.KW * d.Cin


def _trace(op, scope, y):
  if TRACE is not None:
    TRACE.append((op, current_store().full_name(scope) if scope else '', y))
  return y



@contextlib.contextmanager
def variable_store(vs):
  """Makes `vs` the store layer functions create/look up variables in (cf. tf.Graph.as_default)."""
  _STORE_STACK.append(vs)
  try:
    yield vs
  finally:
    _STORE_STACK.pop()


def current_store():
  if not _STORE_STACK:
    raise ValueError('no active VariableStore: wrap the network call in `with nn.variable_store(vs):`')
  return _STORE_STACK[-1]


@contextlib.contextmanager
def variable_scope(name):
  with current_store().scope(name):
    yield


# ---------------------------------------------------------------------------------------------
# initialisers (numpy, seeded by the store)
# ---------------------------------------------------------------------------------------------
def truncated_normal(stddev):
  def init(shape, rng):
    a = rng.normal(0.0, stddev, size=shape)
    bad = np.abs(a) > 2 * stddev
    while bad.any():
      a[bad] = rng.normal(0.0, stddev, size=int(bad.sum()))
      bad = np.abs(a) > 2 * stddev
    return a.astype(np.float32)
  return init


def variance_scaling(fan_in):
  """tf.variance_scaling_initializer() defaults: scale 1, fan_in, truncated normal."""
  std = math.sqrt(1.0 / max(1.0, fan_in)) / .87962566103423978
  return truncated_normal(std)


def glorot_uniform(fan_in, fan_out):
  lim = math.sqrt(6.0 / (fan_in + fan_out))
  return lambda shape, rng: rng.uniform(-lim, lim, size=shape).astype(np.float32)


# ---------------------------------------------------------------------------------------------
# convolution
# ---------------------------------------------------------------------------------------------
def _conv_desc(n, h, w, cin, cout, kh, kw, stride, pt, pl, ho, wo, flags=0):
  d = _lib.ConvDesc()
  d.struct_size = C.sizeof(_lib.ConvDesc)
  d.N, d.H, d.W, d.Cin, d.Cout, d.KH, d.KW = n, h, w, cin, cout, kh, kw
  d.stride, d.pad_top, d.pad_left, d.Ho, d.Wo, d.flags = stride, pt, pl, ho, wo, flags
  return d


def conv_geometry(h, w, kh, kw, stride, padding):
  """padding: 'SAME' | 'VALID' | ('EXPLICIT', pad_begin) -> (Ho, Wo, pad_top, pad_left)."""
  if padding == 'SAME':
    ho, pt = _lib.same_padding(h, kh, stride)
    wo, pl = _lib.same_padding(w, kw, stride)
  elif padding == 'VALID':
    ho, wo, pt, pl = (h - kh) // stride + 1, (w - kw) // stride + 1, 0, 0
  else:  # fixed_padding (film_resnet_model.py:60-86): pad_beg=(k-1)//2, pad_end=k-1-pad_beg, then VALID
    pb_h, pb_w = (kh - 1) // 2, (kw - 1) // 2
    ho = (h + (kh - 1) - kh) // stride + 1
    wo = (w + (kw - 1) - kw) // stride + 1
    pt, pl = pb_h, pb_w
  return ho, wo, pt, pl


# Fused batch-norm statistics: in training, a bf16 convolution also accumulates the per-channel
# sum / sum of squares of its output in the epilogue (t2r_conv2d_fprop_stats) and hangs the fp64
# [2*C] buffer on the output tensor; batch_norm() on exactly that tensor then skips its statistics
# pass (one full HBM read of the activation).  Any op in between creates a new tensor object
# without the attribute, which falls back to t2r_bn_stats.
FUSE_BN_STATS = os.environ.get('T2R_FUSE_BN_STATS', '1') != '0'
# Inference graphs: fold batch norm (+ReLU) into the convolution that feeds it (DeferredConv).
FOLD_INFERENCE_BN = os.environ.get('T2R_FOLD_INFERENCE_BN', '1') != '0'


# Training graphs: batch norm + ReLU and the convolution(s) that consume it run as ONE autograd node
# (_BnReluConvFn).  Two kernel fusions hang off that node:
#   * operand fusion (t2r_conv2d_{fprop,wgrad}_bnrelu): a 1x1 consumer reads the RAW tensor and applies the
#     normalisation to its operand tiles in shared memory, so the normalised activation is never written.  The
#     rewrite costs ~5 instructions per element on four extra warps and is repeated for every N tile of the
#     GEMM, so it pays only where the A operand dominates the traffic and is read once: Cout <= 128 (one N tile),
#     i.e. the 4C -> C reductions of the bottleneck blocks (measured on B200, profiles/r02_bn_fusion.md: 256->64
#     at 118x118, batch 512: apply 1.2 ms saved for +0.37 fprop +0.23 wgrad; 256->1024 at 30x30 loses).
#   * masked / reduced data gradients (t2r_conv2d_dgrad_bnrelu): correct and tested, but the epilogue needs ~24
#     instructions per element against a budget of ~6 at HBM speed, so the stand-alone reduction pass is faster
#     (same file); the C entry point therefore fuses only when T2R_BNBWD_EPI=1.
#   * backward through the consumer's GEMMs (_bn_bwd_gemm_eligible): when the only consumer is a 1x1 stride-1
#     convolution whose data gradient runs on the TMA-epilogue kernel, its weight gradient also yields the two
#     batch-norm sums (t2r_conv2d_wgrad_bnsums) and its data gradient writes dx itself (t2r_conv2d_dgrad_bnapply):
#     g, the reduction pass and the apply pass disappear, and z is not kept for backward.
# T2R_FUSE_BN_NODE=0 restores the separate nodes; T2R_FUSE_BN_OPERAND = 0 | auto | all; T2R_BN_BWD_GEMM=0 restores
# the data gradient + reduction + apply backward everywhere.
FUSE_BN_NODE = os.environ.get('T2R_FUSE_BN_NODE', '1') != '0'
FUSE_BN_OPERAND = os.environ.get('T2R_FUSE_BN_OPERAND', 'auto')
_BN_OPERAND_MAX_COUT = int(os.environ.get('T2R_BN_OPERAND_MAX_COUT', '128'))
FUSE_BN_BWD_EPILOGUE = os.environ.get('T2R_BNBWD_EPI', '0') == '1'
BN_BWD_GEMM = os.environ.get('T2R_BN_BWD_GEMM', '1') != '0'


def _bn_bwd_gemm_eligible(convs, descs):
  if not BN_BWD_GEMM or len(convs) != 1:
    return False
  var = convs[0][0]
  return (var.trainable and var.dgrad is not None
          and _lib.lib().t2r_conv2d_dgrad_bnapply_supported(C.byref(descs[0])) == 1)


def _bn_operand_fusable(cin, cout, kh, kw, pt, pl, has_res):
  del has_res
  if FUSE_BN_OPERAND == '0' or kh != 1 or kw != 1 or pt or pl:
    return False
  if FUSE_BN_OPERAND == 'all':
    return True
  return cout <= _BN_OPERAND_MAX_COUT and cin >= 2 * cout


def _new_bn_stats(channels, device):
  if not (FUSE_BN_STATS and torch.is_grad_enabled()) or channels > 2048:
    return None
  return torch.zeros(2 * channels, dtype=torch.float64, device=device)


class _Conv2dFn(torch.autograd.Function):
  """y = conv(x, W) [+bias] [+residual] [relu] on the tcgen05 implicit-GEMM kernels."""

  @staticmethod
  def forward(ctx, x, residual, var, bias_var, geom, relu, out_f32, stats=None, anchor=None):
    n, h, w, cin = x.shape
    cout, kh, kw, _ = var.shape
    stride, ho, wo, pt, pl = geom
    flags = 0
    if bias_var is not None:
      flags |= _lib.T2R_EPI_BIAS
    if residual is not None:
      flags |= _lib.T2R_EPI_RESIDUAL
    if relu:
      flags |= _lib.T2R_EPI_RELU
    if out_f32:
      flags |= _lib.T2R_EPI_OUT_F32
    d = _conv_desc(n, h, w, cin, cout, kh, kw, stride, pt, pl, ho, wo, flags)
    y = torch.empty((n, ho, wo, cout), dtype=F32 if out_f32 else BF16, device=x.device)
    with _prof('fprop', d):
      _lib.call('t2r_conv2d_fprop_stats', C.byref(d), _p(x), _p(var.bf16),
                _p(bias_var.data if bias_var is not None else None), _p(residual), _p(y), _p(stats), _stream())
    ctx.var, ctx.bias_var, ctx.desc, ctx.relu, ctx.out_f32 = var, bias_var, d, relu, out_f32
    ctx.has_res = residual is not None
    ctx.save_for_backward(x, y if relu else None)
    return y

  @staticmethod
  def backward(ctx, dy):
    x, y = ctx.saved_tensors
    var, d = ctx.var, ctx.desc
    st = _stream()
    if ctx.out_f32:
      dyb = torch.empty(dy.shape, dtype=BF16, device=dy.device)
      _lib.call('t2r_cast_f32_to_bf16', _p(dy.contiguous()), _p(dyb), dy.numel(), st)
      dy = dyb
    dy = dy.contiguous()
    if ctx.relu:
      dz = torch.empty_like(dy)
      _lib.call('t2r_relu_bwd_bf16', _p(dy), _p(y), _p(dz), dy.numel(), st)
      dy = dz
    if ctx.bias_var is not None and ctx.bias_var.trainable:
      rows = dy.numel() // dy.shape[-1]
      ws = torch.empty(2 * dy.shape[-1], dtype=torch.float64, device=dy.device)
      _lib.call('t2r_colsum_bf16', _p(dy), rows, dy.shape[-1], _p(ws), _p(ctx.bias_var.grad), st)
      ctx.bias_var.grad_ready()
    if var.trainable:
      with _prof('wgrad', d):
        _lib.call('t2r_conv2d_wgrad', C.byref(d), _p(x), _p(dy), _p(var.grad), st)
      var.grad_ready()
    dx = None
    if ctx.needs_input_grad[0]:
      if var.dgrad is None:
        raise _lib.T2RError('conv %s needs a data gradient but was built with needs_dgrad=False' % var.name)
      dx = torch.empty_like(x)
      with _prof('dgrad', d):
        _lib.call('t2r_conv2d_dgrad', C.byref(d), _p(dy), _p(var.dgrad), _p(dx), 0, st)
    dres = dy if (ctx.has_res and ctx.needs_input_grad[1]) else None
    return dx, dres, None, None, None, None, None, None, None


class _DualConvFn(torch.autograd.Function):
  """Two convolutions reading the same input (ResNet projection shortcut + first block conv):
  one autograd node, so the two data gradients are accumulated by the second dgrad's epilogue
  instead of a separate elementwise add."""

  @staticmethod
  def forward(ctx, x, var1, geom1, var2, geom2, stats2=None):
    n, h, w, cin = x.shape
    descs, ys = [], []
    for var, (stride, ho, wo, pt, pl), stats in ((var1, geom1, None), (var2, geom2, stats2)):
      cout, kh, kw, _ = var.shape
      d = _conv_desc(n, h, w, cin, cout, kh, kw, stride, pt, pl, ho, wo, 0)
      y = torch.empty((n, ho, wo, cout), dtype=BF16, device=x.device)
      with _prof('fprop', d):
        _lib.call('t2r_conv2d_fprop_stats', C.byref(d), _p(x), _p(var.bf16), None, None, _p(y), _p(stats), _stream())
      descs.append(d)
      ys.append(y)
    ctx.vars, ctx.descs = (var1, var2), descs
    ctx.save_for_backward(x)
    return ys[0], ys[1]

  @staticmethod
  def backward(ctx, dy1, dy2):
    (x,) = ctx.saved_tensors
    st = _stream()
    dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
    wrote = False
    # second convolution first: a strided 1x1 projection reaches only one output phase, so running it
    # last (accumulate) touches that phase only instead of zero-filling the others first
    for var, d, dy in reversed(list(zip(ctx.vars, ctx.descs, (dy1, dy2)))):
      if dy is None:
        continue
      dy = dy.contiguous()
      if var.trainable:
        with _prof('wgrad', d):
          _lib.call('t2r_conv2d_wgrad', C.byref(d), _p(x), _p(dy), _p(var.grad), st)
        var.grad_ready()
      if dx is not None:
        with _prof('dgrad', d):
          _lib.call('t2r_conv2d_dgrad', C.byref(d), _p(dy), _p(var.dgrad), _p(dx), 1 if wrote else 0, st)
        wrote = True
    if dx is not None and not wrote:
      dx.zero_()
    return dx, None, None, None, None, None


def conv2d_pair(x, spec1, spec2):
  """spec = dict(filters, kernel_size, stride, padding, scope, names, regularize).  Returns (y1, y2);
  variables are created in the order (spec1, spec2)."""
  deferred_bn = x if isinstance(x, DeferredBN) else None
  if deferred_bn is None:
    _require_cuda(x, 'conv2d_pair')
  vs = current_store()
  n, h, w, cin = x.shape
  out = []
  for spec in (spec1, spec2):
    k = spec['kernel_size']
    stride, padding = spec.get('stride', 1), spec.get('padding', 'SAME')
    ho, wo, pt, pl = conv_geometry(h, w, k, k, stride, padding)
    with vs.scope(spec['scope']):
      wv = vs.get_variable(spec.get('names', ('weights', 'biases'))[0], (spec['filters'], k, k, cin),
                           spec.get('initializer') or variance_scaling(k * k * cin), True,
                           spec.get('regularize', True), 'conv', 'hwio')
      wv.needs_dgrad = True
    if not vs.finalized:
      _ensure_bf16(wv)
    out.append((wv, (stride, ho, wo, pt, pl)))
  if deferred_bn is not None:
    y1, y2 = deferred_bn.run_convs(out)
    return _trace('conv', spec1['scope'], y1), _trace('conv', spec2['scope'], y2)
  stats2 = _new_bn_stats(out[1][0].shape[0], x.device)
  y1, y2 = _DualConvFn.apply(x, out[0][0], out[0][1], out[1][0], out[1][1], stats2)
  if stats2 is not None:
    y2._t2r_bn_stats = stats2
  return _trace('conv', spec1['scope'], y1), _trace('conv', spec2['scope'], y2)


class _StemConvFn(torch.autograd.Function):
  """Small-Cin convolution (image stem) without im2col: the bf16 NHWC3 image is repacked into a
  persistent zero-padded NHWC4 buffer and read through overlapping-window TMA maps
  (t2r_stem_conv_fprop / _wgrad).  Weights live as [Cout, 1, 1, KH*64] = [Cout][kh][16 px][4 ch]."""

  @staticmethod
  def _padded(vs, x, geom):
    """Packs `x` into the (persistent, zero-bordered) stem image buffer.  Returns (buffer, Hp, Wp, generation):
    the generation counter lets backward skip re-packing when nothing else used the buffer in between."""
    kh, kw, stride, ho, wo, pt, pl = geom
    n, h, w, _ = x.shape
    rows = _stem_rows(kw, stride)
    hp = max(h + pt, stride * (ho - 1) + -(-kh // rows) * rows)
    hp = -(-hp // rows) * rows
    wp = max(w + pl, stride * (wo - 1) + 16 // rows)
    wp = (wp + 1) // 2 * 2                       # row pitch multiple of 16 bytes
    key = ('stem_x4p', n, hp, wp)
    buf = vs.scratch(key, n * hp * wp * 4, BF16)   # zero-initialised once
    _lib.call('t2r_stem_pack_image', _p(x), _p(buf), n, h, w, hp, wp, pt, pl, kw, stride, _stream())
    gens = vs.workspace.setdefault('stem_generations', {})
    gens[key] = gens.get(key, 0) + 1
    return buf, hp, wp, (key, gens[key])

  @staticmethod
  def forward(ctx, x, anchor, var, bias_var, geom, vs):
    n, h, w, cin = x.shape
    cout = var.shape[0]
    kh, kw, stride, ho, wo, pt, pl = geom
    d = _conv_desc(n, h, w, cin, cout, kh, kw, stride, pt, pl, ho, wo)
    x4p, hp, wp, gen = _StemConvFn._padded(vs, x, geom)
    y = torch.empty((n, ho, wo, cout), dtype=BF16, device=x.device)
    with _prof('fprop', d):   # algorithmic flops of the real (unpadded) convolution
      _lib.call('t2r_stem_conv_fprop', C.byref(d), _p(x4p), hp, wp, _p(var.bf16),
                _p(bias_var.data if bias_var is not None else None), _p(y), _stream())
    ctx.var, ctx.bias_var, ctx.desc, ctx.geom, ctx.vs = var, bias_var, d, geom, vs
    ctx.packed = (x4p, hp, wp, gen)
    ctx.save_for_backward(x)   # the packed copy is reused in backward unless another stem call overwrote it
    return y

  @staticmethod
  def backward(ctx, dy):
    (x,) = ctx.saved_tensors
    st = _stream()
    dy = dy.contiguous()
    if ctx.bias_var is not None and ctx.bias_var.trainable:
      rows = dy.numel() // dy.shape[-1]
      ws = torch.empty(2 * dy.shape[-1], dtype=torch.float64, device=dy.device)
      _lib.call('t2r_colsum_bf16', _p(dy), rows, dy.shape[-1], _p(ws), _p(ctx.bias_var.grad), st)
      ctx.bias_var.grad_ready()
    if ctx.var.trainable:
      kh, kw = ctx.geom[0], ctx.geom[1]
      x4p, hp, wp, (key, gen) = ctx.packed
      if ctx.vs.workspace.get('stem_generations', {}).get(key) != gen:
        x4p, hp, wp, _ = _StemConvFn._padded(ctx.vs, x, ctx.geom)
      with _prof('wgrad', ctx.desc):
        _lib.call('t2r_stem_conv_wgrad', C.byref(ctx.desc), _p(x4p), hp, wp, _p(dy), _p(ctx.var.grad), st)
      _lib.call('t2r_stem_mask_grad', _p(ctx.var.grad), ctx.var.shape[0], kh, kw, ctx.geom[2], st)
      ctx.var.grad_ready()
    if ctx.needs_input_grad[0]:
      raise _lib.T2RError('stem convolution %s has no data gradient (image inputs are leaves)' % ctx.var.name)
    return None, None, None, None, None, None


class DeferredConv(object):
  """An inference-mode convolution whose launch is postponed until the batch norm that consumes it:
  batch_norm() then folds its scale into the weights and its shift + ReLU into the epilogue, so the
  pre-normalisation tensor is never written (conv2d(..., defer_for_bn=True))."""

  def __init__(self, x, wv, geom, scope):
    self.x, self.wv, self.geom, self.scope = x, wv, geom, scope
    n = x.shape[0]
    self.shape = (n, geom[1], geom[2], wv.shape[0])
    self.device = x.device

  def run(self, weights_bf16=None, bias=None, relu=False):
    x, wv = self.x, self.wv
    n, h, w, cin = x.shape
    cout, kh, kw, _ = wv.shape
    stride, ho, wo, pt, pl = self.geom
    flags = (_lib.T2R_EPI_BIAS if bias is not None else 0) | (_lib.T2R_EPI_RELU if relu else 0)
    d = _conv_desc(n, h, w, cin, cout, kh, kw, stride, pt, pl, ho, wo, flags)
    y = torch.empty((n, ho, wo, cout), dtype=BF16, device=x.device)
    with _prof('fprop', d):
      _lib.call('t2r_conv2d_fprop', C.byref(d), _p(x), _p(weights_bf16 if weights_bf16 is not None else wv.bf16),
                _p(bias), None, _p(y), _stream())
    return y

  def materialize(self):
    return _trace('conv', self.scope, self.run())



class _BnReluConvFn(torch.autograd.Function):
  """z = relu(batch_norm(x)) consumed by one or two bias-free bf16 convolutions, as one autograd node.

  forward : statistics (from the producer's epilogue when available) -> scale / shift; then either the
            operand-fused 1x1 kernels on the raw x, or t2r_bn_apply + the plain kernels on z.
  backward: weight gradients; data gradients whose LAST launch masks with [z > 0] and reduces
            sum g / sum g*x in its epilogue (t2r_conv2d_dgrad_bnrelu); t2r_bn_backward_presummed.
  Outputs : (y_1[, y_2][, x]) - the trailing x (passthrough) routes an identity shortcut's gradient into
            this node, where the batch-norm apply kernel adds it for free.
  Reference semantics: layers/film_resnet_model.py:50-57 (batch_norm), :283-340 (the block wiring)."""

  @staticmethod
  def forward(ctx, x, residual, bn, vs, convs, fused_stats, passthrough, operand_fused):
    n, h, w, c = x.shape
    rows = n * h * w
    st = _stream()
    mean = torch.empty(c, dtype=F32, device=x.device)
    invstd = torch.empty(c, dtype=F32, device=x.device)
    scale = torch.empty(c, dtype=F32, device=x.device)
    shift = torch.empty(c, dtype=F32, device=x.device)
    if fused_stats is not None:
      stats = fused_stats
    else:
      stats = vs.scratch('bn_stats', 2 * 4096, torch.float64)
      _lib.call('t2r_bn_stats', _p(x), rows, c, _p(stats), st)
    _lib.call('t2r_bn_finalize', _p(stats), rows, c, _p(bn['gamma'].data if bn['gamma'] is not None else None),
              _p(bn['beta'].data), bn['eps'], bn['momentum'], _p(bn['moving_mean'].data),
              _p(bn['moving_variance'].data), _p(mean), _p(invstd), _p(scale), _p(shift), st)
    z = None
    if not operand_fused:
      z = torch.empty_like(x)
      _lib.call('t2r_bn_apply', _p(x), _p(z), rows, c, _p(scale), _p(shift), None, h * w, 1, st)
    outs, descs = [], []
    for var, (stride, ho, wo, pt, pl), ostats in convs:
      cout, kh, kw, _ = var.shape
      flags = _lib.T2R_EPI_RESIDUAL if residual is not None else 0
      d = _conv_desc(n, h, w, c, cout, kh, kw, stride, pt, pl, ho, wo, flags)
      y = torch.empty((n, ho, wo, cout), dtype=BF16, device=x.device)
      with _prof('fprop', d):
        if operand_fused:
          _lib.call('t2r_conv2d_fprop_bnrelu', C.byref(d), _p(x), _p(scale), _p(shift), _p(var.bf16), _p(residual),
                    _p(y), _p(ostats), st)
        else:
          _lib.call('t2r_conv2d_fprop_stats', C.byref(d), _p(z), _p(var.bf16), None, _p(residual), _p(y), _p(ostats), st)
      outs.append(y)
      descs.append(d)
    ctx.bn, ctx.vs, ctx.descs, ctx.vars = bn, vs, descs, [cv[0] for cv in convs]
    ctx.operand_fused, ctx.passthrough, ctx.has_res = operand_fused, passthrough, residual is not None
    ctx.bwd_gemm = ctx.needs_input_grad[0] and _bn_bwd_gemm_eligible(convs, descs)
    ctx.save_for_backward(x, mean, invstd, scale, shift, None if ctx.bwd_gemm else z)
    if passthrough:
      outs.append(x.view_as(x))
    return tuple(outs)

  @staticmethod
  def backward(ctx, *grads):
    x, mean, invstd, scale, shift, z = ctx.saved_tensors
    bn, vs = ctx.bn, ctx.vs
    n, h, w, c = x.shape
    rows = n * h * w
    st = _stream()
    dpass = grads[len(ctx.vars)] if ctx.passthrough else None
    if dpass is not None:
      dpass = dpass.contiguous()
    dys = [g.contiguous() if g is not None else None for g in grads[:len(ctx.vars)]]
    if ctx.bwd_gemm and dys[0] is not None:
      return _BnReluConvFn._backward_gemm(ctx, x, mean, invstd, scale, shift, dys[0], dpass)
    for var, d, dy in zip(ctx.vars, ctx.descs, dys):
      if dy is None or not var.trainable:
        continue
      with _prof('wgrad', d):
        if ctx.operand_fused:
          _lib.call('t2r_conv2d_wgrad_bnrelu', C.byref(d), _p(x), _p(scale), _p(shift), _p(dy), _p(var.grad), st)
        else:
          _lib.call('t2r_conv2d_wgrad', C.byref(d), _p(z), _p(dy), _p(var.grad), st)
      var.grad_ready()
    dx = None
    if ctx.needs_input_grad[0]:
      # the convolution that covers every input pixel first; a strided projection (conv 0 of a pair) then
      # accumulates into its phase only.  The last launch masks and reduces.
      live = [(var, d, dy) for var, d, dy in reversed(list(zip(ctx.vars, ctx.descs, dys))) if dy is not None]
      g = torch.empty_like(x)
      red = torch.zeros(2 * c, dtype=torch.float64, device=x.device)
      if not live:
        g.zero_()
      for i, (var, d, dy) in enumerate(live):
        if var.dgrad is None:
          raise _lib.T2RError('conv %s needs a data gradient but was built with needs_dgrad=False' % var.name)
        with _prof('dgrad', d):
          if i == len(live) - 1 and FUSE_BN_BWD_EPILOGUE:
            _lib.call('t2r_conv2d_dgrad_bnrelu', C.byref(d), _p(dy), _p(var.dgrad), _p(x), _p(scale), _p(shift), _p(g),
                      1 if i else 0, _p(red), st)
          else:
            _lib.call('t2r_conv2d_dgrad', C.byref(d), _p(dy), _p(var.dgrad), _p(g), 1 if i else 0, st)
      gamma = bn['gamma']
      dgamma = gamma.grad if (gamma is not None and gamma.trainable) else vs.scratch('bn_dgamma', 4096, F32)
      dbeta = bn['beta'].grad if bn['beta'].trainable else vs.scratch('bn_dbeta', 4096, F32)
      dx = torch.empty_like(x)
      if FUSE_BN_BWD_EPILOGUE:
        _lib.call('t2r_bn_backward_presummed', _p(g), _p(x), _p(dpass), _p(dx), rows, c, _p(mean), _p(invstd), _p(scale),
                  _p(shift), 1, _p(red), _p(dgamma), _p(dbeta), st)
      else:     # reduction pass + apply pass (the default: see FUSE_BN_NODE above)
        _lib.call('t2r_bn_backward', _p(g), _p(x), _p(dpass), _p(dx), rows, c, _p(gamma.data if gamma is not None else None),
                  _p(mean), _p(invstd), _p(scale), _p(shift), 1, _p(red), _p(dgamma), _p(dbeta), st)
      _bn_grads_ready(bn)
    dres = dys[0] if (ctx.has_res and ctx.needs_input_grad[1]) else None
    return dx, dres, None, None, None, None, None, None

  @staticmethod
  def _backward_gemm(ctx, x, mean, invstd, scale, shift, dy, dpass):
    """Single 1x1 consumer: dual-operand weight gradient (dw and the two batch-norm sums), finalize (dgamma, dbeta
    and the apply coefficients), data gradient whose epilogue writes dx."""
    bn, vs, var, d = ctx.bn, ctx.vs, ctx.vars[0], ctx.descs[0]
    c = x.shape[-1]
    rows = x.numel() // c
    st = _stream()
    sums = torch.zeros(2 * c, dtype=torch.float64, device=x.device)
    coef = torch.empty(2 * c, dtype=F32, device=x.device)
    with _prof('wgrad', d):
      _lib.call('t2r_conv2d_wgrad_bnsums', C.byref(d), _p(x), _p(scale), _p(shift), _p(dy), _p(var.dgrad),
                _p(var.grad), _p(sums), st)
    var.grad_ready()
    gamma = bn['gamma']
    dgamma = gamma.grad if (gamma is not None and gamma.trainable) else vs.scratch('bn_dgamma', 4096, F32)
    dbeta = bn['beta'].grad if bn['beta'].trainable else vs.scratch('bn_dbeta', 4096, F32)
    _lib.call('t2r_bn_backward_gemm_finalize', _p(sums), rows, c, _p(mean), _p(invstd), _p(scale), _p(dgamma),
              _p(dbeta), _p(coef), st)
    _bn_grads_ready(bn)
    dx = torch.empty_like(x)
    with _prof('dgrad', d):
      _lib.call('t2r_conv2d_dgrad_bnapply', C.byref(d), _p(dy), _p(var.dgrad), _p(x), _p(scale), _p(shift), _p(coef),
                _p(dpass), _p(dx), st)
    dres = dy if (ctx.has_res and ctx.needs_input_grad[1]) else None
    return dx, dres, None, None, None, None, None, None


class DeferredBN(object):
  """A training-mode batch norm + ReLU whose launch waits for its consumer: conv2d / conv2d_pair turn the pair
  into one _BnReluConvFn node; anything else calls materialize() (the stand-alone _BatchNormFn).
  `shortcut` (passthrough=True) is the input routed through the node, available once the node has run."""

  def __init__(self, x, bn, vs, scope, fused_stats, passthrough):
    self.x, self.bn, self.vs, self.scope = x, bn, vs, scope
    self.fused_stats, self.passthrough = fused_stats, passthrough
    self.shape, self.device = x.shape, x.device
    self.shortcut = None
    self._z = None
    self._consumed = False

  def _consume(self):
    if self._consumed:
      raise _lib.T2RError('a deferred batch norm (%s) can feed only one consumer; call .materialize() to share it'
                          % self.scope)
    self._consumed = True

  def materialize(self):
    if self._z is None:
      self._consume()
      if self.passthrough:
        z, self.shortcut = _BatchNormFn.apply(self.x, None, self.bn, True, True, self.vs, True, self.fused_stats)
      else:
        z = _BatchNormFn.apply(self.x, None, self.bn, True, True, self.vs, False, self.fused_stats)
      self._z = _trace('bn', self.scope, z)
    return self._z

  def run_convs(self, convs, residual=None):
    """convs: [(weight variable, (stride, ho, wo, pt, pl))] -> list of outputs (with fused bn_stats attached)."""
    self._consume()
    c = self.x.shape[-1]
    fused = all(_bn_operand_fusable(c, var.shape[0], var.shape[1], var.shape[2], geom[3], geom[4], residual is not None)
                for var, geom in convs)
    packed = []
    for var, geom in convs:
      packed.append((var, geom, _new_bn_stats(var.shape[0], self.device)))
    outs = _BnReluConvFn.apply(self.x, residual, self.bn, self.vs, tuple(packed), self.fused_stats, self.passthrough,
                               fused)
    if self.passthrough:
      self.shortcut = outs[-1]
    ys = list(outs[:len(convs)])
    for y, (_, _, ostats) in zip(ys, packed):
      if ostats is not None:
        y._t2r_bn_stats = ostats
    return ys


def _node_fusable_conv(x, wv, bv, relu, out_f32):
  return bv is None and not relu and not out_f32 and wv.trainable and len(wv.shape) == 4 and x.shape[-1] % 64 == 0


def conv2d(x, filters, kernel_size, stride=1, padding='SAME', use_bias=False, scope='conv',
           initializer=None, regularize=True, residual=None, relu=False, needs_dgrad=True,
           trainable=True, out_f32=False, names=('weights', 'biases'), defer_for_bn=False):
  """slim.conv2d / tf.layers.conv2d without normaliser or activation (compose with batch_norm).
  defer_for_bn=True (only honoured without autograd): returns a DeferredConv for batch_norm to fuse."""
  if isinstance(x, (DeferredConv, DeferredContext)):
    x = x.materialize()
  deferred_bn = x if isinstance(x, DeferredBN) else None
  if deferred_bn is None:
    _require_cuda(x, 'conv2d')
  vs = current_store()
  kh, kw = (kernel_size, kernel_size) if isinstance(kernel_size, int) else kernel_size
  n, h, w, cin = x.shape
  ho, wo, pt, pl = conv_geometry(h, w, kh, kw, stride, padding)
  small = cin % 64 != 0
  if small and (cin != 3 or kw > 16 or stride > 2):
    raise _lib.T2RError('conv2d: Cin=%d is supported only as the 3-channel image stem' % cin)
  kpad = -(-kh // _stem_rows(kw, stride)) * 64 if small else 0   # [chunks][rows][16/rows pixels][4 ch]
  with vs.scope(scope):
    if small:
      # stored as [Cout, 1, 1, Kpad] (K-padded OHWI, flattened taps); TF layout handled by to_tf
      wv = vs.get_variable(names[0], (filters, 1, 1, kpad),
                           _padded_init(initializer or variance_scaling(kh * kw * cin), filters, kh, kw, cin, kpad,
                                        stride),
                           trainable, regularize, 'conv', None)
      wv.stem_geom = (kh, kw, cin, stride)
      _install_stem_tf(wv)
    else:
      wv = vs.get_variable(names[0], (filters, kh, kw, cin), initializer or variance_scaling(kh * kw * cin),
                           trainable, regularize, 'conv', 'hwio')
      wv.needs_dgrad = wv.needs_dgrad or needs_dgrad
    bv = vs.get_variable(names[1], (filters,), 0.0, trainable, False) if use_bias else None
  if not vs.finalized:
    _ensure_bf16(wv)
  if _HIGH_PRECISION:
    return _trace('conv', scope, _hp_conv(x, wv, bv, kh, kw, stride, ho, wo, pt, pl, residual, relu, small))
  if deferred_bn is not None:
    if not small and _node_fusable_conv(deferred_bn, wv, bv, relu, out_f32):
      (y,) = deferred_bn.run_convs([(wv, (stride, ho, wo, pt, pl))], residual)
      return _trace('conv', scope, y)
    x = deferred_bn.materialize()
  if small:
    return _trace('conv', scope, _StemConvFn.apply(x.contiguous(), vs.anchor, wv, bv,
                                                   (kh, kw, stride, ho, wo, pt, pl), vs))
  if (defer_for_bn and FOLD_INFERENCE_BN and not torch.is_grad_enabled() and residual is None and bv is None and
      not relu and not out_f32):
    return DeferredConv(x.contiguous(), wv, (stride, ho, wo, pt, pl), scope)
  stats = None if (out_f32 or relu) else _new_bn_stats(filters, x.device)
  # a leaf input (e.g. the FiLM generator's embedding) would leave the node out of the autograd graph and
  # its weights without a gradient: the store's anchor scalar keeps it in
  anchor = vs.anchor if (torch.is_grad_enabled() and not x.requires_grad and trainable) else None
  y = _Conv2dFn.apply(x, residual, wv, bv, (stride, ho, wo, pt, pl), relu, out_f32, stats, anchor)
  if stats is not None:
    y._t2r_bn_stats = stats
  return _trace('conv', scope, y)


def _stem_rows(kw, stride):
  """Filter rows per 64-wide K chunk of the stem layout (t2r_b200.h: t2r_stem_k)."""
  return 2 if (kw <= 8 and stride == 2) else 1


def _stem_pack(w_ohwi, stride):
  """[Cout, KH, KW, 3] -> [Cout, K] in the stem layout: [kh][16 px][4 ch] (rows = 1) or
  [chunk][8 px][2 rows][4 ch] (rows = 2)."""
  cout, kh, kw, cin = w_ohwi.shape
  rows = _stem_rows(kw, stride)
  chunks = -(-kh // rows)
  out = np.zeros((cout, chunks * rows, 16 // rows, 4), np.float32)     # [co][kh][px][ch]
  out[:, :kh, :kw, :cin] = w_ohwi
  if rows == 2:
    out = out.reshape(cout, chunks, 2, 8, 4).transpose(0, 1, 3, 2, 4)  # [co][chunk][px][row][ch]
  return np.ascontiguousarray(out).reshape(cout, chunks * 64)


def _stem_unpack(w_packed, kh, kw, cin, stride):
  """Inverse of _stem_pack: [Cout, K] -> [Cout, KH, KW, cin]."""
  cout = w_packed.shape[0]
  rows = _stem_rows(kw, stride)
  chunks = -(-kh // rows)
  a = w_packed.reshape(cout, chunks, 64)
  if rows == 2:
    a = a.reshape(cout, chunks, 8, 2, 4).transpose(0, 1, 3, 2, 4)      # [co][chunk][row][px][ch]
  a = a.reshape(cout, chunks * rows, 16 // rows, 4)
  return a[:, :kh, :kw, :cin]


def _padded_init(init, filters, kh, kw, cin, kpad, stride):
  def f(shape, rng):
    return _stem_pack(init((filters, kh, kw, cin), rng), stride).reshape(shape)
  return f


def _install_stem_tf(v):
  kh, kw, cin, stride = v.stem_geom

  def to_tf():
    a = _stem_unpack(v.data.detach().float().cpu().numpy().reshape(v.shape[0], -1), kh, kw, cin, stride)
    return np.ascontiguousarray(a.transpose(1, 2, 3, 0))          # HWIO

  def from_tf(a):
    a = np.asarray(a, np.float32).transpose(3, 0, 1, 2)            # OHWI
    v.data.copy_(torch.from_numpy(_stem_pack(a, stride).reshape(v.shape)).to(v.data.device))
  v.to_tf, v.from_tf = to_tf, from_tf


def _ensure_bf16(v):
  """Before finalize() (the build pass) variables are stand-alone tensors: give them compute copies."""
  st = _stream()
  if v.bf16 is None or v.bf16.numel() != v.numel:
    v.bf16 = torch.empty(v.shape, dtype=BF16, device=v.data.device)
  _lib.call('t2r_cast_f32_to_bf16', _p(v.data), _p(v.bf16), v.numel, st)
  if v.kind == 'conv' and v.needs_dgrad and len(v.shape) == 4:
    cout, kh, kw, cin = v.shape
    v.dgrad = torch.empty(v.numel, dtype=BF16, device=v.data.device)
    _lib.call('t2r_pack_weights', _p(v.data), None, _p(v.dgrad), cout, kh * kw, cin, st)
  if v.grad is None:
    v.grad = torch.zeros(v.shape, dtype=F32, device=v.data.device)


def dense(x, units, scope='fc', use_bias=False, initializer=None, regularize=True, relu=False,
          needs_dgrad=True, trainable=True, out_f32=False, names=('weights', 'biases')):
  """slim.fully_connected on a [rows, K] bf16 matrix through the tensor-core path (K % 64 == 0)."""
  vs = current_store()
  rows, k = x.shape
  y = conv2d(x.view(1, 1, rows, k), units, 1, 1, 'VALID', use_bias, scope,
             initializer or glorot_uniform(k, units), regularize, None, relu, needs_dgrad, trainable, out_f32,
             names)
  v = vs.vars[vs.full_name(scope + '/' + names[0])]
  v.tf_layout = 'io_hwc'
  return y.view(rows, units)


# ---------------------------------------------------------------------------------------------
# batch norm (+ReLU, +FiLM)
# ---------------------------------------------------------------------------------------------
def _bn_grads_ready(bn):
  for key in ('gamma', 'beta'):
    if bn[key] is not None and bn[key].trainable:
      bn[key].grad_ready()


class _BatchNormFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, film, bn, training, relu, vs, passthrough=False, fused_stats=None):
    c = x.shape[-1]
    rows = x.numel() // c
    st = _stream()
    y = torch.empty_like(x)
    scale = torch.empty(c, dtype=F32, device=x.device)
    shift = torch.empty(c, dtype=F32, device=x.device)
    rows_per_image = rows // x.shape[0]
    if training:
      mean = torch.empty(c, dtype=F32, device=x.device)
      invstd = torch.empty(c, dtype=F32, device=x.device)
      if fused_stats is not None:
        stats = fused_stats
      else:
        stats = vs.scratch('bn_stats', 2 * 4096, torch.float64)
        _lib.call('t2r_bn_stats', _p(x), rows, c, _p(stats), st)
      _lib.call('t2r_bn_finalize', _p(stats), rows, c, _p(bn['gamma'].data if bn['gamma'] is not None else None),
                _p(bn['beta'].data), bn['eps'], bn['momentum'], _p(bn['moving_mean'].data),
                _p(bn['moving_variance'].data), _p(mean), _p(invstd), _p(scale), _p(shift), st)
      ctx.save_for_backward(x, mean, invstd, scale, shift, film)
    else:
      _lib.call('t2r_bn_infer_params', c, _p(bn['gamma'].data if bn['gamma'] is not None else None),
                _p(bn['beta'].data), _p(bn['moving_mean'].data), _p(bn['moving_variance'].data), bn['eps'],
                _p(scale), _p(shift), st)
    _lib.call('t2r_bn_apply', _p(x), _p(y), rows, c, _p(scale), _p(shift), _p(film), rows_per_image,
              1 if relu else 0, st)
    ctx.bn, ctx.relu, ctx.training, ctx.vs = bn, relu, training, vs
    if passthrough:
      # `x` is also consumed elsewhere (the residual branch): returning it as a second output routes
      # that branch's gradient into THIS backward, where the kernel adds it for free (dres).
      return y, x.view_as(x)
    return y

  @staticmethod
  def backward(ctx, dy, dpass=None):
    if not ctx.training:
      raise _lib.T2RError('backward through inference-mode batch norm is not supported')
    x, mean, invstd, scale, shift, film = ctx.saved_tensors
    bn = ctx.bn
    c = x.shape[-1]
    rows = x.numel() // c
    st = _stream()
    dy = dy.contiguous()
    dx = torch.empty_like(x)
    red = ctx.vs.scratch('bn_red', 2 * 4096, torch.float64)
    gamma = bn['gamma']
    dgamma = gamma.grad if (gamma is not None and gamma.trainable) else ctx.vs.scratch('bn_dgamma', 4096, F32)
    dbeta = bn['beta'].grad if bn['beta'].trainable else ctx.vs.scratch('bn_dbeta', 4096, F32)
    if dpass is not None:
      dpass = dpass.contiguous()
    if film is not None:
      n = x.shape[0]
      dfilm = torch.empty_like(film)
      sums = torch.empty((n, 2, c), dtype=F32, device=x.device)
      _lib.call('t2r_bn_film_backward', _p(dy), _p(x), _p(film), _p(dpass), _p(dx), _p(dfilm), rows, c, rows // n,
                _p(mean), _p(invstd), _p(scale), _p(shift), 1 if ctx.relu else 0, _p(sums), _p(dgamma), _p(dbeta), st)
      _bn_grads_ready(bn)
      return dx, (dfilm if ctx.needs_input_grad[1] else None), None, None, None, None, None, None
    _lib.call('t2r_bn_backward', _p(dy), _p(x), _p(dpass), _p(dx), rows, c,
              _p(gamma.data if gamma is not None else None), _p(mean), _p(invstd), _p(scale), _p(shift),
              1 if ctx.relu else 0, _p(red), _p(dgamma), _p(dbeta), st)
    _bn_grads_ready(bn)
    return dx, None, None, None, None, None, None, None


def batch_norm(x, training, scope='BatchNorm', scale=True, relu=False, momentum=0.997, eps=1e-5,
               film=None, trainable=True, passthrough=False, defer=False):
  """slim.batch_norm / tf.layers.batch_normalization(fused=True) followed by an optional ReLU.
  defer=True (honoured in training graphs with relu, without FiLM): returns a DeferredBN for the consuming
  convolution to fuse with; every other consumer must call .materialize()."""
  deferred = x if isinstance(x, (DeferredConv, DeferredContext)) else None
  if deferred is not None and (training or film is not None or passthrough):
    x, deferred = deferred.materialize(), None
  if deferred is None:
    _require_cuda(x, 'batch_norm')
  vs = current_store()
  c = x.shape[-1]
  if c > 4096:
    raise ValueError('batch_norm supports up to 4096 channels')
  with vs.scope(scope):
    bn = {
        'gamma': vs.get_variable('gamma', (c,), 1.0, trainable, False) if scale else None,
        'beta': vs.get_variable('beta', (c,), 0.0, trainable, False),
        'moving_mean': vs.get_variable('moving_mean', (c,), 0.0, False, False),
        'moving_variance': vs.get_variable('moving_variance', (c,), 1.0, False, False),
        'eps': float(eps), 'momentum': float(momentum),
    }
  if not vs.finalized:
    for k in ('gamma', 'beta'):
      if bn[k] is not None and bn[k].grad is None:
        bn[k].grad = torch.zeros(bn[k].shape, dtype=F32, device=x.device)
  if _HIGH_PRECISION:
    if training or film is not None or passthrough:
      raise _lib.T2RError('high-precision mode is inference without FiLM')
    return _trace('bn', scope, _hp_batch_norm(x, bn, relu))
  if deferred is not None:
    # y = relu(conv(u, W) * scale + shift) = relu(conv(u, W * scale) + shift)
    st = _stream()
    scale_t = torch.empty(c, dtype=F32, device=x.device)
    shift_t = torch.empty(c, dtype=F32, device=x.device)
    _lib.call('t2r_bn_infer_params', c, _p(bn['gamma'].data if bn['gamma'] is not None else None),
              _p(bn['beta'].data), _p(bn['moving_mean'].data), _p(bn['moving_variance'].data), bn['eps'],
              _p(scale_t), _p(shift_t), st)
    if isinstance(deferred, DeferredContext):
      return _trace('bn', scope, deferred.run(scale_t, shift_t, relu))
    wv = deferred.wv
    folded = torch.empty(wv.shape, dtype=BF16, device=x.device)
    _lib.call('t2r_fold_bn_weights', _p(wv.data), _p(scale_t), _p(folded), wv.shape[0], wv.numel // wv.shape[0], st)
    return _trace('bn', scope, deferred.run(folded, shift_t, relu))
  fused = getattr(x, '_t2r_bn_stats', None) if (training and x.is_contiguous()) else None
  if (defer and FUSE_BN_NODE and training and relu and film is None and torch.is_grad_enabled() and TRACE is None and
      x.dtype == BF16 and x.dim() == 4 and x.requires_grad):
    return DeferredBN(x.contiguous(), bn, vs, scope, fused, passthrough)
  if passthrough:
    y, x_pass = _BatchNormFn.apply(x.contiguous(), film, bn, training, relu, vs, True, fused)
    return _trace('bn', scope, y), x_pass
  return _trace('bn', scope, _BatchNormFn.apply(x.contiguous(), film, bn, training, relu, vs, False, fused))


# ---------------------------------------------------------------------------------------------
# pooling / reshaping
# ---------------------------------------------------------------------------------------------
class _SpatialSoftmaxFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, want_map):
    n, h, w, c = x.shape
    points = torch.empty((n, 2 * c), dtype=F32, device=x.device)
    heat = torch.empty_like(x) if want_map else None
    _lib.call('t2r_spatial_softmax_fwd', _p(x), _p(points), _p(heat), n, h, w, c, _stream())
    ctx.save_for_backward(x, points)
    if want_map:
      ctx.mark_non_differentiable(heat)
      return points, heat
    return points

  @staticmethod
  def backward(ctx, dpoints, _dheat=None):
    x, points = ctx.saved_tensors
    n, h, w, c = x.shape
    dx = torch.empty_like(x)
    _lib.call('t2r_spatial_softmax_bwd', _p(x), _p(points), _p(dpoints.contiguous().float()), _p(dx), n, h, w, c,
              _stream())
    return dx, None


def spatial_softmax(features, return_softmax=False):
  """layers/spatial_softmax.py:29-88 (BuildSpatialSoftmax, deterministic branch): bf16 [N,H,W,C] ->
  fp32 expected feature points [N, 2C] (interleaved x, y per channel, as the reference's reshape
  yields) and optionally the softmax heat map (no gradient flows through the map)."""
  _require_cuda(features, 'spatial_softmax')
  if features.dtype == F32:      # the small pose_env tower (csrc/vision_small.cu)
    return _SpatialSoftmaxF32Fn.apply(features.contiguous(), return_softmax)
  if features.shape[-1] % 8 != 0:
    raise ValueError('spatial_softmax needs a multiple of 8 channels')
  out = _SpatialSoftmaxFn.apply(features.contiguous(), return_softmax)
  return out

class _MaxPoolFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, k, stride, geom):
    n, h, w, c = x.shape
    ho, wo, pt, pl = geom
    y = torch.empty((n, ho, wo, c), dtype=BF16, device=x.device)
    arg = torch.empty((n, ho, wo, c), dtype=torch.uint8, device=x.device)
    _lib.call('t2r_maxpool_fwd', _p(x), _p(y), _p(arg), n, h, w, c, k, stride, pt, pl, ho, wo, _stream())
    ctx.save_for_backward(arg)
    ctx.geom = (n, h, w, c, k, stride, pt, pl, ho, wo)
    return y

  @staticmethod
  def backward(ctx, dy):
    (arg,) = ctx.saved_tensors
    n, h, w, c, k, stride, pt, pl, ho, wo = ctx.geom
    dx = torch.empty((n, h, w, c), dtype=BF16, device=dy.device)
    _lib.call('t2r_maxpool_bwd', _p(dy.contiguous()), _p(arg), _p(dx), n, h, w, c, k, stride, pt, pl, ho, wo, _stream())
    return dx, None, None, None


def max_pool2d(x, kernel_size, stride, padding='SAME'):
  """slim.max_pool2d / tf.layers.max_pooling2d."""
  _require_cuda(x, 'max_pool2d')
  _, h, w, _ = x.shape
  geom = conv_geometry(h, w, kernel_size, kernel_size, stride, padding)
  if _HIGH_PRECISION:
    x = _hp_f32(x)
    n, _, _, c = x.shape
    ho, wo, pt, pl = geom
    y = torch.empty((n, ho, wo, c), dtype=F32, device=x.device)
    _lib.call('t2r_maxpool_f32_fwd', _p(x), _p(y), n, h, w, c, kernel_size, stride, pt, pl, ho, wo, _stream())
    return _trace('pool', None, y)
  return _trace('pool', None, _MaxPoolFn.apply(x.contiguous(), kernel_size, stride, geom))


class _GlobalMeanFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x):
    n, h, w, c = x.shape
    y = torch.empty((n, c), dtype=BF16, device=x.device)
    _lib.call('t2r_global_mean_fwd', _p(x), _p(y), n, h * w, c, _stream())
    ctx.shape = (n, h, w, c)
    return y

  @staticmethod
  def backward(ctx, dy):
    n, h, w, c = ctx.shape
    dx = torch.empty((n, h, w, c), dtype=BF16, device=dy.device)
    _lib.call('t2r_global_mean_bwd', _p(dy.contiguous()), _p(dx), n, h * w, c, _stream())
    return dx


def global_mean(x):
  """tf.reduce_mean over the spatial axes (film_resnet_model.py:611-616)."""
  _require_cuda(x, 'global_mean')
  if _HIGH_PRECISION:
    x = _hp_f32(x)
    n, h, w, c = x.shape
    y = torch.empty((n, c), dtype=F32, device=x.device)
    _lib.call('t2r_global_mean_f32_fwd', _p(x), _p(y), n, h * w, c, _stream())
    return y
  return _GlobalMeanFn.apply(x.contiguous())


class _AddContextFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, context, a):
    b, h, w, c = x.shape
    y = torch.empty((b * a, h, w, c), dtype=BF16, device=x.device)
    _lib.call('t2r_add_context_fwd', _p(x), _p(context), _p(y), b, a, h * w, c, _stream())
    ctx.geom = (b, a, h, w, c)
    return y

  @staticmethod
  def backward(ctx, dy):
    b, a, h, w, c = ctx.geom
    dy = dy.contiguous()
    dx = torch.empty((b, h, w, c), dtype=BF16, device=dy.device) if ctx.needs_input_grad[0] else None
    dctx = torch.empty((b * a, c), dtype=BF16, device=dy.device) if ctx.needs_input_grad[1] else None
    _lib.call('t2r_add_context_bwd', _p(dy), _p(dx), _p(dctx), b, a, h * w, c, _stream())
    return dx, dctx, None


class DeferredContext(object):
  """Inference-mode merge whose consumer is a batch norm: batch_norm() runs ONE pass
  relu((x + ctx) * scale + shift) instead of add, read, normalise, write (add_context(defer_for_bn=True))."""

  def __init__(self, x, context, a):
    self.x, self.context, self.a = x, context, a
    self.shape = (context.shape[0],) + tuple(x.shape[1:])
    self.device = x.device

  def run(self, scale, shift, relu):
    x, a = self.x, self.a
    b, h, w, c = x.shape
    y = torch.empty(self.shape, dtype=BF16, device=x.device)
    _lib.call('t2r_add_context_affine_fwd', _p(x), _p(self.context), _p(scale), _p(shift), _p(y), b, a, h * w, c,
              1 if relu else 0, _stream())
    return y

  def materialize(self):
    return _trace('add_context', None, _AddContextFn.apply(self.x, self.context, self.a))


def add_context(x, context, action_batch_size=1, defer_for_bn=False):
  """tile_batch(x, A) + context[:, None, None, :] without materialising the tile
  (research/qtopt/networks.py:513-522; research/dql_grasping_lib/tf_modules.py:74-93)."""
  _require_cuda(x, 'add_context')
  if context.shape[0] != x.shape[0] * action_batch_size:
    raise ValueError('context rows %d != batch %d * action_batch %d' % (context.shape[0], x.shape[0], action_batch_size))
  if _HIGH_PRECISION:
    x, context = _hp_f32(x), _hp_f32(context)
    b, h, w, c = x.shape
    y = torch.empty((b * action_batch_size, h, w, c), dtype=F32, device=x.device)
    _lib.call('t2r_add_context_f32_fwd', _p(x), _p(context), _p(y), b, action_batch_size, h * w, c, _stream())
    return _trace('add_context', None, y)
  if defer_for_bn and FOLD_INFERENCE_BN and not torch.is_grad_enabled():
    return DeferredContext(x.contiguous(), context.contiguous(), action_batch_size)
  return _trace('add_context', None, _AddContextFn.apply(x.contiguous(), context.contiguous(), action_batch_size))


class _ReluFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x):
    y = torch.empty_like(x)
    _lib.call('t2r_relu_fwd_bf16' if x.dtype == BF16 else 't2r_relu_f32_fwd', _p(x), _p(y), x.numel(), _stream())
    ctx.save_for_backward(y)
    return y

  @staticmethod
  def backward(ctx, dy):
    (y,) = ctx.saved_tensors
    dy = dy.contiguous()
    dx = torch.empty_like(dy)
    _lib.call('t2r_relu_bwd_bf16' if y.dtype == BF16 else 't2r_relu_f32_bwd', _p(dy), _p(y), _p(dx), dy.numel(), _stream())
    return dx


class _AddReluFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, a, b):
    y = torch.empty_like(a)
    _lib.call('t2r_add_relu_bf16', _p(a), _p(b), _p(y), a.numel(), _stream())
    ctx.save_for_backward(y)
    return y

  @staticmethod
  def backward(ctx, dy):
    (y,) = ctx.saved_tensors
    dy = dy.contiguous()
    g = torch.empty_like(dy)
    _lib.call('t2r_relu_bwd_bf16', _p(dy), _p(y), _p(g), dy.numel(), _stream())
    return g, g


def add_relu(a, b):
  """relu(a + b) on two bf16 NHWC tensors of the same shape in one pass: the shortcut add that closes a ResNet v1
  block (layers/film_resnet_model.py:156-166)."""
  _require_cuda(a, 'add_relu')
  _require_cuda(b, 'add_relu')
  if _HIGH_PRECISION:
    y = torch.empty_like(_hp_f32(a))
    _lib.call('t2r_add_f32', _p(_hp_f32(a)), _p(_hp_f32(b)), _p(y), y.numel(), _stream())
    _lib.call('t2r_relu_f32_fwd', _p(y), _p(y), y.numel(), _stream())
    return y
  if a.shape != b.shape or a.dtype != BF16 or b.dtype != BF16 or a.numel() % 8:
    raise ValueError('add_relu expects two bf16 tensors of the same shape (a multiple of 8 elements)')
  return _AddReluFn.apply(a.contiguous(), b.contiguous())


def relu(x):
  """tf.nn.relu on a bf16 or fp32 CUDA tensor (stand-alone; conv / norm epilogues fuse their own)."""
  _require_cuda(x, 'relu')
  if x.dtype not in (BF16, F32):
    raise ValueError('relu expects bf16 or fp32 activations')
  if x.numel() == 0:
    return x
  return _ReluFn.apply(x.contiguous())


class _NPairsLossFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, anchor, positive, reg_lambda):
    b, d = anchor.shape
    dev = anchor.device
    sim = torch.empty((b, b), dtype=F32, device=dev)
    rows = torch.empty(b, dtype=F32, device=dev)
    loss = torch.empty(1, dtype=F32, device=dev)
    da, dp = torch.empty_like(anchor), torch.empty_like(positive)
    _lib.call('t2r_npairs_loss', _p(anchor), _p(positive), b, d, float(reg_lambda), _p(sim), _p(rows), _p(loss),
              _p(da), _p(dp), _stream())
    ctx.save_for_backward(da, dp)
    return loss.reshape(())

  @staticmethod
  def backward(ctx, dloss):
    da, dp = ctx.saved_tensors
    return da * dloss, dp * dloss, None


def npairs_loss(anchor, positive, reg_lambda=0.002):
  """tf.contrib.losses.metric_learning.npairs_loss(labels=range(B), anchor, positive, reg_lambda) on fp32
  [B, D] CUDA embeddings (research/grasp2vec/losses.py:176-178)."""
  _require_cuda(anchor, 'npairs_loss')
  if anchor.dtype != F32 or positive.dtype != F32 or anchor.shape != positive.shape or anchor.dim() != 2:
    raise ValueError('npairs_loss expects two fp32 [B, D] tensors of the same shape')
  return _NPairsLossFn.apply(anchor.contiguous(), positive.contiguous(), reg_lambda)


class _TripletSemihardFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, emb, labels, margin):
    m, d = emb.shape
    ws = torch.empty(3 * m * m + m + 2, dtype=F32, device=emb.device)
    loss = torch.empty(1, dtype=F32, device=emb.device)
    d_emb = torch.empty_like(emb)
    _lib.call('t2r_triplet_semihard_loss', _p(emb), _p(labels), m, d, float(margin), _p(ws), _p(loss), _p(d_emb),
              _stream())
    ctx.save_for_backward(d_emb)
    return loss.reshape(())

  @staticmethod
  def backward(ctx, dloss):
    (d_emb,) = ctx.saved_tensors
    return d_emb * dloss, None, None


def triplet_semihard_loss(labels, embeddings, margin=1.0):
  """tf.contrib.losses.metric_learning.triplet_semihard_loss on fp32 [M, D] CUDA embeddings with int labels
  (research/grasp2vec/losses.py:69-71; mining restated in layers/tec.py:322-383)."""
  _require_cuda(embeddings, 'triplet_semihard_loss')
  if embeddings.dtype != F32 or embeddings.dim() != 2:
    raise ValueError('triplet_semihard_loss expects fp32 [M, D] embeddings')
  labels = labels.to(device=embeddings.device, dtype=torch.int32).contiguous()
  return _TripletSemihardFn.apply(embeddings.contiguous(), labels, margin)


class _CastFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, to_bf16):
    y = torch.empty(x.shape, dtype=BF16 if to_bf16 else F32, device=x.device)
    _lib.call('t2r_cast_f32_to_bf16' if to_bf16 else 't2r_cast_bf16_to_f32', _p(x), _p(y), x.numel(), _stream())
    ctx.to_bf16 = to_bf16
    return y

  @staticmethod
  def backward(ctx, dy):
    dy = dy.contiguous()
    dx = torch.empty(dy.shape, dtype=F32 if ctx.to_bf16 else BF16, device=dy.device)
    _lib.call('t2r_cast_bf16_to_f32' if ctx.to_bf16 else 't2r_cast_f32_to_bf16', _p(dy), _p(dx), dy.numel(), _stream())
    return dx, None


def to_bf16(x):
  if _HIGH_PRECISION:      # activations stay fp32 in the high-precision mode
    return x if x.dtype == F32 else _CastFn.apply(x.contiguous(), False)
  return x if x.dtype == BF16 else _CastFn.apply(x.contiguous(), True)


def to_f32(x):
  return x if x.dtype == F32 else _CastFn.apply(x.contiguous(), False)


# ---------------------------------------------------------------------------------------------
# fp32 fully connected (tiny layers: action context input, logits)
# ---------------------------------------------------------------------------------------------
class _Fc32Fn(torch.autograd.Function):
  """y[M,N] = x[M,K] @ W[K,N] + sum_rows(bias[R,N]); W is stored in the TF [in,out] layout."""

  @staticmethod
  def forward(ctx, x, anchor, wv, bv):
    m, k = x.shape
    n = wv.shape[1]
    st = _stream()
    y = torch.empty((m, n), dtype=F32, device=x.device)
    _lib.call('t2r_sgemm', 0, 0, m, n, k, 1.0, _p(x), k, _p(wv.data), n, 0.0, _p(y), n, st)
    if bv is not None:
      r = bv.shape[0]
      if r == 1:
        bias = bv.data
      else:
        bias = torch.empty(n, dtype=F32, device=x.device)
        _lib.call('t2r_colsum_f32', _p(bv.data), _p(bias), r, n, st)
      _lib.call('t2r_bias_add_f32', _p(y), _p(bias), m, n, st)
    ctx.wv, ctx.bv = wv, bv
    ctx.save_for_backward(x)
    return y

  @staticmethod
  def backward(ctx, dy):
    (x,) = ctx.saved_tensors
    wv, bv = ctx.wv, ctx.bv
    m, k = x.shape
    n = wv.shape[1]
    st = _stream()
    dy = dy.contiguous()
    if wv.trainable:   # dW[K,N] = x^T dy
      _lib.call('t2r_sgemm', 1, 0, k, n, m, 1.0, _p(x), k, _p(dy), n, 0.0, _p(wv.grad), n, st)
      wv.grad_ready()
    if bv is not None and bv.trainable:
      db = torch.empty(n, dtype=F32, device=x.device)
      _lib.call('t2r_colsum_f32', _p(dy), _p(db), m, n, st)
      r = bv.shape[0]
      ones = torch.ones(r, dtype=F32, device=x.device)   # every summed bias row receives db
      _lib.call('t2r_sgemm', 0, 0, r, n, 1, 1.0, _p(ones), 1, _p(db), n, 0.0, _p(bv.grad), n, st)
      bv.grad_ready()
    dx = None
    if ctx.needs_input_grad[0]:   # dx[M,K] = dy W^T
      dx = torch.empty((m, k), dtype=F32, device=x.device)
      _lib.call('t2r_sgemm', 0, 1, m, k, n, 1.0, _p(dy), n, _p(wv.data), n, 0.0, _p(dx), k, st)
    return dx, None, None, None


def dense_f32(x, units, scope='fc', bias_rows=1, initializer=None, regularize=True, trainable=True,
              names=('weights', 'biases'), bias_initializer=0.0):
  """fp32 slim.fully_connected for inner dimensions that are not multiples of 64.

  bias_rows > 1 models `tf.add_n` of several FC blocks that share the output (the reference's
  fcgrasp_* blocks, networks.py:481-501): their weights are the row blocks of W, their biases the
  rows of a [bias_rows, units] matrix that is summed."""
  _require_cuda(x, 'dense_f32')
  vs = current_store()
  k = x.shape[1]
  with vs.scope(scope):
    wv = vs.get_variable(names[0], (k, units), initializer or glorot_uniform(k, units), trainable, regularize,
                         'fc32', None)
    bv = vs.get_variable(names[1], (bias_rows, units), bias_initializer, trainable, False, 'fc32', None) if bias_rows else None
  if not vs.finalized:
    for v in (wv, bv):
      if v is not None and v.grad is None:
        v.grad = torch.zeros(v.shape, dtype=F32, device=x.device)
  return _trace('fc32', scope, _Fc32Fn.apply(x.contiguous(), vs.anchor, wv, bv))


# ---------------------------------------------------------------------------------------------
# fp32 layers of the small pose_env networks (csrc/vision_small.cu): 32-channel convolutions, slim
# layer_norm, the tile + broadcast-add action merge and the bias-transform concat.
# ---------------------------------------------------------------------------------------------
def xavier_uniform(fan_in, fan_out):
  """slim.xavier_initializer() (uniform): limit = sqrt(6 / (fan_in + fan_out))."""
  return glorot_uniform(fan_in, fan_out)


def _ensure_grad(vs, device, *variables):
  if not vs.finalized:
    for v in variables:
      if v is not None and v.trainable and v.grad is None:
        v.grad = torch.zeros(v.shape, dtype=F32, device=device)


class _DirectConvFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, anchor, wv, bv, geom):
    n, h, w, cin = x.shape
    kh, kw, _, cout = wv.shape
    stride, pt, pl, ho, wo = geom
    y = torch.empty((n, ho, wo, cout), dtype=F32, device=x.device)
    ctx.dims = (n, h, w, cin, cout, kh, kw, stride, pt, pl, ho, wo)
    _lib.call('t2r_conv2d_direct_f32_fwd', _p(x), _p(wv.data), _p(bv.data if bv is not None else None), _p(y),
              *ctx.dims, _stream())
    ctx.wv, ctx.bv = wv, bv
    ctx.save_for_backward(x)
    return y

  @staticmethod
  def backward(ctx, dy):
    (x,) = ctx.saved_tensors
    wv, bv = ctx.wv, ctx.bv
    dy = dy.contiguous()
    st = _stream()
    if wv.trainable:
      _lib.call('t2r_conv2d_direct_f32_wgrad', _p(x), _p(dy), _p(wv.grad), *ctx.dims, st)
      wv.grad_ready()
    if bv is not None and bv.trainable:
      _lib.call('t2r_colsum_f32', _p(dy), _p(bv.grad), dy.numel() // dy.shape[-1], dy.shape[-1], st)
      bv.grad_ready()
    dx = None
    if ctx.needs_input_grad[0]:
      dx = torch.empty_like(x)
      _lib.call('t2r_conv2d_direct_f32_dgrad', _p(dy), _p(wv.data), _p(dx), *ctx.dims, st)
    return dx, None, None, None, None


def conv2d_f32(x, filters, kernel_size, stride=1, padding='VALID', use_bias=True, scope='conv', initializer=None,
               bias_initializer=0.0, regularize=False, trainable=True):
  """slim.conv2d in fp32 for layers below one tensor-core tile (3 / 32 channels): x fp32 NHWC, weights in the
  TF HWIO layout under `<scope>/weights`, optional `<scope>/biases`."""
  _require_cuda(x, 'conv2d_f32')
  if x.dtype != F32:
    raise ValueError('conv2d_f32 expects fp32 activations')
  kh, kw = (kernel_size, kernel_size) if isinstance(kernel_size, int) else kernel_size
  n, h, w, cin = x.shape
  ho, wo, pt, pl = conv_geometry(h, w, kh, kw, stride, padding)
  vs = current_store()
  with vs.scope(scope):
    wv = vs.get_variable('weights', (kh, kw, cin, filters), initializer or xavier_uniform(kh * kw * cin, kh * kw * filters),
                         trainable, regularize, 'other', None)
    bv = vs.get_variable('biases', (filters,), bias_initializer, trainable, False, 'other', None) if use_bias else None
  _ensure_grad(vs, x.device, wv, bv)
  return _trace('conv32', scope, _DirectConvFn.apply(x.contiguous(), vs.anchor, wv, bv, (stride, pt, pl, ho, wo)))


class _LayerNormFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, anchor, gv, bv, eps, relu):
    n, c = x.shape[0], x.shape[-1]
    d = x.numel() // n
    y = torch.empty_like(x)
    mean = torch.empty(n, dtype=F32, device=x.device)
    rstd = torch.empty(n, dtype=F32, device=x.device)
    _lib.call('t2r_layer_norm_f32_fwd', _p(x), _p(gv.data), _p(bv.data), _p(y), _p(mean), _p(rstd), n, d, c, eps,
              int(relu), _stream())
    ctx.gv, ctx.bv, ctx.relu = gv, bv, relu
    ctx.save_for_backward(x, mean, rstd)
    return y

  @staticmethod
  def backward(ctx, dy):
    x, mean, rstd = ctx.saved_tensors
    gv, bv = ctx.gv, ctx.bv
    n, c = x.shape[0], x.shape[-1]
    dx = torch.empty_like(x)
    want = gv.trainable
    _lib.call('t2r_layer_norm_f32_bwd', _p(x), _p(dy.contiguous()), _p(gv.data), _p(bv.data), _p(mean), _p(rstd), _p(dx),
              _p(gv.grad if want else None), _p(bv.grad if want else None), n, x.numel() // n, c, int(ctx.relu), _stream())
    if want:
      gv.grad_ready()
      bv.grad_ready()
    return dx, None, None, None, None, None


def layer_norm(x, scope='LayerNorm', relu=False, eps=1e-12, trainable=True):
  """slim.layer_norm (center, scale; moments over every non-batch axis, parameters per channel) with an optional
  fused ReLU.  x: fp32 [N, ..., C]."""
  _require_cuda(x, 'layer_norm')
  if x.dtype != F32:
    raise ValueError('layer_norm expects fp32 activations')
  c = x.shape[-1]
  vs = current_store()
  with vs.scope(scope):
    bv = vs.get_variable('beta', (c,), 0.0, trainable, False, 'other', None)
    gv = vs.get_variable('gamma', (c,), 1.0, trainable, False, 'other', None)
  _ensure_grad(vs, x.device, gv, bv)
  return _trace('layer_norm', scope, _LayerNormFn.apply(x.contiguous(), vs.anchor, gv, bv, eps, relu))


class _SpatialSoftmaxF32Fn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, want_map):
    n, h, w, c = x.shape
    points = torch.empty((n, 2 * c), dtype=F32, device=x.device)
    heat = torch.empty_like(x) if want_map else None
    _lib.call('t2r_spatial_softmax_f32_fwd', _p(x), _p(points), _p(heat), n, h, w, c, _stream())
    ctx.save_for_backward(x, points)
    if want_map:
      ctx.mark_non_differentiable(heat)
      return points, heat
    return points

  @staticmethod
  def backward(ctx, dpoints, _dheat=None):
    x, points = ctx.saved_tensors
    n, h, w, c = x.shape
    dx = torch.empty_like(x)
    _lib.call('t2r_spatial_softmax_f32_bwd', _p(x), _p(points), _p(dpoints.contiguous().float()), _p(dx), n, h, w, c,
              _stream())
    return dx, None


class _TileAddContextFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, context):
    nx, h, w, c = x.shape
    nc = context.shape[0]
    y = torch.empty((nc, h, w, c), dtype=F32, device=x.device)
    _lib.call('t2r_tile_add_context_f32_fwd', _p(x), _p(context), _p(y), nx, nc, h * w, c, _stream())
    ctx.dims = (nx, nc, h, w, c)
    return y

  @staticmethod
  def backward(ctx, dy):
    nx, nc, h, w, c = ctx.dims
    dy = dy.contiguous()
    dx = torch.empty((nx, h, w, c), dtype=F32, device=dy.device) if ctx.needs_input_grad[0] else None
    dc = torch.empty((nc, c), dtype=F32, device=dy.device) if ctx.needs_input_grad[1] else None
    _lib.call('t2r_tile_add_context_f32_bwd', _p(dy), _p(dx), _p(dc), nx, nc, h * w, c, _stream())
    return dx, dc


def tile_add_context(net, context):
  """The pose_env critic's action merge (research/pose_env/pose_env_models.py:141-149): the image batch is tiled
  (tf.tile: row j of the result is net[j mod B]) up to the context batch and context [Bc, C] is added at every
  position.  fp32."""
  _require_cuda(net, 'tile_add_context')
  if net.dtype != F32 or context.dtype != F32:
    raise ValueError('tile_add_context expects fp32 tensors')
  if context.shape[0] % net.shape[0] != 0 or context.shape[1] != net.shape[-1]:
    raise ValueError('context %s does not tile over net %s' % (tuple(context.shape), tuple(net.shape)))
  return _TileAddContextFn.apply(net.contiguous(), context.contiguous())


class _BiasTransformFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, anchor, bv):
    ctx.bv, ctx.k = bv, x.shape[1]
    return torch.cat([x, bv.data.reshape(1, -1).expand(x.shape[0], -1)], 1)

  @staticmethod
  def backward(ctx, dy):
    bv, k = ctx.bv, ctx.k
    if bv.trainable:
      tail = dy[:, k:].contiguous()
      _lib.call('t2r_colsum_f32', _p(tail), _p(bv.grad), tail.shape[0], tail.shape[1], _stream())
      bv.grad_ready()
    return dy[:, :k].contiguous(), None, None


def bias_transform(x, size, scope='BiasAdd', initializer=0.01):
  """vision_layers.py:325-329: concat([x, zeros[B, size] + biases], 1) with a learned bias vector."""
  _require_cuda(x, 'bias_transform')
  vs = current_store()
  with vs.scope(scope):
    bv = vs.get_variable('biases', (size,), initializer, True, False, 'other', None)
  _ensure_grad(vs, x.device, bv)
  return _BiasTransformFn.apply(x.contiguous(), vs.anchor, bv)



class _EluFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x):
    y = torch.empty_like(x)
    _lib.call('t2r_elu_f32_fwd', _p(x), _p(y), x.numel(), _stream())
    ctx.save_for_backward(y)
    return y

  @staticmethod
  def backward(ctx, dy):
    (y,) = ctx.saved_tensors
    dy = dy.contiguous()
    dx = torch.empty_like(dy)
    _lib.call('t2r_elu_f32_bwd', _p(dy), _p(y), _p(dx), dy.numel(), _stream())
    return dx


def elu(x):
  """tf.nn.elu on an fp32 CUDA tensor."""
  _require_cuda(x, 'elu')
  if x.dtype != F32:
    raise ValueError('elu expects fp32 activations')
  return _EluFn.apply(x.contiguous())


class _BnInferF32Fn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, anchor, gv, bv, mv, vv, eps):
    c = x.shape[-1]
    y = torch.empty_like(x)
    _lib.call('t2r_bn_infer_f32_fwd', _p(x), _p(gv.data), _p(bv.data), _p(mv.data), _p(vv.data), _p(y), x.numel() // c, c,
              eps, _stream())
    ctx.vars, ctx.eps = (gv, bv, mv, vv), eps
    ctx.save_for_backward(x)
    return y

  @staticmethod
  def backward(ctx, dy):
    (x,) = ctx.saved_tensors
    gv, bv, mv, vv = ctx.vars
    c = x.shape[-1]
    dx = torch.empty_like(x)
    want = gv.trainable
    _lib.call('t2r_bn_infer_f32_bwd', _p(x), _p(dy.contiguous()), _p(gv.data), _p(mv.data), _p(vv.data), _p(dx),
              _p(gv.grad if want else None), _p(bv.grad if want else None), x.numel() // c, c, ctx.eps, _stream())
    if want:
      gv.grad_ready()
      bv.grad_ready()
    return dx, None, None, None, None, None, None


def batch_normalization_f32(x, scope, eps=1e-3, trainable=True):
  """tf.layers.batch_normalization(x, name=scope) with its default training=False on an fp32 [..., C] tensor: the moving
  statistics (zeros / ones unless a checkpoint says otherwise) normalise, gamma / beta train (utils/mocks.py:171-172)."""
  _require_cuda(x, 'batch_normalization_f32')
  if x.dtype != F32:
    raise ValueError('batch_normalization_f32 expects fp32 activations')
  c = x.shape[-1]
  vs = current_store()
  with vs.scope(scope):
    gv = vs.get_variable('gamma', (c,), 1.0, trainable, False, 'other', None)
    bv = vs.get_variable('beta', (c,), 0.0, trainable, False, 'other', None)
    mv = vs.get_variable('moving_mean', (c,), 0.0, False, False, 'other', None)
    vv = vs.get_variable('moving_variance', (c,), 1.0, False, False, 'other', None)
  _ensure_grad(vs, x.device, gv, bv)
  return _BnInferF32Fn.apply(x.contiguous(), vs.anchor, gv, bv, mv, vv, eps)


class _FilmReluF32Fn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, film):
    n, c = x.shape[0], x.shape[-1]
    hw = x.numel() // (n * c)
    y = torch.empty_like(x)
    _lib.call('t2r_film_relu_f32_fwd', _p(x), _p(film), _p(y), n, hw, c, _stream())
    ctx.save_for_backward(x, film)
    return y

  @staticmethod
  def backward(ctx, dy):
    x, film = ctx.saved_tensors
    n, c = x.shape[0], x.shape[-1]
    dx, dfilm = torch.empty_like(x), torch.empty_like(film)
    _lib.call('t2r_film_relu_f32_bwd', _p(x), _p(film), _p(dy.contiguous()), _p(dx), _p(dfilm), n, x.numel() // (n * c), c,
              _stream())
    return dx, dfilm


def film_relu_f32(x, film):
  """relu((1 + gamma[n]) * x + beta[n]) on fp32 [N, ..., C] with film = [N, 2C] = (gammas | betas): the FiLM
  conditioning of the spatial-softmax tower (layers/vision_layers.py:100-141)."""
  _require_cuda(x, 'film_relu_f32')
  if x.dtype != F32 or film.dtype != F32 or film.shape != (x.shape[0], 2 * x.shape[-1]):
    raise ValueError('film_relu_f32 expects fp32 x [N, ..., C] and film [N, 2C]')
  return _FilmReluF32Fn.apply(x.contiguous(), film.contiguous())


class _BnTrainF32Fn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, x, anchor, gv, bv, mv, vv, eps, decay, relu):
    c = x.shape[-1]
    rows = x.numel() // c
    y = torch.empty_like(x)
    mean = torch.empty(c, dtype=F32, device=x.device)
    rstd = torch.empty(c, dtype=F32, device=x.device)
    _lib.call('t2r_bn_train_f32_fwd', _p(x), _p(gv.data if gv is not None else None), _p(bv.data), _p(y), _p(mv.data),
              _p(vv.data), _p(mean), _p(rstd), rows, c, eps, decay, int(relu), _stream())
    ctx.vars, ctx.relu = (gv, bv), relu
    ctx.save_for_backward(x, y, mean, rstd)
    return y

  @staticmethod
  def backward(ctx, dy):
    x, y, mean, rstd = ctx.saved_tensors
    gv, bv = ctx.vars
    c = x.shape[-1]
    dx = torch.empty_like(x)
    dgamma = gv.grad if (gv is not None and gv.trainable) else None
    dbeta = bv.grad if bv.trainable else None
    _lib.call('t2r_bn_train_f32_bwd', _p(x), _p(y), _p(dy.contiguous()), _p(gv.data if gv is not None else None), _p(mean),
              _p(rstd), _p(dx), _p(dgamma), _p(dbeta), x.numel() // c, c, int(ctx.relu), _stream())
    if dgamma is not None:
      gv.grad_ready()
    if dbeta is not None:
      bv.grad_ready()
    return dx, None, None, None, None, None, None, None, None


def batch_norm_f32(x, is_training, scope='BatchNorm', scale=False, decay=0.99, eps=1e-4, relu=False, trainable=True):
  """slim.batch_norm on an fp32 [..., C] tensor (the normalizer_fn=slim.batch_norm variant of
  layers/vision_layers.py:72-86: decay .99, epsilon 1e-4, scale only on the last 1x1 convolution): batch statistics
  and moving-average update in training, moving statistics otherwise; optional fused ReLU."""
  _require_cuda(x, 'batch_norm_f32')
  if x.dtype != F32:
    raise ValueError('batch_norm_f32 expects fp32 activations')
  c = x.shape[-1]
  vs = current_store()
  with vs.scope(scope):
    gv = vs.get_variable('gamma', (c,), 1.0, trainable, False, 'other', None) if scale else None
    bv = vs.get_variable('beta', (c,), 0.0, trainable, False, 'other', None)
    mv = vs.get_variable('moving_mean', (c,), 0.0, False, False, 'other', None)
    vv = vs.get_variable('moving_variance', (c,), 1.0, False, False, 'other', None)
  _ensure_grad(vs, x.device, gv, bv)
  if is_training and torch.is_grad_enabled():
    return _BnTrainF32Fn.apply(x.contiguous(), vs.anchor, gv, bv, mv, vv, float(eps), float(decay), relu)
  ones = gv if gv is not None else None
  if ones is None:   # scale=False: gamma is the constant one
    class _One(object):
      data = torch.ones(c, dtype=F32, device=x.device)
      grad = None
      trainable = False
    ones = _One()
  y = _BnInferF32Fn.apply(x.contiguous(), vs.anchor, ones, bv, mv, vv, float(eps))
  return relu_f32(y) if relu else y


def relu_f32(x):
  return _ReluFn.apply(x.contiguous())


# ---------------------------------------------------------------------------------------------
# losses
# ---------------------------------------------------------------------------------------------
class _SigmoidLogLossFn(torch.autograd.Function):

  @staticmethod
  def forward(ctx, logit, label):
    n = logit.numel()
    q = torch.empty_like(logit)
    dlogit = torch.empty_like(logit)
    loss = torch.zeros(1, dtype=F32, device=logit.device)
    _lib.call('t2r_sigmoid_logloss', _p(logit), _p(label), _p(q), _p(loss), _p(dlogit), n, _stream())
    ctx.save_for_backward(dlogit)
    ctx.mark_non_differentiable(q)
    return loss[0], q

  @staticmethod
  def backward(ctx, dloss, _dq):
    (dlogit,) = ctx.saved_tensors
    return dlogit * dloss, None


class _WeightedLossesFn(torch.autograd.Function):
  """t2r_weighted_losses: every segment's loss and gradient in one launch (csrc/losses.cu)."""

  @staticmethod
  def forward(ctx, specs, *preds):
    dev = preds[0].device
    n = len(specs)
    segs = (_lib.LossSegment * n)()
    losses = torch.empty(n + 1, dtype=F32, device=dev)
    keep, dpreds, sigmoids = [], [], []
    for i, (spec, pred) in enumerate(zip(specs, preds)):
      seg = segs[i]
      seg.struct_size = C.sizeof(_lib.LossSegment)
      seg.kind = {'huber': _lib.T2R_LOSS_HUBER, 'mse': _lib.T2R_LOSS_MSE, 'sigmoid_log': _lib.T2R_LOSS_SIGMOID_LOG}[spec['kind']]
      seg.predictions = pred.data_ptr()
      labels = spec['labels']
      if torch.is_tensor(labels):
        labels = labels.to(device=dev, dtype=F32).contiguous()
        keep.append(labels)
        seg.labels = labels.data_ptr()
      else:
        seg.labels, seg.label_const = None, float(labels)
      mask = spec.get('row_mask')
      if mask is not None:
        mask = mask.to(device=dev, dtype=F32).contiguous()
        keep.append(mask)
        seg.row_mask = mask.data_ptr()
      seg.row_mask_is_complement = 1 if spec.get('complement') else 0
      seg.n, seg.cols = pred.numel(), pred.shape[-1]
      seg.row_mod = int(spec.get('row_mod', 0))
      seg.in_total = 1 if spec.get('in_total', True) else 0
      seg.weight, seg.delta = float(spec.get('weight', 1.0)), float(spec.get('delta', 1.0))
      d = torch.empty_like(pred) if spec.get('differentiable', True) else None
      dpreds.append(d)
      seg.dpredictions = d.data_ptr() if d is not None else None
      q = torch.empty_like(pred) if spec['kind'] == 'sigmoid_log' else None
      sigmoids.append(q)
      seg.sigmoid_out = q.data_ptr() if q is not None else None
    _lib.call('t2r_weighted_losses', segs, n, _p(losses), _stream())
    ctx.in_total = [bool(sp.get('in_total', True)) for sp in specs]
    ctx.n = n
    ctx.save_for_backward(*[d if d is not None else losses.new_zeros(0) for d in dpreds])
    outs = [q for q in sigmoids if q is not None]
    ctx.mark_non_differentiable(*outs)
    return (losses,) + tuple(outs)

  @staticmethod
  def backward(ctx, dlosses, *_):
    grads = [None]
    for i, d in enumerate(ctx.saved_tensors):
      if d.numel() == 0:
        grads.append(None)
        continue
      g = dlosses[i] + dlosses[ctx.n] if ctx.in_total[i] else dlosses[i]
      grads.append(d * g)
    return tuple(grads)


def weighted_losses(specs):
  """Several tf.losses-style weighted losses (Reduction.SUM_BY_NONZERO_WEIGHTS) in one kernel launch.

  specs: list of dicts - kind 'huber' | 'mse' | 'sigmoid_log' (log loss of sigmoid(predictions)), predictions (fp32
  CUDA tensor [..., cols]; logits for 'sigmoid_log'), labels (tensor of the same shape or a float), weight (float),
  row_mask ([rows] tensor multiplied into the weights; complement=True uses 1 - row_mask), row_mod (> 0: only rows with
  row % row_mod == 0 count), delta (huber), in_total, differentiable.  Returns (losses [len(specs) + 1] with the
  in_total sum last, list of sigmoid(predictions) per 'sigmoid_log' spec in order).
  Reference: research/bcz/model.py:476-585."""
  if not specs or len(specs) > _lib.T2R_MAX_LOSS_SEGMENTS:
    raise ValueError('weighted_losses takes 1..%d segments' % _lib.T2R_MAX_LOSS_SEGMENTS)
  preds = []
  for spec in specs:
    _require_cuda(spec['predictions'], 'weighted_losses')
    preds.append(to_f32(spec['predictions']).contiguous())
  meta = [{k: v for k, v in spec.items() if k != 'predictions'} for spec in specs]
  out = _WeightedLossesFn.apply(meta, *preds)
  return out[0], list(out[1:])


def sigmoid_log_loss(logit, label):
  """tf.losses.log_loss(label, sigmoid(logit)) computed with the reference's eps=1e-7; returns
  (loss, q_predicted)."""
  _require_cuda(logit, 'sigmoid_log_loss')
  return _SigmoidLogLossFn.apply(to_f32(logit).contiguous(), label.to(F32).contiguous())


def sigmoid(logit):
  logit = to_f32(logit).contiguous()
  q = torch.empty_like(logit)
  _lib.call('t2r_sigmoid_f32', _p(logit), _p(q), logit.numel(), _stream())
  return q


def l2_regularization_loss(l2, vs=None):
  """slim.l2_regularizer(l2)(w) summed over regularised weights = l2 * sum(w^2) / 2."""
  vs = vs or current_store()
  out = torch.zeros(1, dtype=F32, device=vs.device)
  if vs.finalized and vs.n_decay > 0:
    _lib.call('t2r_sumsq_f32', _p(vs.flat), _p(out), vs.n_decay, 0.5 * l2, _stream())
  return out[0]
