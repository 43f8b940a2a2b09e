"""Batch-norm backward through the 1x1 consumer's GEMMs (t2r_conv2d_wgrad_bnsums, t2r_bn_backward_gemm_finalize,
t2r_conv2d_dgrad_bnapply) against the data gradient + reduction + apply path it replaces and against a float64
restatement on the same bf16 inputs.

Node:  z = relu(scale * x + shift), y = conv1x1(z, W), scale = gamma * invstd, shift = beta - mean * scale.
Given dy: dW = dy^T z, g = [z > 0] * (dy W), dbeta = sum g, dgamma = invstd * (sum g x - mean * dbeta) and
dx = scale * (g - dbeta / rows - xhat * dgamma * invstd / rows) (+ dpass), xhat = (x - mean) * invstd."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64


def _p(t):
  return None if t is None else C.c_void_p(t.data_ptr())


def _desc(n, h, w, cin, cout):
  from tensor2robot_b200 import _lib
  d = _lib.ConvDesc()
  d.struct_size = C.sizeof(_lib.ConvDesc)
  d.N, d.H, d.W, d.Cin, d.Cout = n, h, w, cin, cout
  d.KH = d.KW = d.stride = 1
  d.pad_top = d.pad_left = d.flags = 0
  d.Ho, d.Wo = h, w
  return d


def _node(n, h, w, c, cout, dpass, gamma_mode='normal', seed=0):
  g = torch.Generator(device='cpu').manual_seed(seed)
  x = (torch.randn(n, h, w, c, generator=g) * 1.5 + 0.3).to(BF16).cuda()
  wt = (torch.randn(cout, c, generator=g) / np.sqrt(c)).to(BF16).cuda()
  dy = torch.randn(n, h, w, cout, generator=g).to(BF16).cuda()
  dp = torch.randn(n, h, w, c, generator=g).to(BF16).cuda() if dpass else None
  gamma = 0.5 + torch.rand(c, generator=g)
  beta = 0.3 * torch.randn(c, generator=g)
  if gamma_mode == 'negative':
    gamma = -gamma
  elif gamma_mode == 'zero':
    gamma = gamma * 1e-7
  elif gamma_mode == 'masked':
    beta[:3] = -1e4             # channels 0-2: scale * x + shift < 0 everywhere
  xf = x.double().reshape(-1, c)
  mean = xf.mean(0)
  invstd = 1.0 / torch.sqrt(xf.var(0, unbiased=False) + 1e-3)
  mean, invstd = mean.float(), invstd.float()
  scale = gamma.cuda().float() * invstd
  shift = beta.cuda().float() - mean * scale
  return dict(x=x, w=wt, wd=wt.t().contiguous(), dy=dy, dpass=dp, mean=mean, invstd=invstd, scale=scale, shift=shift)


def _reference(t):
  """float64 restatement on the bf16 inputs and the fp32 batch-norm parameters."""
  c = t['x'].shape[-1]
  x = t['x'].double().reshape(-1, c)
  rows = x.shape[0]
  sc, sh, mean, invstd = (t[k].double() for k in ('scale', 'shift', 'mean', 'invstd'))
  zl = x * sc + sh
  m = (zl > 0).double()
  dy = t['dy'].double().reshape(rows, -1)
  w = t['w'].double()
  dw = dy.t() @ (m * zl)
  gg = m * (dy @ w)
  dbeta = gg.sum(0)
  dgamma = invstd * ((gg * x).sum(0) - mean * dbeta)
  dx = sc * (gg - dbeta / rows - (x - mean) * invstd * dgamma * invstd / rows)
  if t['dpass'] is not None:
    dx = dx + t['dpass'].double().reshape(rows, c)
  return dict(dx=dx, dw=dw, dgamma=dgamma, dbeta=dbeta)


def _old_path(t):
  """t2r_bn_apply + plain wgrad on z, plain dgrad into g, t2r_bn_backward (reduction + apply)."""
  from tensor2robot_b200 import _lib
  n, h, w, c = t['x'].shape
  cout = t['w'].shape[0]
  rows = n * h * w
  d = _desc(n, h, w, c, cout)
  z = torch.empty_like(t['x'])
  _lib.call('t2r_bn_apply', _p(t['x']), _p(z), rows, c, _p(t['scale']), _p(t['shift']), None, h * w, 1, None)
  dw = torch.zeros(cout, c, dtype=F32, device='cuda')
  gbuf = torch.empty_like(t['x'])
  red = torch.zeros(2 * c, dtype=F64, device='cuda')
  dgamma = torch.empty(c, dtype=F32, device='cuda')
  dbeta = torch.empty(c, dtype=F32, device='cuda')
  dx = torch.empty_like(t['x'])
  torch.cuda.synchronize()
  l0 = _lib.launch_count()
  _lib.call('t2r_conv2d_wgrad', C.byref(d), _p(z), _p(t['dy']), _p(dw), None)
  _lib.call('t2r_conv2d_dgrad', C.byref(d), _p(t['dy']), _p(t['wd']), _p(gbuf), 0, None)
  _lib.call('t2r_bn_backward', _p(gbuf), _p(t['x']), _p(t['dpass']), _p(dx), rows, c, None, _p(t['mean']),
            _p(t['invstd']), _p(t['scale']), _p(t['shift']), 1, _p(red), _p(dgamma), _p(dbeta), None)
  launches = _lib.launch_count() - l0
  torch.cuda.synchronize()
  return dict(dx=dx, dw=dw, dgamma=dgamma, dbeta=dbeta), launches


def _new_path(t):
  from tensor2robot_b200 import _lib
  n, h, w, c = t['x'].shape
  cout = t['w'].shape[0]
  rows = n * h * w
  d = _desc(n, h, w, c, cout)
  assert _lib.lib().t2r_conv2d_dgrad_bnapply_supported(C.byref(d)) == 1
  dw = torch.zeros(cout, c, dtype=F32, device='cuda')
  sums = torch.zeros(2 * c, dtype=F64, device='cuda')
  coef = torch.empty(2 * c, dtype=F32, device='cuda')
  dgamma = torch.empty(c, dtype=F32, device='cuda')
  dbeta = torch.empty(c, dtype=F32, device='cuda')
  dx = torch.empty_like(t['x'])
  torch.cuda.synchronize()
  l0 = _lib.launch_count()
  _lib.call('t2r_conv2d_wgrad_bnsums', C.byref(d), _p(t['x']), _p(t['scale']), _p(t['shift']), _p(t['dy']),
            _p(t['wd']), _p(dw), _p(sums), None)
  _lib.call('t2r_bn_backward_gemm_finalize', _p(sums), rows, c, _p(t['mean']), _p(t['invstd']), _p(t['scale']),
            _p(dgamma), _p(dbeta), _p(coef), None)
  _lib.call('t2r_conv2d_dgrad_bnapply', C.byref(d), _p(t['dy']), _p(t['wd']), _p(t['x']), _p(t['scale']),
            _p(t['shift']), _p(coef), _p(t['dpass']), _p(dx), None)
  launches = _lib.launch_count() - l0
  torch.cuda.synchronize()
  return dict(dx=dx, dw=dw, dgamma=dgamma, dbeta=dbeta), launches


def _rel(a, ref):
  a = a.double().reshape(ref.shape)
  return float(torch.linalg.norm(a - ref) / max(float(torch.linalg.norm(ref)), 1e-30))


def _check(t):
  ref = _reference(t)
  old, n_old = _old_path(t)
  new, n_new = _new_path(t)
  errs = {k: (_rel(new[k], ref[k]), _rel(old[k], ref[k])) for k in ref}
  print('launches %d -> %d; rel err (new, old): %s' % (n_old, n_new, errs))
  for k, (e_new, e_old) in errs.items():
    assert np.isfinite(e_new) and e_new <= 1.25 * e_old + 1e-6, (k, e_new, e_old)
  assert n_new <= n_old
  return new, ref


@pytest.mark.parametrize('n,hw,c,cout,dpass', [
    (2, (118, 118), 256, 64, True),     # layer 1: 4C -> C reduction of an identity block (BN1, pass-through)
    (2, (118, 118), 64, 256, False),    # layer 1: C -> 4C expansion (BN3)
    (4, (59, 59), 512, 128, True),      # layer 2
    (4, (59, 59), 128, 512, False),
    (8, (30, 30), 1024, 256, True),     # layer 3 reduction: 256-multiple data-gradient width with K = 256
    (8, (30, 30), 1024, 256, False),
    (3, (7, 13), 256, 64, True),        # ragged maps: tiles hang over the image edge
    (2, (15, 15), 64, 256, False),
    (2, (15, 15), 128, 512, True),
])
def test_bn_bwd_gemm_matches_two_pass(n, hw, c, cout, dpass):
  _check(_node(n, hw[0], hw[1], c, cout, dpass, seed=n + c))


@pytest.mark.parametrize('gamma_mode', ['negative', 'zero', 'masked'])
def test_bn_bwd_gemm_adversarial_parameters(gamma_mode):
  new, ref = _check(_node(2, 15, 15, 256, 64, True, gamma_mode, seed=3))
  if gamma_mode == 'masked':
    assert float(new['dw'][:, :3].abs().max()) == 0.0
    assert float(new['dbeta'][:3].abs().max()) == 0.0 and float(new['dgamma'][:3].abs().max()) == 0.0


def test_bn_bwd_gemm_rejects_unsupported_geometry():
  from tensor2robot_b200 import _lib
  t = _node(1, 8, 8, 2048, 512, False)
  d = _desc(1, 8, 8, 2048, 512)           # data gradient 512 -> 2048 runs on the register-epilogue kernel
  assert _lib.lib().t2r_conv2d_dgrad_bnapply_supported(C.byref(d)) == 0
  coef = torch.zeros(2 * 2048, dtype=F32, device='cuda')
  dx = torch.empty_like(t['x'])
  with pytest.raises(_lib.T2RError):
    _lib.call('t2r_conv2d_dgrad_bnapply', C.byref(d), _p(t['dy']), _p(t['wd']), _p(t['x']), _p(t['scale']),
              _p(t['shift']), _p(coef), None, _p(dx), None)


def _block_step(filters, hw, gemm, b=4):
  """One identity bottleneck block (layers/film_resnet_model.py:283-340) through nn, forward + backward."""
  from tensor2robot_b200 import _lib, nn
  from tensor2robot_b200.layers import film_resnet_model as rm
  old = nn.BN_BWD_GEMM
  nn.BN_BWD_GEMM = gemm
  try:
    rng = np.random.RandomState(7)
    c = 4 * filters
    x0 = torch.from_numpy(rng.standard_normal((b, hw, hw, c)).astype(np.float32)).cuda().to(BF16)
    vs = nn.VariableStore('cuda', seed=5)

    def call(x, training):
      return rm._bottleneck_block_v2(x, filters, training, None, 1, rm._Namer(), 1e-4)

    with torch.no_grad(), nn.variable_store(vs):
      call(x0, False)
    vs.finalize()
    x = x0.clone().requires_grad_(True)
    launches0 = _lib.launch_count()
    with nn.variable_store(vs):
      y = call(x, True)
      wts = torch.from_numpy(rng.standard_normal(tuple(y.shape)).astype(np.float32)).cuda()
      loss = (y.float() * wts).sum()
      vs.zero_grad()
      loss.backward()
    torch.cuda.synchronize()
    return dict(dx=x.grad.float().cpu().numpy(), grad=vs.flat_grad.cpu().numpy(), state=vs.state_flat.cpu().numpy(),
                launches=_lib.launch_count() - launches0)
  finally:
    nn.BN_BWD_GEMM = old


@pytest.mark.parametrize('filters,hw', [(64, 30), (128, 17), (256, 15)])
def test_block_backward_gemm_matches_two_pass(filters, hw):
  ref = _block_step(filters, hw, False)
  got = _block_step(filters, hw, True)

  def rel(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b.astype(np.float64)), 1e-30))

  errs = dict(dx=rel(got['dx'], ref['dx']), grad=rel(got['grad'], ref['grad']), state=rel(got['state'], ref['state']))
  print('filters=%d: launches %d -> %d, %s' % (filters, ref['launches'], got['launches'], errs))
  assert errs['dx'] < 5e-3 and errs['grad'] < 5e-3 and errs['state'] < 1e-5
  assert got['launches'] < ref['launches']


def test_native_harness_bn_bwd_gemm():
  """tests/native/test_bn_bwd_gemm.cu: the three entry points against CPU loops in double, no Python in the process."""
  binary = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'native', 'test_bn_bwd_gemm')
  if not os.path.exists(binary):
    pytest.fail('tests/native/test_bn_bwd_gemm is not built: run __graft_entry__.build()')
  out = subprocess.run([binary], cwd=os.path.dirname(binary), stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, timeout=600)
  print(out.stdout)
  failures = [l for l in out.stdout.splitlines() if l.startswith(('[FAIL]', '[FATAL]'))]
  assert out.returncode == 0 and not failures, '\n'.join(failures[:20] + out.stdout.splitlines()[-3:])
  assert 'SUMMARY' in out.stdout and 'fail=0' in out.stdout and out.stdout.count('[PASS]') == 20
