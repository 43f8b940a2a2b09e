"""Times the backward of one batch-norm + ReLU + 1x1-convolution node of ResNet-50 at batch 512, old path against the
GEMM path, alternating, with CUDA events:

  old : t2r_conv2d_wgrad on z, t2r_conv2d_dgrad into g, t2r_bn_backward (reduction pass + apply pass)
  new : t2r_conv2d_wgrad_bnsums (dw and the two batch-norm sums), t2r_bn_backward_gemm_finalize,
        t2r_conv2d_dgrad_bnapply (dx in the epilogue)

and the two new kernels alone, as algorithmic bytes over time against the 7.7 TB/s HBM figure of the B200 data sheet.
Inputs are several GB per tensor, far beyond the 126 MB L2.

  python scripts/bn_bwd_gemm_ab.py [REPS]"""
import ctypes as C
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tensor2robot_b200 import _lib, nn   # noqa: E402

PEAK = 7.7e12
# (name, image size, normalised channels c, consumer output channels, pass-through gradient)
SHAPES = [
    ('layer1 BN1 256->64', 118, 256, 64, True),
    ('layer1 BN3 64->256', 118, 64, 256, False),
    ('layer2 BN1 512->128', 59, 512, 128, True),
    ('layer2 BN3 128->512', 59, 128, 512, False),
    ('layer3 BN1 1024->256', 30, 1024, 256, True),
]


def p(t):
  return C.c_void_p(t.data_ptr()) if t is not None else None


def timed(fn, reps):
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(reps):
    fn()
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / reps


def main():
  reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
  smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip()
  print('device: %s' % smi)
  n = 512
  dev = torch.device('cuda')
  st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
  for name, hw, c, cout, has_dpass in SHAPES:
    rows = n * hw * hw
    x = (torch.randn(n, hw, hw, c, device=dev) * 0.7).to(torch.bfloat16)
    dy = torch.randn(n, hw, hw, cout, device=dev).to(torch.bfloat16)
    dpass = torch.randn(n, hw, hw, c, device=dev).to(torch.bfloat16) if has_dpass else None
    w = (torch.randn(cout, 1, 1, c, device=dev) / c ** 0.5).float()
    wd = torch.empty(c * cout, dtype=torch.bfloat16, device=dev)
    _lib.call('t2r_pack_weights', p(w), None, p(wd), cout, 1, c, st)
    mean = torch.randn(c, device=dev) * 0.1
    invstd = torch.rand(c, device=dev) + 0.5
    scale = invstd * (torch.rand(c, device=dev) + 0.5)
    shift = torch.randn(c, device=dev) * 0.3
    d = nn._conv_desc(n, hw, hw, c, cout, 1, 1, 1, 0, 0, hw, hw, 0)
    z = torch.empty_like(x)
    _lib.call('t2r_bn_apply', p(x), p(z), rows, c, p(scale), p(shift), None, hw * hw, 1, st)
    g = torch.empty_like(x)
    dx = torch.empty_like(x)
    dw = torch.zeros(cout, c, device=dev)
    red = torch.zeros(2 * c, dtype=torch.float64, device=dev)
    sums = torch.zeros(2 * c, dtype=torch.float64, device=dev)
    coef = torch.empty(2 * c, device=dev)
    dgamma = torch.empty(c, device=dev)
    dbeta = torch.empty(c, device=dev)

    def old():
      _lib.call('t2r_conv2d_wgrad', C.byref(d), p(z), p(dy), p(dw), st)
      _lib.call('t2r_conv2d_dgrad', C.byref(d), p(dy), p(wd), p(g), 0, st)
      _lib.call('t2r_bn_backward', p(g), p(x), p(dpass), p(dx), rows, c, None, p(mean), p(invstd), p(scale), p(shift),
                1, p(red), p(dgamma), p(dbeta), st)

    def wgrad_new():
      sums.zero_()
      _lib.call('t2r_conv2d_wgrad_bnsums', C.byref(d), p(x), p(scale), p(shift), p(dy), p(wd), p(dw), p(sums), st)

    def dgrad_new():
      _lib.call('t2r_conv2d_dgrad_bnapply', C.byref(d), p(dy), p(wd), p(x), p(scale), p(shift), p(coef), p(dpass),
                p(dx), st)

    def new():
      wgrad_new()
      _lib.call('t2r_bn_backward_gemm_finalize', p(sums), rows, c, p(mean), p(invstd), p(scale), p(dgamma), p(dbeta),
                p(coef), st)
      dgrad_new()

    for fn in (old, new):
      fn()
    torch.cuda.synchronize()
    t_old, t_new = [], []
    for _ in range(reps):
      t_old.append(timed(old, 3))
      t_new.append(timed(new, 3))
    t_wg = statistics.median(timed(wgrad_new, 3) for _ in range(reps))
    t_dg = statistics.median(timed(dgrad_new, 3) for _ in range(reps))
    t_wg_plain = statistics.median(timed(lambda: _lib.call('t2r_conv2d_wgrad', C.byref(d), p(z), p(dy), p(dw), st), 3)
                                   for _ in range(reps))
    t_dg_plain = statistics.median(timed(lambda: _lib.call('t2r_conv2d_dgrad', C.byref(d), p(dy), p(wd), p(g), 0, st),
                                         3) for _ in range(reps))
    s_x, s_y = x.numel() * 2, dy.numel() * 2
    wg_bytes = s_x + s_y                                        # reads x, dy
    dg_bytes = s_y + s_x * (3 if has_dpass else 2)              # reads dy, x (, dpass); writes dx
    print('%-22s node old %7.3f ms  new %7.3f ms  (medians of %d; old %s new %s)' % (
        name, statistics.median(t_old), statistics.median(t_new), reps,
        ' '.join('%.3f' % v for v in t_old), ' '.join('%.3f' % v for v in t_new)))
    print('%-22s   wgrad_bnsums %6.3f ms %5.2f TB/s = %.2f of 7.7 | plain wgrad on z %6.3f ms' % (
        '', t_wg, wg_bytes / t_wg / 1e9, wg_bytes / t_wg / 1e9 / 7.7, t_wg_plain))
    print('%-22s   dgrad_bnapply %6.3f ms %5.2f TB/s = %.2f of 7.7 | plain dgrad %6.3f ms' % (
        '', t_dg, dg_bytes / t_dg / 1e9, dg_bytes / t_dg / 1e9 / 7.7, t_dg_plain))
    del x, dy, dpass, z, g, dx
    torch.cuda.empty_cache()


if __name__ == '__main__':
  main()
