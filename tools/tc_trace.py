"""Timeline of the middle CTA of the gather engine (conv_tc_kernel) for DCN / plain-conv layer shapes at B=16:
   python tools/tc_trace.py      (cycles; see tc_stamp in csrc/conv_tc.cu for the stamp ids)"""
import ctypes as C
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from centertrack_b200 import _lib as L       # noqa
from gpu_helpers import run_conv             # noqa

lib = L.lib()
# (name, B, Cin, Cout, H, W, k, stride, dcn, n_tile); dcn: True = global gather (CT_A_DCN), 'win' = shared-memory window
cases = [('DCN 64->64 128x128 B32 global', 32, 64, 64, 128, 128, 3, 1, True, 64),
         ('DCN 64->64 128x128 B32 window', 32, 64, 64, 128, 128, 3, 1, 'win', 64),
         ('DCN 128->128 64x64 B32 window', 32, 128, 128, 64, 64, 3, 1, 'win', 128),
         ('DCN 64->64 128x128', 16, 64, 64, 128, 128, 3, 1, True, 64),
         ('DCN 128->64 64x64', 16, 128, 64, 64, 64, 3, 1, True, 64),
         ('DCN 512->256 16x16 nt32', 16, 512, 256, 16, 16, 3, 1, True, 32),
         ('conv 256->256 32x32 nt128 (level4)', 16, 256, 256, 32, 32, 3, 1, False, 128),
         ('conv 512->512 16x16 nt64 (level5)', 16, 512, 512, 16, 16, 3, 1, False, 64),
         ('conv s2 16->32 512x512 (level1)', 16, 16, 32, 512, 512, 3, 2, False, 32)]
g = torch.Generator().manual_seed(0)
for (name, B, Cin, Cout, H, W, k, stride, dcn, nt) in cases:
  if os.environ.get('CTB_TRACE_ONLY') and os.environ['CTB_TRACE_ONLY'] not in name:
    continue
  x = torch.randn(B, Cin, H, W, generator=g).cuda()
  w = torch.randn(Cout, Cin, k, k, generator=g) * 0.05
  b = torch.zeros(Cout)
  kw = dict(n_tile=nt)
  if dcn:
    wo = torch.randn(27, Cin, 3, 3, generator=g) * (0.6 / (Cin * 9) ** 0.5)
    bo = torch.randn(27, generator=g) * (0.7 if B == 32 else 1.5)      # B=32 cases: the benchmark network's offset scale
    # experiments on what the sampler's time depends on: scale the spread / the per-tap bias of the offsets
    wo[:18] *= float(os.environ.get('CTB_TRACE_OFF_SPREAD', '1'))
    bo[:18] *= float(os.environ.get('CTB_TRACE_OFF_BIAS', '1'))
    if 'CTB_TRACE_OFF_CONST' in os.environ:
      bo[:18] = float(os.environ['CTB_TRACE_OFF_CONST'])
    om = run_conv(L.CT_ENGINE_TCGEN05, L.CT_BF16, x, wo, bo, 1, relu=False, out_mode=L.CT_OUT_NHWC_F32, sig_from=18, n_tile=32)
    kw.update(a_mode=L.CT_A_DCN_WIN if dcn == 'win' else L.CT_A_DCN, om=om.permute(0, 2, 3, 1).contiguous())
  tr = torch.zeros(256, dtype=torch.int64, device='cuda')
  run_conv(L.CT_ENGINE_TCGEN05, L.CT_BF16, x, w, b, stride, True, **kw)      # warm
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ev0.record()
  for _ in range(5):
    run_conv(L.CT_ENGINE_TCGEN05, L.CT_BF16, x, w, b, stride, True, **kw)
  ev1.record()
  torch.cuda.synchronize()
  print('==== %s: %.1f us per call incl. host overhead of run_conv' % (name, ev0.elapsed_time(ev1) * 200))
  L.check(lib.ct_debug_trace(C.c_void_p(tr.data_ptr())))
  torch.cuda.synchronize()
  run_conv(L.CT_ENGINE_TCGEN05, L.CT_BF16, x, w, b, stride, True, **kw)
  torch.cuda.synchronize()
  L.check(lib.ct_debug_trace(None))
  t = tr.cpu().numpy().astype(np.int64)
  if dcn == 'win':                                       # the persistent window kernel
    q = t[16:16 + 240].reshape(60, 4)
    n = int((q[:, 3] > 0).sum())
    base = q[0, 0]
    print('  persistent CTA, per slice (cycles since the first): stage acquired | A written | MMA saw full | MMA committed   [period]')
    for i in range(min(n, 30)):
      print('   %2d  %7d %7d %7d %7d   [%d]  A %d  full-after-A %d' % (i, q[i, 0] - base, q[i, 1] - base, q[i, 2] - base, q[i, 3] - base,
                                                                   (q[i, 1] - q[i - 1, 1]) if i else 0, q[i, 1] - q[i, 0], q[i, 2] - q[i, 1]))
    continue
  t0 = t[0]
  sl = t[8:]
  n = int((sl > 0).sum())
  d = np.diff(np.concatenate([[t[2] if t[2] > 0 else t[1]], sl[:n]]))
  print('==== %s : k_slices %d' % (name, n))
  print('  after alloc+sync %d' % (t[7] - t0))
  print('  rows set up %d | table built %d | first slice done %d | last slice done %d | mma committed %d | epilogue start %d | end %d'
        % (t[1] - t0, (t[2] - t0) if t[2] > 0 else -1, sl[0] - t0, sl[n - 1] - t0, t[4] - t0, t[5] - t0, t[6] - t0))
  print('  cycles per slice: first %d, mean %.0f, min %d, max %d' % (d[0], d.mean(), d.min(), d.max()))
