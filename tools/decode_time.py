"""Time ct_decode alone at the benchmark's shape (32 x 80 x 128 x 128), on i.i.d. and on smooth heat-maps, with the
phase knobs of CTB_DEC_DEBUG (1: streaming NMS only, 2: no per-image merge):   python tools/decode_time.py"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from centertrack_b200.decode import generic_decode          # noqa


class Opt:
  pass


B, C, H, W, K = 32, 80, 128, 128, 100
g = torch.Generator().manual_seed(0)
for kind in ('iid', 'smooth'):
  z = torch.randn(B, C, H, W, generator=g)
  if kind == 'smooth':                                      # band-limited maps like a network's: ~10x fewer local maxima
    z = torch.nn.functional.avg_pool2d(z, 5, 1, 2) * 4
  out = {'hm': torch.sigmoid(2 * z - 4.6).cuda(), 'reg': torch.rand(B, 2, H, W, generator=g).cuda(),
         'wh': (torch.randn(B, 2, H, W, generator=g) * 6).cuda(), 'tracking': torch.randn(B, 2, H, W, generator=g).cuda()}
  # One decode per CUDA-graph replay (no host time between the events), a cache flush between replays
  from centertrack_b200 import _lib as L
  ws = torch.zeros(L.lib().ct_decode_workspace_bytes(B, C, 0, K), dtype=torch.uint8, device='cuda')
  rec = generic_decode(out, K, Opt(), workspace=ws).records
  torch.cuda.synchronize()
  st = torch.cuda.Stream()
  with torch.cuda.stream(st):
    generic_decode(out, K, Opt(), records_out=rec, workspace=ws)
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr, stream=st):
      generic_decode(out, K, Opt(), records_out=rec, workspace=ws)
  torch.cuda.synchronize()
  flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
  ts = []
  for _ in range(12):
    flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    gr.replay()
    e1.record()
    torch.cuda.synchronize()
    ts.append(e0.elapsed_time(e1) * 1000)
  ts.sort()
  print('%s maps, CTB_DEC_DEBUG=%s: median %.1f us, min %.1f us' % (
      kind, os.environ.get('CTB_DEC_DEBUG', '0'), ts[len(ts) // 2], ts[0]))
