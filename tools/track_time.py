"""Time ct_track_step alone at B = 32 streams, K = 100 detections, on crowded synthetic records: greedy, --hungarian and
--public_det --hungarian association, each with --max_age -1 and 2.  Three frames are stepped first so the track
tables hold matched, new and (max_age 2) coasting tracks; the fourth frame is then timed with CUDA events around
replays of a CUDA graph holding that one launch, the track state restored before every replay (outside the events).
    python tools/track_time.py --out profiles/track_time.json"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from centertrack_b200 import _lib as L                       # noqa: E402
from centertrack_b200.device_tracker import DeviceTracker     # noqa: E402
from helpers import make_opt                                  # noqa: E402

B, K, F, INP = 32, 100, 13, 512
LAYOUT = {'wh': (9, 2), 'tracking': (11, 2)}
MODES = [('greedy', []), ('hungarian', ['--hungarian']), ('public_hungarian', ['--public_det', '--hungarian'])]


def frames(n_frames, rng):
  """Records [B,K,F] per frame on the 128 x 128 output grid: 100 objects per stream moving a little each frame, 85 %
  of them seen per frame, the tracking head pointing back to the previous position; plus the public detections
  (output-grid predicted centres, jittered, of 70 % of the seen objects)."""
  out_w = INP // 4
  pos = rng.uniform(4, out_w - 4, (B, K, 2))
  wh = rng.uniform(2, 12, (B, K, 2))
  cls = rng.randint(0, 2, (B, K))
  seq = []
  for _ in range(n_frames):
    move = rng.normal(0, 0.6, (B, K, 2))
    pos = pos + move
    rec = np.zeros((B, K, F), np.float32)
    pubs = []
    for b in range(B):
      seen = np.nonzero(rng.uniform(size=K) < 0.85)[0]
      n = len(seen)
      rec[b, :n, 0] = np.sort(rng.uniform(0.35, 1.0, n))[::-1]
      rec[b, n:, 0] = np.sort(rng.uniform(0.0, 0.2, K - n))[::-1]
      order = np.concatenate([seen, np.setdiff1d(np.arange(K), seen)])
      p, s = pos[b, order], wh[b, order]
      rec[b, :, 1] = cls[b, order]
      rec[b, :, 2:4] = np.floor(p)
      rec[b, :, 4:6] = p - s / 2
      rec[b, :, 6:8] = p + s / 2
      rec[b, :, 9:11] = s
      rec[b, :, 11:13] = -move[b, order] + rng.normal(0, 0.3, (K, 2))
      pubs.append([(p[i] + rec[b, i, 11:13] + rng.normal(0, 0.3, 2)) for i in range(n) if rng.uniform() < 0.7])
    seq.append((torch.from_numpy(rec).cuda(), pubs))
  return seq


def time_mode(extra, max_age, seq, replays, warmup):
  opt = make_opt('coco_tracking', ['--max_age', str(max_age)] + extra)
  trk = DeviceTracker(opt, B, K, F, LAYOUT, INP, INP, 'cuda')
  t_out = trk.trans_out_inv.cpu().numpy().reshape(B, 2, 3).astype(np.float64)

  def set_public(pubs):                                   # output grid -> image coordinates
    trk.set_public(None, [[{'ct': t_out[b] @ np.array([q[0], q[1], 1.0])} for q in pubs[b]] for b in range(B)])

  for rec, pubs in seq[:-1]:
    if trk.public_det:
      set_public(pubs)
    trk.step(rec)
  rec, pubs = seq[-1]
  if trk.public_det:
    set_public(pubs)
  torch.cuda.synchronize()
  saved = (trk.tracks.clone(), trk.counts.clone(), trk.boxes.clone())
  n_tracks_before = saved[1][:, 0].float().mean().item()
  st = torch.cuda.Stream()
  with torch.cuda.stream(st):
    trk.step(rec)                                         # sets the smem attribute outside the capture
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
      trk.step(rec)
  torch.cuda.synchronize()
  ts = []
  for it in range(warmup + replays):
    trk.tracks.copy_(saved[0]); trk.counts.copy_(saved[1]); trk.boxes.copy_(saved[2])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    if it >= warmup:
      ts.append(e0.elapsed_time(e1) * 1000)
  ts = np.sort(np.array(ts))
  return {'median_us': round(float(np.median(ts)), 1), 'min_us': round(float(ts[0]), 1),
          'p90_us': round(float(ts[int(0.9 * (len(ts) - 1))]), 1),
          'tracks_before_mean': round(n_tracks_before, 1),
          'detections_mean': round(float((rec[:, :, 0] > opt.out_thresh).sum(1).float().mean().item()), 1),
          'tracks_after_mean': round(trk.counts[:, 0].float().mean().item(), 1)}


def gpu_facts():
  facts = {'gpu': torch.cuda.get_device_name(0)}
  try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    facts['power_limit'], facts['max_sm_clock'] = [x.strip() for x in q.split(',')]
  except Exception as e:  # noqa: BLE001 -- the numbers stand without it, but say why it is missing
    facts['power_limit'] = 'unavailable (%s)' % type(e).__name__
  return facts


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--out', default=None, help='JSON file to write (default: print only)')
  ap.add_argument('--replays', type=int, default=300)
  ap.add_argument('--warmup', type=int, default=30)
  args = ap.parse_args()
  seq = frames(4, np.random.RandomState(0))
  res = dict(gpu_facts(), B=B, K=K, replays=args.replays, warmup=args.warmup,
             what='one ct_track_step launch per CUDA-graph replay, CUDA events, track state restored between replays',
             modes={})
  for name, extra in MODES:
    for max_age in (-1, 2):
      key = '%s_age%d' % (name, max_age)
      res['modes'][key] = time_mode(extra, max_age, seq, args.replays, args.warmup)
      print(key, res['modes'][key], flush=True)
  if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
      json.dump(res, f, indent=1)
  print(json.dumps(res))


if __name__ == '__main__':
  main()
