"""-m gpu: --hungarian and the MOT --public_det protocol in ct_track_step (DeviceTracker / StreamRunner with
device_tracking) against the reference's Tracker golden (tests/golden/track_modes.npz) and against the host Tracker
that golden pins."""
import copy

import numpy as np
import pytest
import torch

from centertrack_b200 import _lib as L
from centertrack_b200 import synthetic as wt
from helpers import make_model, make_opt

pytestmark = pytest.mark.gpu
DEV = torch.device('cuda')

TRACK_MODES = [('greedy_age2', ['--max_age', '2']), ('hungarian', ['--hungarian']),
               ('hungarian_age2', ['--hungarian', '--max_age', '2']), ('public', ['--public_det']),
               ('public_hungarian_age2', ['--public_det', '--hungarian', '--max_age', '2'])]
F = 13
LAYOUT = {'wh': (9, 2), 'tracking': (11, 2)}


def _rows(out):
  return np.array([[o['tracking_id'], o['age'], o['active'], o['class'], o['score']] + list(map(float, o['bbox']))
                   for o in out], np.float64).reshape(-1, 9)


def _identity_tracker(opt, B, K):
  """A DeviceTracker whose output-grid -> image map is the identity (records carry image coordinates) and that
  hands every detection to the tracker (out_thresh 0), as the host Tracker sees the synthetic streams."""
  from centertrack_b200.device_tracker import DeviceTracker
  trk = DeviceTracker(opt, B, K, F, LAYOUT, 320, 320, DEV)
  trk.trans_out_inv.copy_(torch.tensor([1, 0, 0, 0, 1, 0], dtype=torch.float32).expand(B, 6))
  trk.desc.out_thresh = 0.0
  return trk


def _identity_records(dets_per_stream, K):
  rec = np.zeros((len(dets_per_stream), K, F), np.float32)
  for b, dets in enumerate(dets_per_stream):
    assert len(dets) <= K
    for i, d in enumerate(dets):
      ct, trk = np.asarray(d['ct'], np.float32), np.asarray(d['tracking'], np.float32)
      # the kernel forms the predicted centre as ((ct + tracking) - ct) + ct: equal to ct + tracking for this data
      assert np.array_equal((((ct + trk) - ct) + ct).astype(np.float32), (ct + trk).astype(np.float32))
      rec[b, i, 0], rec[b, i, 1] = d['score'], d['class'] - 1
      rec[b, i, 2:4] = ct
      rec[b, i, 4:8] = d['bbox']
      rec[b, i, 11:13] = trk
  return torch.from_numpy(rec).to(DEV)


def _run_streams(extra, seeds, K, stream_kw):
  """Seeded synthetic streams side by side in one DeviceTracker; yields (frame, device results, per-stream inputs)."""
  opt = make_opt('coco_tracking', ['--track_thresh', '0.2', '--new_thresh', '0.3'] + extra)
  streams = [wt.synthetic_track_stream(s, **stream_kw) for s in seeds]
  trk = _identity_tracker(opt, len(seeds), K)
  for f in range(len(streams[0])):
    dets = [s[f][0] for s in streams]
    pubs = [s[f][1] for s in streams]
    if opt.public_det:
      trk.set_public(None, pubs)
    trk.step(_identity_records(dets, K))
    torch.cuda.synchronize()
    got = trk.results(trk.tracks.cpu().numpy(), trk.counts.cpu().numpy())
    yield opt, f, got, trk.counts.cpu().numpy(), dets, pubs


@pytest.mark.parametrize('mode', range(len(TRACK_MODES)), ids=[m[0] for m in TRACK_MODES])
def test_device_modes_match_reference_golden(mode, golden_dir):
  """Seeds 0-3 as four streams of one tracker (K = 64): every row (id, age, active, class, score, bbox) and the
  id_count equal what the reference's Tracker produced."""
  import os
  g = np.load(os.path.join(golden_dir, 'track_modes.npz'))
  name, extra = TRACK_MODES[mode]
  born = 0
  for opt, f, got, counts, _, _ in _run_streams(extra, range(4), 64, {}):
    for s in range(4):
      key = '%s.s%d.f%d' % (name, s, f)
      assert [len(got[s]), int(counts[s, 1])] == list(g[key + '.n']), key
      assert np.array_equal(_rows(got[s]), g[key]), key
    born = int(counts[:, 1].sum())
  assert born > 0


@pytest.mark.parametrize('extra', [['--hungarian'], ['--public_det'], ['--public_det', '--hungarian', '--max_age', '3'],
                                   ['--hungarian', '--max_age', '1']], ids=lambda e: '_'.join(x.strip('-') for x in e))
def test_device_modes_equal_host_tracker_on_many_streams(extra):
  """Seeds 10-33, 24 crowded streams in one tracker, against the host Tracker stream by stream: rows exact."""
  from centertrack_b200.tracker import Tracker
  seeds = list(range(10, 34))
  hosts = None
  for opt, f, got, counts, dets, pubs in _run_streams(extra, seeds, 96, {'frames': 5, 'crowd': 40}):
    if hosts is None:
      hosts = [Tracker(opt) for _ in seeds]
      for h in hosts:
        h.init_track([])
    for b, h in enumerate(hosts):
      want = h.step(copy.deepcopy(dets[b]), pubs[b])
      assert np.array_equal(_rows(got[b]), _rows(want)), (extra, seeds[b], f)
      assert int(counts[b, 1]) == h.id_count


def _check_tracks(got, want, ctx):
  assert len(got) == len(want), (ctx, len(got), len(want))
  for a, b in zip(got, want):
    assert (a['tracking_id'], a['age'], a['active'], a['class']) == \
        (int(b['tracking_id']), int(b['age']), int(b['active']), int(b['class'])), (ctx, a, b)
    # a track seeded by Tracker.init_track has no 'tracking' until it is matched; the device row holds zeros there
    assert 'tracking' in b or np.array_equal(a['tracking'], np.zeros(2, np.float32)), ctx
    for k in [k for k in ('ct', 'tracking', 'bbox') if k in b]:
      assert np.allclose(np.asarray(a[k], np.float64), np.asarray(b[k], np.float64), rtol=1e-4, atol=1e-3), (ctx, k)
    assert abs(a['score'] - float(b['score'])) < 1e-6


@pytest.mark.parametrize('extra', [['--hungarian', '--max_age', '2'], ['--public_det'],
                                   ['--public_det', '--hungarian', '--max_age', '2']],
                         ids=lambda e: '_'.join(x.strip('-') for x in e))
@pytest.mark.parametrize('seed', range(3))
def test_device_modes_equal_host_pipeline_on_random_records(extra, seed):
  """Random decode records under non-identity affines (B = 3 streams), device tracker vs views -> generic_post_process
  -> host Tracker.  The streams cover N > M and N < M, a scene cut (every pair blocked, so the solver forces and
  rejects them), empty frames, frames without public detections and frames with more public detections than
  detections."""
  from centertrack_b200.decode import views_from_records
  from centertrack_b200.device_tracker import DeviceTracker
  from centertrack_b200.post_process import generic_post_process
  from centertrack_b200.tracker import Tracker
  rng = np.random.RandomState(100 + seed)
  B, K = 3, 64
  inp_h, inp_w = 256, 320
  out_h, out_w = inp_h // 4, inp_w // 4
  opt = make_opt('coco_tracking', ['--track_thresh', '0.2', '--new_thresh', '0.3', '--pre_thresh', '0.25',
                                   '--input_h', str(inp_h), '--input_w', str(inp_w)] + extra)
  img_hw = [(240, 320), (300, 260), (256, 320)]
  centers = [np.array([w / 2., h / 2.], np.float32) for h, w in img_hw]
  scales = [max(h, w) * 1.0 for h, w in img_hw]
  dev_trk = DeviceTracker(opt, B, K, F, LAYOUT, inp_h, inp_w, DEV, centers=centers, scales=scales, max_public=2 * K)
  hosts = [Tracker(opt) for _ in range(B)]
  for t in hosts:
    t.init_track([])
  sizes = [[5, 30, 0, 40, 12, 50], [40, 8, 25, 25, 0, 3], [20, 20, 20, 20, 20, 20]]
  for frame in range(6):
    rec = np.zeros((B, K, F), np.float32)
    for b in range(B):
      n = sizes[b][frame]
      sc = np.sort(rng.uniform(0.21, 1.0, n).astype(np.float32))[::-1]
      rec[b, :n, 0] = sc
      rec[b, n:, 0] = np.sort(rng.uniform(0.0, 0.19, K - n).astype(np.float32))[::-1]
      rec[b, :, 1] = rng.randint(0, 2, K)
      rec[b, :, 2] = rng.randint(0, out_w // 2, K)           # crowded: half the grid
      rec[b, :, 3] = rng.randint(0, out_h // 2, K)
      wh = rng.uniform(2, 24, (K, 2))
      cx, cy = rec[b, :, 2] + rng.rand(K), rec[b, :, 3] + rng.rand(K)
      rec[b, :, 4], rec[b, :, 5], rec[b, :, 6], rec[b, :, 7] = cx - wh[:, 0] / 2, cy - wh[:, 1] / 2, cx + wh[:, 0] / 2, cy + wh[:, 1] / 2
      rec[b, :, 9:11] = wh
      rec[b, :, 11:13] = rng.normal(0, 1.5, (K, 2))
      if b == 2 and frame == 3:                             # scene cut: a class no track has
        rec[b, :, 1] = 2
    views = {k: v.numpy() for k, v in views_from_records(torch.from_numpy(rec), LAYOUT).items()}
    results, pubs = [], []
    for b in range(B):
      one = {k: v[b:b + 1] for k, v in views.items()}
      res = generic_post_process(opt, one, [centers[b]], [scales[b]], out_h, out_w, opt.num_classes)[0]
      res = [r for r in res if r['score'] > opt.out_thresh]
      results.append(res)
      if b == 1 and frame in (1, 4):
        pub = []                                            # no public detections at all
      elif b == 0 and frame in (0, 2):                      # more public detections than detections
        pub = [{'ct': (np.asarray(r['ct']) + np.asarray(r['tracking'])).astype(np.float32)} for r in res] + \
              [{'ct': rng.uniform(0, 300, 2).astype(np.float32)} for _ in range(len(res) + 3)]
      else:
        pub = [{'ct': (np.asarray(r['ct']) + np.asarray(r['tracking']) + rng.normal(0, 3, 2)).astype(np.float32)}
               for r in res if rng.uniform() < 0.7]
      pubs.append(pub)
    if opt.public_det:
      dev_trk.set_public(None, pubs)
    dev_trk.step(torch.from_numpy(rec).to(DEV))
    torch.cuda.synchronize()
    got = dev_trk.results(dev_trk.tracks.cpu().numpy(), dev_trk.counts.cpu().numpy())
    for b in range(B):
      want = hosts[b].step(copy.deepcopy(results[b]), pubs[b])
      _check_tracks(got[b], want, (extra, seed, frame, b))
      assert int(dev_trk.counts[b, 1]) == hosts[b].id_count


def test_stream_runner_public_hungarian_closes_the_loop_like_the_host_pipeline():
  """StreamRunner(device_tracking=True) with --public_det --hungarian --max_age 2 (fp32 engine, B = 2, 5 frames):
  seeded from pre_dets at t = 0, public detections uploaded with each frame through step_host, graphs replayed --
  equal to the host loop (Tracker.init_track(pre_dets), _get_additional_inputs, network, decode, post-process,
  Tracker.step(results, public)) frame by frame."""
  from centertrack_b200.decode import generic_decode
  from centertrack_b200.image import get_affine_transform
  from centertrack_b200.post_process import generic_post_process
  from centertrack_b200.runner import StreamRunner
  from centertrack_b200.tracker import Tracker
  from test_gpu_stream import _host_detector
  B, H, W, K = 2, 64, 96, 30
  opt, model, sd = make_model('coco_tracking', extra=['--track_thresh', '0.1', '--new_thresh', '0.1', '--pre_thresh', '0.1',
                                                       '--input_h', str(H), '--input_w', str(W), '--max_age', '2',
                                                       '--public_det', '--hungarian'])
  model = model.cuda()
  runner = StreamRunner(model, B, H, W, K=K, precision='fp32', device='cuda', opt=opt, device_tracking=True)
  runner.warm()
  rng = np.random.RandomState(5)
  pre_dets = []
  for b in range(B):
    one = []
    for _ in range(6):
      x, y, w, h = rng.uniform(0, 80), rng.uniform(0, 50), rng.uniform(4, 20), rng.uniform(4, 20)
      one.append({'score': float(rng.uniform(0.05, 1)), 'class': int(rng.randint(1, 3)),
                  'bbox': np.array([x, y, x + w, y + h], np.float32)})
    pre_dets.append(one)
  runner.reset_tracking(pre_dets)
  eng = model.engine_for(B, H, W, DEV, 'fp32')
  det = _host_detector(opt)
  hosts = [Tracker(opt) for _ in range(B)]
  for b, t in enumerate(hosts):
    t.init_track(copy.deepcopy(pre_dets[b]))
  assert sum(len(t.tracks) for t in hosts) > 0
  c = np.array([W / 2., H / 2.], np.float32)
  s = max(H, W) * 1.0
  meta = {'inp_width': W, 'inp_height': H, 'out_width': W // 4, 'out_height': H // 4,
          'trans_input': get_affine_transform(c, s, 0, [W, H]), 'trans_output': get_affine_transform(c, s, 0, [W // 4, H // 4])}
  opt.device = torch.device('cpu')
  frames = [wt.synthetic_inputs(B, H, W, seed=60 + t)[0] for t in range(5)]
  pre = None
  born = 0
  for t, img in enumerate(frames):
    # host loop first: its detections decide this frame's public detections
    hms = [det._get_additional_inputs(hosts[b].tracks, meta, with_hm=True)[0] for b in range(B)]
    hm = torch.cat(hms, 0).cuda()
    x = img.cuda()
    out = dict(eng.forward(x, x if pre is None else pre, hm))
    res = generic_decode(out, K=K)
    views = {k: v.cpu().numpy() for k, v in res.items()}
    results, pubs = [], []
    for b in range(B):
      one = {k: v[b:b + 1] for k, v in views.items()}
      r = [q for q in generic_post_process(opt, one, [c], [s], H // 4, W // 4, opt.num_classes)[0]
           if q['score'] > opt.out_thresh]
      results.append(r)
      pubs.append([{'ct': (np.asarray(q['ct']) + np.asarray(q['tracking']) + rng.normal(0, 1, 2)).astype(np.float32)}
                   for q in r if rng.uniform() < 0.6])
    runner.step_host(img.pin_memory(), public_dets=pubs)
    tracks_np, counts_np = runner.fetch_tracks()
    got = runner.tracker.results(tracks_np, counts_np)
    for b in range(B):
      before = hosts[b].id_count
      want = hosts[b].step(results[b], pubs[b])
      _check_tracks(got[b], want, (t, b))
      assert int(counts_np[b, 1]) == hosts[b].id_count
      born += hosts[b].id_count - before
    pre = x
  assert born > 0
