"""--hungarian / --public_det on the device tracker, the parts that need no GPU: the assignment restatement the kernel
follows against scipy, the new argument checks of ct_track_step, and DeviceTracker's host-side public-detection and
seeding paths."""
import ctypes

import numpy as np
import pytest
import torch

from centertrack_b200 import _lib as L
from helpers import make_opt
from lsap_restated import lsap


@pytest.mark.parametrize('kind', ['int_ties', 'blocked_50', 'blocked_90', 'gated_tracker'])
def test_lsap_restatement_equals_scipy_pair_for_pair(kind):
  """Integer ties, half and 90 % blocked (all blocked pairs exactly 1e18), and tracker-like gated matrices; both
  N < M and N > M.  The tie rule decides which pairs come back forced through a blocked cell."""
  from scipy.optimize import linear_sum_assignment
  rng = np.random.RandomState(['int_ties', 'blocked_50', 'blocked_90', 'gated_tracker'].index(kind))
  for t in range(800):
    n, m = rng.randint(1, 25), rng.randint(1, 25)
    if kind == 'int_ties':
      c = rng.randint(0, 4, (n, m)).astype(np.float64)
    elif kind == 'gated_tracker':
      a = rng.uniform(0, 100, (n, 2)).astype(np.float32)
      b = (a[rng.randint(0, n, m)] + rng.normal(0, 3, (m, 2))).astype(np.float32)
      c = ((b[None] - a[:, None]) ** 2).sum(2).astype(np.float64)
      c[c > 30] = 1e18
    else:
      c = (rng.uniform(0, 50, (n, m)) ** 2).astype(np.float32).astype(np.float64)
      c[rng.uniform(size=(n, m)) < (0.5 if kind == 'blocked_50' else 0.9)] = 1e18
    want = linear_sum_assignment(c)
    got = lsap(c)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (kind, t, n, m)


def _desc():
  d = L.TrackDesc()
  p = 4096                                         # never dereferenced: validation precedes any launch
  d.B, d.K, d.F, d.rec_tracking, d.max_tracks = 2, 8, 13, 11, 16
  d.records = d.trans_out_inv = d.tracks = d.counts = p
  return d


def test_track_step_rejects_bad_association_arguments_without_a_gpu(built_lib):
  lib = L.lib()
  d = _desc()
  d.assign = 2
  assert lib.ct_track_step(ctypes.byref(d), None) == -1           # CT_ERR_INVALID
  assert b'unknown assign mode' in lib.ct_last_error()
  d = _desc()
  d.assign, d.public_det, d.max_public = L.CT_ASSIGN_HUNGARIAN, 4096, 4
  assert lib.ct_track_step(ctypes.byref(d), None) == -1
  assert b'public_det needs public_count' in lib.ct_last_error()
  d = _desc()
  d.max_public = -1
  assert lib.ct_track_step(ctypes.byref(d), None) == -1
  assert b'max_public < 0' in lib.ct_last_error()
  # the solver's scratch is part of the shared-memory budget
  assert lib.ct_track_smem_bytes(100, 300) >= lib.ct_track_smem_bytes(100, 100) + 200 * (16 + 16)


def _cpu_tracker(extra, max_public=None, B=2, K=8):
  from centertrack_b200.device_tracker import DeviceTracker
  opt = make_opt('coco_tracking', ['--track_thresh', '0.2', '--new_thresh', '0.3', '--pre_thresh', '0.25',
                                   '--input_h', '64', '--input_w', '96'] + extra)
  return opt, DeviceTracker(opt, B, K, 13, {'tracking': (11, 2)}, 64, 96, 'cpu', max_public=max_public)


def test_set_public_over_capacity_raises_and_never_truncates(built_lib):
  _, trk = _cpu_tracker(['--public_det', '--hungarian'], max_public=3)
  assert trk.desc.assign == L.CT_ASSIGN_HUNGARIAN and trk.desc.max_public == 3
  pub = [{'ct': np.array([i, 2 * i], np.float32)} for i in range(3)]
  trk.set_public(1, pub)
  assert trk.public_count.tolist() == [0, 3]
  assert trk.public[1].tolist() == [[0, 0], [1, 2], [2, 4]]
  with pytest.raises(ValueError, match='max_public'):
    trk.set_public(0, pub + [{'ct': [9, 9]}])
  assert trk.public_count.tolist() == [0, 3]
  trk.set_public(None, [[], pub[:1]])
  assert trk.public_count.tolist() == [0, 1]
  _, greedy = _cpu_tracker([])
  assert greedy.desc.assign == L.CT_ASSIGN_GREEDY and greedy.desc.public_det is None
  with pytest.raises(ValueError):
    greedy.set_public(0, pub)


def test_init_track_rows_and_prior_boxes_equal_the_host_tracker_and_detector(built_lib):
  """init_track seeds each stream like Tracker.init_track (score > new_thresh, ct from the box centre when absent)
  and writes the boxes the first frame's prior heat-map is drawn from, as Detector._get_additional_inputs draws it."""
  from centertrack_b200.detector import prior_splats
  from centertrack_b200.tracker import Tracker
  opt, trk = _cpu_tracker(['--public_det'])
  rng = np.random.RandomState(3)
  pre = []
  for b in range(2):
    one = []
    for _ in range(6):
      x, y, w, h = rng.uniform(-10, 100), rng.uniform(-10, 70), rng.uniform(1, 30), rng.uniform(1, 30)
      d = {'score': float(rng.uniform(0, 1)), 'class': int(rng.randint(1, 3)),
           'bbox': np.array([x, y, x + w, y + h], np.float32)}
      if rng.uniform() < 0.5:
        d['ct'] = np.array([x + 1, y + 2], np.float32)
      one.append(d)
    pre.append(one)
  trk.init_track(pre)
  got = trk.results(trk.tracks.numpy(), trk.counts.numpy())
  for b in range(2):
    host = Tracker(opt)
    host.init_track([dict(d) for d in pre[b]])
    assert len(got[b]) == len(host.tracks) == int(trk.counts[b, 1]) > 0
    for g, h in zip(got[b], host.tracks):
      assert (g['tracking_id'], g['age'], g['active'], g['class']) == (h['tracking_id'], 1, 1, h['class'])
      assert np.array_equal(g['ct'], np.asarray(h['ct'], np.float32)) and np.array_equal(g['bbox'], h['bbox'])
      assert np.array_equal(g['tracking'], np.zeros(2, np.float32))
    want = {h['tracking_id']: (c, r) for h, c, r in prior_splats(host.tracks, trk._t_in[b].reshape(2, 3), 96, 64,
                                                                  opt.pre_thresh)}
    bx = trk.boxes[b].numpy()
    for r in range(trk.T):
      tid = got[b][r]['tracking_id'] if r < len(got[b]) else None
      if tid in want:
        assert bx[r].tolist() == [b, want[tid][0][0], want[tid][0][1], want[tid][1], 0]
      else:
        assert bx[r, 3] == -1
