"""Per-stream tracker state kept on the GPU between frames (SURVEY 8f-1): the reference's
`generic_post_process` affine (utils/post_process.py:21-91), `Tracker.step` association (utils/tracker.py:28-138)
and the prior heat-map render of `Detector._get_additional_inputs` (detector.py:254-290) as two launches on the decode
records -- `ct_track_step` and `ct_render_tracks` -- so that a stream never returns to the host between frames:
records(t) -> tracks(t) -> pre_hm(t+1) are all device-resident and CUDA-graph capturable (fixed launch shapes).

All three association modes of the reference run on the device: greedy matching (default), `--hungarian` (a
minimum-cost assignment that returns what scipy's linear_sum_assignment returns, tie for tie) and the MOT
`--public_det` protocol (a track may only start on a detection that a public detection claims; `set_public` uploads
a frame's public detections, `init_track` seeds the streams from `pre_dets` like Tracker.init_track).
Results are rows of CT_TRK_FLOATS fp32 (score, class, ct, tracking, bbox, tracking_id, age, active) in the
reference's output order (matched detections, new tracks, coasting tracks); `results()` turns a host copy into the
reference's list of dicts.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L
from .image import get_affine_transform


class DeviceTracker(object):

  def __init__(self, opt, B, K, rec_floats, layout, inp_h, inp_w, device, centers=None, scales=None, max_tracks=None,
               max_public=None):
    """centers/scales: per-stream (c, s) of the source rectangle (Detector._input_geometry); default = a source image
    of exactly the network input size (the synthetic benchmark streams).  max_public: capacity of the per-stream
    public-detection list with --public_det (default K)."""
    self.opt, self.B, self.K, self.F = opt, B, K, rec_floats
    self.inp_h, self.inp_w = inp_h, inp_w
    self.device = torch.device(device)
    self.T = int(max_tracks or (K * (1 + max(0, int(opt.max_age)))))
    self.T = max(self.T, K)
    down = getattr(opt, 'down_ratio', 4)
    out_w, out_h = inp_w // down, inp_h // down
    t_out = np.zeros((B, 6), np.float32)
    t_in = np.zeros((B, 6), np.float64)
    for b in range(B):
      c = np.array([inp_w / 2., inp_h / 2.], np.float32) if centers is None else np.asarray(centers[b], np.float32)
      s = max(inp_h, inp_w) * 1.0 if scales is None else scales[b]
      t_out[b] = get_affine_transform(c, s, 0, (out_w, out_h), inv=1).astype(np.float32).reshape(6)
      t_in[b] = get_affine_transform(c, s, 0, [inp_w, inp_h]).reshape(6)
    self.trans_out_inv = torch.from_numpy(t_out).to(self.device)
    self.trans_input = torch.from_numpy(t_in).to(self.device)
    self._t_in = t_in
    self.tracks = torch.zeros((B, self.T, L.CT_TRK_FLOATS), dtype=torch.float32, device=self.device)
    self.counts = torch.zeros((B, 2), dtype=torch.int32, device=self.device)
    self.boxes = torch.zeros((B, self.T, 5), dtype=torch.float32, device=self.device)
    self.boxes[:, :, 3] = -1.0                       # no tracks yet: nothing to splat (first frame: pre_hm = 0)
    d = L.TrackDesc()
    d.B, d.K, d.F = B, K, rec_floats
    d.rec_tracking = layout['tracking'][0] if 'tracking' in layout else -1
    d.max_tracks = self.T
    d.out_thresh, d.new_thresh, d.pre_thresh = float(opt.out_thresh), float(opt.new_thresh), float(opt.pre_thresh)
    d.max_age = int(opt.max_age)
    d.inp_h, d.inp_w = inp_h, inp_w
    d.trans_out_inv, d.trans_input = self.trans_out_inv.data_ptr(), self.trans_input.data_ptr()
    d.tracks, d.counts, d.boxes = self.tracks.data_ptr(), self.counts.data_ptr(), self.boxes.data_ptr()
    d.assign = L.CT_ASSIGN_HUNGARIAN if getattr(opt, 'hungarian', False) else L.CT_ASSIGN_GREEDY
    self.public_det = bool(getattr(opt, 'public_det', False))
    self.max_public = int(K if max_public is None else max_public)
    if self.max_public < 0:
      raise ValueError('max_public < 0')
    self.public = self.public_count = None
    if self.public_det:                              # this frame's public detections: centres, count per stream
      self.public, self.public_count = self.new_public_buffers(self.device)
      d.public_det, d.public_count = self.public.data_ptr(), self.public_count.data_ptr()
      d.max_public = self.max_public
    self.desc = d
    if L.lib().ct_track_smem_bytes(K, self.T) > 200 * 1024:
      raise ValueError('track table of %d rows does not fit in shared memory' % self.T)

  def new_public_buffers(self, device, pin=False):
    """Zeroed (centres [B,max_public,2] fp32, counts [B] int32) in the layout ct_track_step reads."""
    pub = torch.zeros((self.B, max(1, self.max_public), 2), dtype=torch.float32, device=device)
    cnt = torch.zeros((self.B,), dtype=torch.int32, device=device)
    return (pub.pin_memory(), cnt.pin_memory()) if pin else (pub, cnt)

  def fill_public(self, pub, cnt, b_or_all, dets):
    """Writes public detections (the reference's `cur_dets`: dicts with 'ct' in image coordinates) into host or
    device buffers of `new_public_buffers`: `dets` is one stream's list when b_or_all is a stream index, else (None)
    a list per stream.  A stream with more than max_public detections raises ValueError; nothing is dropped."""
    streams = range(self.B) if b_or_all is None else [int(b_or_all)]
    lists = dets if b_or_all is None else [dets]
    if len(lists) != len(streams):
      raise ValueError('expected public detections for %d streams, got %d' % (len(streams), len(lists)))
    for b, one in zip(streams, lists):
      n = len(one)
      if n > self.max_public:
        raise ValueError('stream %d has %d public detections, more than max_public = %d' % (b, n, self.max_public))
      if n:
        ct = np.array([np.asarray(x['ct'], np.float32)[:2] for x in one], np.float32).reshape(n, 2)
        pub[b, :n].copy_(torch.from_numpy(ct))
      cnt[b] = n

  def set_public(self, b_or_all, dets):
    """This frame's public detections for stream b (or, with b_or_all=None, for every stream), read by the next
    `step` (--public_det only)."""
    if not self.public_det:
      raise ValueError('set_public needs --public_det')
    self.fill_public(self.public, self.public_count, b_or_all, dets)

  def reset(self):
    """Detector.reset_tracking / Tracker.reset for every stream."""
    self.tracks.zero_()
    self.counts.zero_()
    self.boxes.zero_()
    self.boxes[:, :, 3] = -1.0

  def init_track(self, pre_dets_per_stream):
    """Tracker.init_track for every stream at once (the first frame of the MOT --public_det protocol seeds the
    tracker from the loaded detections, `pre_dets`): detections with score > new_thresh start tracks with ids
    1, 2, ... in order (age 1, active 1, tracking 0, `ct` from the box centre when absent), and the boxes of the
    first frame's prior heat-map are computed from them as Detector._get_additional_inputs does on the host."""
    from .detector import prior_splats
    if len(pre_dets_per_stream) != self.B:
      raise ValueError('expected pre_dets for %d streams, got %d' % (self.B, len(pre_dets_per_stream)))
    tracks = np.zeros((self.B, self.T, L.CT_TRK_FLOATS), np.float32)
    counts = np.zeros((self.B, 2), np.int32)
    boxes = np.zeros((self.B, self.T, 5), np.float32)
    boxes[:, :, 0] = np.arange(self.B, dtype=np.float32)[:, None]
    boxes[:, :, 3] = -1.0
    for b, dets in enumerate(pre_dets_per_stream):
      born = []
      for item in dets:
        if item['score'] <= self.opt.new_thresh:
          continue
        trk = dict(item, tracking_id=len(born) + 1, age=1, active=1)
        if 'ct' not in trk:
          x0, y0, x1, y1 = trk['bbox'][:4]
          trk['ct'] = [(x0 + x1) / 2, (y0 + y1) / 2]
        born.append(trk)
      if len(born) > self.T:
        raise ValueError('stream %d: %d initial tracks do not fit the %d-row track table' % (b, len(born), self.T))
      for r, trk in enumerate(born):
        row = tracks[b, r]
        row[L.CT_TRK_SCORE], row[L.CT_TRK_CLASS] = trk['score'], trk['class']
        row[L.CT_TRK_CT:L.CT_TRK_CT + 2] = np.asarray(trk['ct'], np.float32)[:2]
        row[L.CT_TRK_BBOX:L.CT_TRK_BBOX + 4] = np.asarray(trk['bbox'], np.float32)[:4]
        row[L.CT_TRK_ID], row[L.CT_TRK_AGE], row[L.CT_TRK_ACTIVE] = trk['tracking_id'], 1, 1
      counts[b] = len(born), len(born)
      trans_input = self._t_in[b].reshape(2, 3)
      row_of = {id(t): r for r, t in enumerate(born)}
      for trk, centre, radius in prior_splats(born, trans_input, self.inp_w, self.inp_h, self.opt.pre_thresh):
        boxes[b, row_of[id(trk)], 1:4] = centre[0], centre[1], radius
    self.tracks.copy_(torch.from_numpy(tracks))
    self.counts.copy_(torch.from_numpy(counts))
    self.boxes.copy_(torch.from_numpy(boxes))

  def step(self, records, public=None):
    """records [B,K,F] (ct_decode) -> updates tracks/counts/boxes in place, on the current stream.  public: optional
    (centres, counts) device buffers of `new_public_buffers` to read instead of the tracker's own (--public_det)."""
    assert records.is_cuda and records.dtype == torch.float32 and tuple(records.shape) == (self.B, self.K, self.F)
    self.desc.records = records.data_ptr()
    if self.public_det:
      pub, cnt = public if public is not None else (self.public, self.public_count)
      self.desc.public_det, self.desc.public_count = pub.data_ptr(), cnt.data_ptr()
    L.check(L.lib().ct_track_step(C.byref(self.desc), L.stream_ptr()), 'ct_track_step')

  def render(self, pre_hm):
    """pre_hm [B,1,H,W] fp32 <- splat of the current tracks (what the NEXT frame's network reads)."""
    assert pre_hm.is_cuda and pre_hm.dtype == torch.float32 and tuple(pre_hm.shape) == (self.B, 1, self.inp_h, self.inp_w)
    L.check(L.lib().ct_render_tracks(L.ptr(self.boxes), self.B * self.T, L.ptr(pre_hm), self.B, self.inp_h,
                                     self.inp_w, L.stream_ptr()), 'ct_render_tracks')

  @property
  def d2h_bytes(self):
    return self.tracks.numel() * 4 + self.counts.numel() * 4

  @staticmethod
  def results(tracks_np, counts_np):
    """Host copies -> [[{score, class, ct, tracking, bbox, tracking_id, age, active}, ...] per stream]."""
    out = []
    for b in range(tracks_np.shape[0]):
      rows = tracks_np[b, :int(counts_np[b, 0])]
      out.append([{'score': float(r[L.CT_TRK_SCORE]), 'class': int(r[L.CT_TRK_CLASS]),
                   'ct': r[L.CT_TRK_CT:L.CT_TRK_CT + 2].copy(), 'tracking': r[L.CT_TRK_TRACKING:L.CT_TRK_TRACKING + 2].copy(),
                   'bbox': r[L.CT_TRK_BBOX:L.CT_TRK_BBOX + 4].copy(), 'tracking_id': int(r[L.CT_TRK_ID]),
                   'age': int(r[L.CT_TRK_AGE]), 'active': int(r[L.CT_TRK_ACTIVE])} for r in rows])
    return out
