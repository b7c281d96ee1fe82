"""StreamRunner: the batched, graph-captured form of `Detector.run`'s device half for B independent video streams
on one GPU (SURVEY 8e: streams shard across GPUs, replicas of the weights, no data-path collective).

One step = for every stream its current frame: network (pre_img = that stream's previous frame, kept on
the device exactly like detector.py:148) + fused sigmoid + fused decode -> one packed record buffer
[B,K,F].  THREE input slots rotate: step t reads slot t%3 (images) and slot (t-1)%3 (pre_images: the previous
step's images, never copied) while the copy stream uploads step t+1's frames into slot (t+1)%3 -- with two slots
the upload would have to wait for the step that still reads its target as pre_images.  One CUDA graph per slot
replays the whole step as a single launch.  The FIRST step of a stream uses the frame itself as pre_images
(detector.py:99-103).

Two ways to feed the prior heat-map (`--pre_hm`):
  * device_tracking=False: the caller supplies pre_hm per step (what Detector._get_additional_inputs renders on the
    host).  With the one-step software pipeline of `step_host` the caller cannot have seen records(t-1) when it
    submits step t, so a host-rendered pre_hm is necessarily one frame stale -- this mode is for detection-style
    pipelines and for measuring the hot path with given inputs.
  * device_tracking=True (SURVEY 8f-1): the reference's dependency chain closed ON THE DEVICE, inside the same graph:
        pre_hm(t) = splat(tracks(t-1))  ->  network + decode -> records(t)  ->  tracks(t) = Tracker.step(records(t))
    (`DeviceTracker`: ct_render_tracks, ct_track_step).  Exact reference semantics (no stale prior), no host round
    trip; the host uploads only the frame and downloads the track table (ids, boxes, ages).  Greedy, --hungarian and
    --public_det association all run in the graph.  With --public_det each input slot also has its own buffer of
    public detections (the reference's `cur_dets`), uploaded with that slot's frame and read by that slot's graph;
    `reset_tracking(pre_dets)` seeds every stream's tracker at t = 0 like Tracker.init_track(meta['pre_dets']).

The end-to-end form (`step_host`) takes HOST frames: pinned staging, H2D on a copy stream overlapped
with the previous step's compute, graph replay, D2H of the records (and tracks).
"""
import numpy as np
import torch

from . import _lib as L
from .decode import generic_decode
from .device_tracker import DeviceTracker


NS = 3          # input slots


class StreamRunner(object):

  def __init__(self, model, B, H, W, K=100, precision='bf16', device='cuda', use_graph=True, opt=None,
               device_tracking=False, max_public=None):
    self.B, self.H, self.W, self.K = B, H, W, K
    self.device = torch.device(device)
    self.model = model
    self.opt = opt if opt is not None else getattr(model, 'opt', None)
    self.eng = model.engine_for(B, H, W, self.device, precision)
    self.eng.set_fused_activations(True)
    f32 = torch.float32
    self.img = [torch.zeros((B, 3, H, W), dtype=f32, device=self.device) for _ in range(NS)]
    self.hm = [torch.zeros((B, 1, H, W), dtype=f32, device=self.device) for _ in range(NS)]
    self.h_img = [torch.zeros((B, 3, H, W), dtype=f32).pin_memory() for _ in range(NS)]
    self.h_hm = [torch.zeros((B, 1, H, W), dtype=f32).pin_memory() for _ in range(NS)]
    self.rec = None
    self.layout = None
    self.ws = None                                           # private decode workspace (captured by the graphs)
    self.use_graph = use_graph
    self.graphs = [None] * NS
    self.compute = torch.cuda.Stream(device=self.device)
    self.copy = torch.cuda.Stream(device=self.device)
    self.ev_in = [torch.cuda.Event() for _ in range(NS)]     # slot uploaded
    self.ev_done = [torch.cuda.Event() for _ in range(NS)]   # slot no longer read (neither as images nor pre_images)
    self.t = 0
    self.tracker = None
    self.device_tracking = device_tracking
    self._eager(0, first=True)                               # sizes the record buffer
    self.pub = self.h_pub = None
    if device_tracking:
      assert self.opt is not None, 'device tracking needs opt (thresholds, max_age)'
      self.tracker = DeviceTracker(self.opt, B, K, self.rec.shape[2], self.layout, H, W, self.device,
                                   max_public=max_public)
      if self.tracker.public_det:                            # per slot: public detections of that slot's frame
        self.pub = [self.tracker.new_public_buffers(self.device) for _ in range(NS)]
        self.h_pub = [self.tracker.new_public_buffers('cpu', pin=True) for _ in range(NS)]
    torch.cuda.synchronize(self.device)
    self.h_rec = [torch.zeros_like(self.rec, device='cpu').pin_memory() for _ in range(2)]
    if self.tracker is not None:
      self.h_trk = [torch.zeros_like(self.tracker.tracks, device='cpu').pin_memory() for _ in range(2)]
      self.h_cnt = [torch.zeros_like(self.tracker.counts, device='cpu').pin_memory() for _ in range(2)]
    # launches of one step: the network plan + decode (+ memset-free: render + track step)
    self.launches_per_step = self.eng.n_launches + 1 + (2 if device_tracking else 0)

  # one step, eager launches on the current stream
  def _eager(self, slot, first=False):
    if self.tracker is not None:
      self.tracker.render(self.hm[slot])                     # pre_hm(t) from tracks(t-1)
    pre = self.img[slot] if first else self.img[(slot - 1) % NS]
    out = dict(self.eng.forward(self.img[slot], pre, self.hm[slot]))
    if self.ws is None:
      cat = out['hm'].shape[1]
      J = out['hm_hp'].shape[1] if ('hm_hp' in out and 'hps' in out) else 0
      self.ws = torch.zeros(L.lib().ct_decode_workspace_bytes(self.B, cat, J, self.K), dtype=torch.uint8,
                            device=self.device)
    res = generic_decode(out, K=self.K, records_out=self.rec, workspace=self.ws)
    if self.rec is None:
      self.rec, self.layout = res.records, res.layout
    if self.tracker is not None:
      self.tracker.step(self.rec, None if self.pub is None else self.pub[slot])     # tracks(t)
    return res

  def _graph(self, slot):
    if self.graphs[slot] is None:
      saved = None
      if self.tracker is not None:                           # capture must not disturb live stream state
        saved = (self.tracker.tracks.clone(), self.tracker.counts.clone(), self.tracker.boxes.clone())
      s = torch.cuda.Stream(device=self.device)
      s.wait_stream(torch.cuda.current_stream())
      with torch.cuda.stream(s):
        self._eager(slot)
      torch.cuda.current_stream().wait_stream(s)
      g = torch.cuda.CUDAGraph()
      with torch.cuda.graph(g):
        self._eager(slot)
      self.graphs[slot] = g
      if saved is not None:
        self.tracker.tracks.copy_(saved[0]); self.tracker.counts.copy_(saved[1]); self.tracker.boxes.copy_(saved[2])
    return self.graphs[slot]

  def warm(self):
    for s in range(NS):
      if self.use_graph:
        self._graph(s)
      else:
        self._eager(s)
    if self.tracker is not None:
      self.tracker.reset()
    torch.cuda.synchronize(self.device)

  def reset_tracking(self, pre_dets=None):
    """Restarts every stream at t = 0; pre_dets (a list of detection dicts per stream, device_tracking) seeds the
    trackers as Tracker.init_track does on the first frame of a --public_det video."""
    self.t = 0
    if self.tracker is not None:
      self.tracker.reset()
      if pre_dets is not None:
        self.tracker.init_track(pre_dets)

  def load_device_inputs(self, images, pre_hms, slot, public=None):
    """public (--public_det): device (centres [B,P,2] fp32, counts [B] int32) of this slot's frame, P <= max_public."""
    self.img[slot].copy_(images)
    if pre_hms is not None:
      self.hm[slot].copy_(pre_hms)
    if public is not None:
      centres, counts = public
      if self.pub is None:
        raise ValueError('public detections need device_tracking with --public_det')
      if centres.shape[1] > self.tracker.max_public or int(counts.max()) > self.tracker.max_public:
        raise ValueError('more public detections than max_public = %d' % self.tracker.max_public)
      self.pub[slot][0][:, :centres.shape[1]].copy_(centres)
      self.pub[slot][1].copy_(counts)

  def _launch(self, slot):
    if self.t == 0:
      self._eager(slot, first=True)                          # first frame of the streams: pre_images = images
    elif self.use_graph:
      self._graph(slot).replay()
    else:
      self._eager(slot)

  def step_device(self):
    """Inputs already resident in the slot buffers; runs on the current stream."""
    slot = self.t % NS
    self._launch(slot)
    self.t += 1
    return self.rec

  def step_host(self, images, pre_hms=None, public_dets=None):
    """images [B,3,H,W] (and pre_hms [B,1,H,W] unless device_tracking): float32 HOST tensors (what
    Detector.pre_process / _get_additional_inputs produce).  public_dets (device_tracking with --public_det): this
    frame's public detections, a list per stream of dicts with 'ct' (the reference's meta['cur_dets']); None = none.
    Returns the records of the PREVIOUS call (None the first time) -- a one-step software pipeline: this step's H2D
    overlaps the previous step's compute."""
    slot = self.t % NS
    if self.pub is not None:                         # staged on the host now, uploaded with the frame below
      h_pub, h_cnt = self.h_pub[slot]
      h_cnt.zero_()
      self.tracker.fill_public(h_pub, h_cnt, None, public_dets if public_dets is not None else [[]] * self.B)
    elif public_dets is not None:
      raise ValueError('public detections need device_tracking with --public_det')
    use_hm = self.tracker is None and pre_hms is not None
    src_img, src_hm = images, pre_hms
    if not images.is_pinned() or (use_hm and not pre_hms.is_pinned()):   # pageable input: stage through pinned memory
      self.h_img[slot].copy_(images)
      src_img = self.h_img[slot]
      if use_hm:
        self.h_hm[slot].copy_(pre_hms)
        src_hm = self.h_hm[slot]
    with torch.cuda.stream(self.copy):
      self.copy.wait_event(self.ev_done[slot])       # slot's old contents were last read as pre_images of step t-2
      self.img[slot].copy_(src_img, non_blocking=True)
      if use_hm:
        self.hm[slot].copy_(src_hm, non_blocking=True)
      if self.pub is not None:
        self.pub[slot][0].copy_(self.h_pub[slot][0], non_blocking=True)
        self.pub[slot][1].copy_(self.h_pub[slot][1], non_blocking=True)
      self.ev_in[slot].record(self.copy)
    prev = self.fetch() if self.t > 0 else None
    with torch.cuda.stream(self.compute):
      self.compute.wait_event(self.ev_in[slot])
      self._launch(slot)
      self.h_rec[self.t & 1].copy_(self.rec, non_blocking=True)
      if self.tracker is not None:
        self.h_trk[self.t & 1].copy_(self.tracker.tracks, non_blocking=True)
        self.h_cnt[self.t & 1].copy_(self.tracker.counts, non_blocking=True)
      # this step's pre_images slot may be overwritten once this step is done
      self.ev_done[(slot - 1) % NS].record(self.compute)
    self.t += 1
    return prev

  def fetch(self, copy=True):
    """Blocks until the last submitted step finished; returns its records as numpy [B,K,F].  A copy by default: the
    two pinned buffers are reused by the asynchronous D2H of later steps (copy=False hands out the pinned view, valid
    until the step after next is submitted)."""
    self.compute.synchronize()
    rec = self.h_rec[(self.t - 1) & 1].numpy()
    return rec.copy() if copy else rec

  def fetch_tracks(self):
    """(tracks [B,T,CT_TRK_FLOATS], counts [B,2]) of the last submitted step (device_tracking), as numpy copies."""
    self.compute.synchronize()
    i = (self.t - 1) & 1
    return self.h_trk[i].numpy().copy(), self.h_cnt[i].numpy().copy()

  @property
  def h2d_bytes_per_step(self):
    pub = 0 if self.pub is None else self.pub[0][0].numel() * 4 + self.pub[0][1].numel() * 4
    return self.B * (3 if self.tracker is not None else 4) * self.H * self.W * 4 + pub

  @property
  def d2h_bytes_per_step(self):
    return self.rec.numel() * 4 + (self.tracker.d2h_bytes if self.tracker is not None else 0)

  def views(self, rec_np):
    from .decode import views_from_records
    return {k: v.numpy() for k, v in views_from_records(torch.from_numpy(rec_np), self.layout).items()}
