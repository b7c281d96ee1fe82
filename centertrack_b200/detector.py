"""`Detector` with the reference's surface (src/lib/detector.py:23-458): `Detector(opt)`,
`run(image_or_path_or_tensor, meta={})`, `pre_process`, `process`, `post_process`, `merge_outputs`,
`reset_tracking`, attributes `.pause .tracker .pre_images .opt .model`; `run` returns the same dict
(`results` + the `tot/load/pre/net/dec/post/merge/track/display` wall-clock fields).

What differs underneath (`process`, detector.py:335-354): the network is a plan of libctb200 launches
(DLA34Engine) with the `_sigmoid_output` transforms fused into the head epilogues, decode is ONE fused
launch, and the 7-13 per-key blocking D2H copies become one copy of the packed record buffer.
Visualisation (`Debugger`, opt.debug >= 1) is outside the hot-path scope and is ignored.
"""
import ctypes as C
import math
import os
import time

import numpy as np
import torch

from . import _lib as L

from .dataset_info import get_dataset
from .decode import generic_decode
from .image import affine_transform, draw_umich_gaussian, gaussian_radius, get_affine_transform
from .model import create_model, load_model
from .post_process import generic_post_process
from .tracker import Tracker

_STAGES = ('load', 'pre', 'net', 'dec', 'post', 'merge', 'track', 'display')


class _StageClock(object):
  """Wall-clock bookkeeping of `run` (the reference reports these eight stage totals plus `tot`)."""

  def __init__(self):
    self.t0 = self.mark = time.time()
    self.acc = dict.fromkeys(_STAGES, 0.0)

  def lap(self, stage, now=None):
    now = time.time() if now is None else now
    self.acc[stage] += now - self.mark
    self.mark = now
    return now

  def report(self, results):
    out = {'results': results, 'tot': self.mark - self.t0}
    out.update(self.acc)
    return out


def trans_bbox(bbox, trans, width, height):
  """Box corners through a 2x3 affine map, clipped to [0, width-1] x [0, height-1] (detector.py:242-251)."""
  corners = np.asarray(bbox, dtype=np.float32).reshape(2, 2)
  moved = np.stack([affine_transform(corners[0], trans), affine_transform(corners[1], trans)]).astype(np.float32)
  return np.clip(moved, 0, np.array([width - 1, height - 1], dtype=np.float32)).reshape(4)


def prior_splats(dets, trans_input, inp_w, inp_h, pre_thresh):
  """The tracks the prior heat-map is drawn from (detector.py:259-276): active, score >= pre_thresh and a box of
  positive size once mapped onto the network input.  Yields (track, int32 centre on the input grid, radius).
  Detector._get_additional_inputs splats these on the host; DeviceTracker.init_track hands them to ct_render_tracks."""
  for trk in dets:
    if trk['active'] == 0 or trk['score'] < pre_thresh:
      continue
    x0, y0, x1, y1 = trans_bbox(trk['bbox'], trans_input, inp_w, inp_h)
    if not (y1 - y0 > 0 and x1 - x0 > 0):
      continue
    radius = max(0, int(gaussian_radius((math.ceil(y1 - y0), math.ceil(x1 - x0)))))
    centre = np.array([(x0 + x1) / 2, (y0 + y1) / 2], dtype=np.float32)
    yield trk, centre.astype(np.int32), radius


def _round_up(v, m):
  return (v + m - 1) // m * m


class Detector(object):

  def __init__(self, opt):
    self.model = self._init_device_model(opt)
    self.opt = opt
    ds = self.trained_dataset = get_dataset(opt.dataset)
    self.mean = np.asarray(ds.mean, dtype=np.float32).reshape(1, 1, 3)
    self.std = np.asarray(ds.std, dtype=np.float32).reshape(1, 1, 3)
    self.rest_focal_length = opt.test_focal_length if opt.test_focal_length >= 0 else ds.rest_focal_length
    self.flip_idx = ds.flip_idx
    self.pause = not opt.no_pause
    self.cnt = 0
    self.pre_images = None
    self.pre_image_ori = None
    self.tracker = Tracker(opt)
    self._graphs = {}

  @staticmethod
  def _init_device_model(opt):
    """detector.py:26-36: pick the device, build the network, load the checkpoint.  No CPU fallback."""
    if opt.gpus[0] < 0 or not torch.cuda.is_available():
      raise RuntimeError('centertrack_b200.Detector needs a CUDA device (B200, sm_100a); there is no '
                         'CPU fallback (got --gpus %s)' % getattr(opt, 'gpus_str', opt.gpus))
    opt.device = torch.device('cuda')
    print('Creating model...')
    model = create_model(opt.arch, opt.heads, opt.head_conv, opt=opt)
    if opt.load_model:
      model = load_model(model, opt.load_model, opt)
    else:
      print('Warning: no --load_model given; running with randomly initialised weights')
    return model.to(opt.device).eval()

  # ------------------------------------------------------------------------------------ run
  def _open_input(self, source):
    """ndarray (BGR HWC) | path | the dict test.py's DataLoader yields (already pre-processed per scale)."""
    if isinstance(source, np.ndarray):
      return source, None
    if isinstance(source, str):
      import cv2
      return cv2.imread(source), None
    return source['image'][0].numpy(), source

  @staticmethod
  def _scale_entry(packed, scale):
    """(images, meta) of one test scale out of the DataLoader dict (detector.py:84-92)."""
    meta = {k: v.numpy()[0] for k, v in packed['meta'][scale].items()}
    for k in ('pre_dets', 'cur_dets'):
      if k in packed['meta']:
        meta[k] = packed['meta'][k]
    return packed['images'][scale][0], meta

  def _tracking_inputs(self, images, meta):
    """First frame: the frame is its own pre_image and the tracker starts from `pre_dets`; then the prior heat-map
    rendered from the live tracks (detector.py:97-110)."""
    if not self.opt.tracking:
      return None, None
    if self.pre_images is None:
      print('Initialize tracking!')
      self.pre_images = images
      self.tracker.init_track(meta.get('pre_dets', []))
    if not self.opt.pre_hm:
      return None, None
    return self._get_additional_inputs(self.tracker.tracks, meta, with_hm=not self.opt.zero_pre_hm)

  def run(self, image_or_path_or_tensor, meta={}):
    """detector.py:55-172 without the visualisation branches; same return dict."""
    clock = _StageClock()
    image, packed = self._open_input(image_or_path_or_tensor)
    clock.lap('load')
    per_scale = []
    for scale in self.opt.test_scales:
      if packed is None:
        pre = self.pre_process_device if getattr(self.opt, 'b200_device_pre', False) else self.pre_process
        images, meta = pre(image, scale, meta)
      else:
        images, meta = self._scale_entry(packed, scale)
      images = images.to(self.opt.device, non_blocking=self.opt.non_block_test)
      pre_hms, pre_inds = self._tracking_inputs(images, meta)
      clock.lap('pre')
      _, dets, t_forward = self.process(images, self.pre_images, pre_hms, pre_inds, return_time=True)
      clock.lap('net', t_forward)
      clock.lap('dec')
      per_scale.append(self.post_process(dets, meta, scale))
      clock.lap('post')
    results = self.merge_outputs(per_scale)
    torch.cuda.synchronize()
    t_merged = clock.lap('merge')
    if self.opt.tracking:
      results = self.tracker.step(results, meta['cur_dets'] if self.opt.public_det else None)
      self.pre_images = images
    clock.lap('track')
    self.cnt += 1
    clock.acc['display'] += time.time() - t_merged        # the reference's display span starts at the merge mark
    ret = clock.report(results)
    if getattr(self.opt, 'save_video', False):            # detector.py:162-165: the frame demo.py writes to the video
      ret['generic'] = self._render_generic(image, results)
    return ret

  def _render_generic(self, image, results):
    """Stand-in for Debugger's 'generic' canvas (detector.py:379-445, out of the hot-path scope): the input frame with
    each result's box and `class[:tracking id] score` label.  BGR uint8, same size as the input frame."""
    import cv2
    canvas = np.ascontiguousarray(image).copy()
    for r in results:
      if r['score'] <= getattr(self.opt, 'vis_thresh', 0.3):
        continue
      x0, y0, x1, y1 = [int(round(float(v))) for v in r['bbox'][:4]]
      tid = int(r.get('tracking_id', 0))
      colour = ((37 * tid) % 255, (17 * tid + 80) % 255, (29 * tid + 160) % 255)
      cv2.rectangle(canvas, (x0, y0), (x1, y1), colour, 2)
      label = '%d:%d %.2f' % (int(r['class']), tid, float(r['score'])) if 'tracking_id' in r else \
          '%d %.2f' % (int(r['class']), float(r['score']))
      cv2.putText(canvas, label, (x0, max(0, y0 - 3)), cv2.FONT_HERSHEY_SIMPLEX, 0.5, colour, 1, cv2.LINE_AA)
    return canvas

  # ------------------------------------------------------------------------------------ host pre
  def _input_geometry(self, height, width, scale):
    """Network input size and the (centre, scale) of the source rectangle mapped onto it, for the three resolution
    policies of detector.py:175-204: --fix_short (short side fixed, long side rounded up to 64), fixed resolution
    (default), or keep_res (image size padded up to (size | pad) + 1)."""
    opt = self.opt
    sh, sw = int(height * scale), int(width * scale)
    if opt.fix_short > 0:
      long_side = lambda a, b: _round_up(int(a / b * opt.fix_short), 64)
      inp_h, inp_w = (opt.fix_short, long_side(width, height)) if height < width else \
                     (long_side(height, width), opt.fix_short)
      centre = np.array([width / 2, height / 2], dtype=np.float32)
      extent = np.array([width, height], dtype=np.float32)
    elif opt.fix_res:
      inp_h, inp_w = opt.input_h, opt.input_w
      centre = np.array([sw / 2., sh / 2.], dtype=np.float32)
      extent = max(height, width) * 1.0
    else:
      inp_h, inp_w = (sh | opt.pad) + 1, (sw | opt.pad) + 1
      centre = np.array([sw // 2, sh // 2], dtype=np.float32)
      extent = np.array([inp_w, inp_h], dtype=np.float32)
    return (sh, sw), centre, extent, inp_w, inp_h

  def _transform_scale(self, image, scale=1):
    """Reference-named helper (detector.py:175): resized image + geometry tuple."""
    import cv2
    height, width = image.shape[:2]
    (sh, sw), c, s, inp_w, inp_h = self._input_geometry(height, width, scale)
    return cv2.resize(image, (sw, sh)), c, s, inp_w, inp_h, height, width

  def pre_process(self, image, scale, input_meta={}):
    """detector.py:207-239 (CPU only and fork-safe: test.py hands it to a DataLoader worker).
    Like the reference (hazard H5) `scale` is not forwarded to the geometry."""
    import cv2
    resized, c, s, inp_w, inp_h, height, width = self._transform_scale(image)
    out_w, out_h = inp_w // self.opt.down_ratio, inp_h // self.opt.down_ratio
    to_input = get_affine_transform(c, s, 0, [inp_w, inp_h])
    to_output = get_affine_transform(c, s, 0, [out_w, out_h])
    warped = cv2.warpAffine(resized, to_input, (inp_w, inp_h), flags=cv2.INTER_LINEAR)
    chw = ((warped / 255. - self.mean) / self.std).astype(np.float32).transpose(2, 0, 1)
    images = chw.reshape(1, 3, inp_h, inp_w)
    if self.opt.flip_test:                                  # detector.py:225-226
      images = np.concatenate((images, images[:, :, :, ::-1]), axis=0)
    images = torch.from_numpy(np.ascontiguousarray(images))
    calib = np.array(input_meta['calib'], dtype=np.float32) if 'calib' in input_meta \
        else self._get_default_calib(width, height)
    meta = dict(calib=calib, c=c, s=s, height=height, width=width, out_height=out_h, out_width=out_w,
                inp_height=inp_h, inp_width=inp_w, trans_input=to_input, trans_output=to_output)
    meta.update({k: input_meta[k] for k in ('pre_dets', 'cur_dets') if k in input_meta})
    return images, meta

  def pre_process_device(self, image, scale, input_meta={}):
    """SURVEY 8f-2: the same contract as `pre_process`, with the per-pixel work -- cv2.warpAffine(INTER_LINEAR),
    (x/255 - mean)/std, HWC -> CHW -- done by ct_warp_affine_normalize on the GPU from the raw uint8 frame (the
    geometry stays on the host; `pre_process` itself must remain CPU-only and fork-safe for test.py's DataLoader).
    Returns CUDA `images`."""
    height, width = image.shape[:2]
    (sh, sw), c, s, inp_w, inp_h = self._input_geometry(height, width, 1)     # hazard H5: scale is not forwarded
    if (sh, sw) != (height, width):
      import cv2
      image = cv2.resize(image, (sw, sh))
    out_w, out_h = inp_w // self.opt.down_ratio, inp_h // self.opt.down_ratio
    to_input = get_affine_transform(c, s, 0, [inp_w, inp_h])
    to_output = get_affine_transform(c, s, 0, [out_w, out_h])
    M = np.asarray(to_input, np.float64).reshape(6).copy()                   # cv::warpAffine inverts the map like this
    D = M[0] * M[4] - M[1] * M[3]
    D = 1. / D if D != 0 else 0.
    A11, A22 = M[4] * D, M[0] * D
    M[0] = A11; M[1] *= -D; M[3] *= -D; M[4] = A22
    b1, b2 = -M[0] * M[2] - M[1] * M[5], -M[3] * M[2] - M[4] * M[5]
    M[2], M[5] = b1, b2
    dev = self.opt.device
    src = torch.from_numpy(np.ascontiguousarray(image)).to(dev, non_blocking=True)
    minv = torch.from_numpy(M.reshape(1, 6)).to(dev)
    out = torch.empty((1, 3, inp_h, inp_w), dtype=torch.float32, device=dev)
    mean = np.ascontiguousarray(self.mean.reshape(3), dtype=np.float32)
    std = np.ascontiguousarray(self.std.reshape(3), dtype=np.float32)
    L.check(L.lib().ct_warp_affine_normalize(L.ptr(src), 1, image.shape[0], image.shape[1], image.shape[1] * 3,
                                             L.ptr(minv), C.c_void_p(mean.ctypes.data), C.c_void_p(std.ctypes.data),
                                             L.ptr(out), inp_h, inp_w, L.stream_ptr()), 'ct_warp_affine_normalize')
    images = torch.cat((out, out.flip(3)), 0) if self.opt.flip_test else out
    calib = np.array(input_meta['calib'], dtype=np.float32) if 'calib' in input_meta \
        else self._get_default_calib(width, height)
    meta = dict(calib=calib, c=c, s=s, height=height, width=width, out_height=out_h, out_width=out_w,
                inp_height=inp_h, inp_width=inp_w, trans_input=to_input, trans_output=to_output)
    meta.update({k: input_meta[k] for k in ('pre_dets', 'cur_dets') if k in input_meta})
    return images, meta

  def _trans_bbox(self, bbox, trans, width, height):
    """Box corners through a 2x3 affine map, clipped to [0, width-1] x [0, height-1] (detector.py:242-251)."""
    return trans_bbox(bbox, trans, width, height)

  def _get_additional_inputs(self, dets, meta, with_hm=True):
    """detector.py:254-290: the prior heat-map [1,1,inp_h,inp_w] splatted from the tracks that are active and score at
    least pre_thresh, plus their centre indices on the output grid."""
    inp_w, inp_h, out_w, out_h = meta['inp_width'], meta['inp_height'], meta['out_width'], meta['out_height']
    canvas = np.zeros((1, inp_h, inp_w), dtype=np.float32)
    inds = []
    for trk, centre, radius in prior_splats(dets, meta['trans_input'], inp_w, inp_h, self.opt.pre_thresh):
      if with_hm:
        draw_umich_gaussian(canvas[0], centre, radius)
      ox0, oy0, ox1, oy1 = self._trans_bbox(trk['bbox'], meta['trans_output'], out_w, out_h)
      cell = np.array([(ox0 + ox1) / 2, (oy0 + oy1) / 2], dtype=np.int32)
      inds.append(cell[1] * out_w + cell[0])
    if with_hm:
      canvas = canvas[np.newaxis]
      if self.opt.flip_test:                                 # detector.py:285-286
        canvas = np.concatenate((canvas, canvas[:, :, :, ::-1]), axis=0)
      canvas = torch.from_numpy(np.ascontiguousarray(canvas)).to(self.opt.device)
    pre_inds = torch.from_numpy(np.array(inds, np.int64).reshape(1, -1)).to(self.opt.device)
    return canvas, pre_inds

  def _get_default_calib(self, width, height):
    return np.array([[self.rest_focal_length, 0, width / 2, 0],
                     [0, self.rest_focal_length, height / 2, 0],
                     [0, 0, 1, 0]])

  def _sigmoid_output(self, output):
    """detector.py:300-308 (kept for callers that run the nn.Module surface themselves; `process`
    fuses these transforms into the head epilogues)."""
    if 'hm' in output:
      output['hm'] = output['hm'].sigmoid_()
    if 'hm_hp' in output:
      output['hm_hp'] = output['hm_hp'].sigmoid_()
    if 'dep' in output:
      output['dep'] = 1. / (output['dep'].sigmoid() + 1e-6) - 1.
      output['dep'] *= self.opt.depth_scale
    return output

  # ------------------------------------------------------------------------------------ hot path
  def _flip_plan(self, eng):
    """Which heads Detector._flip_output (detector.py:311-332) averages with the mirrored pass, and how:
    {head: (perm or None, sign or None)}; every other head keeps its un-flipped pass."""
    plan = {}
    dev = eng.device
    pairs = {}
    for a, b in getattr(self, 'flip_idx', None) or get_dataset(self.opt.dataset).flip_idx:
      pairs[a], pairs[b] = b, a
    for h, t in eng.outputs.items():
      c = t.shape[1]
      if h in ('hm', 'wh', 'dep', 'dim'):
        plan[h] = (None, None)
      elif h == 'amodel_offset':                              # flipped copy with its x components negated
        plan[h] = (None, torch.tensor([-1. if i % 2 == 0 else 1. for i in range(c)], dtype=torch.float32, device=dev))
      elif h == 'hps':                                        # flip_lr_off: mirror, negate x offsets, swap left/right joints
        perm = [2 * pairs.get(i // 2, i // 2) + (i % 2) for i in range(c)]
        plan[h] = (torch.tensor(perm, dtype=torch.int32, device=dev),
                   torch.tensor([-1. if i % 2 == 0 else 1. for i in range(c)], dtype=torch.float32, device=dev))
      elif h == 'hm_hp':                                      # flip_lr: mirror, swap left/right joints
        plan[h] = (torch.tensor([pairs.get(i, i) for i in range(c)], dtype=torch.int32, device=dev), None)
    return plan

  def _flip_output(self, output, plan, merged):
    """Device form of detector.py:311-332 on the post-activation maps of a (frame, mirrored frame) pair."""
    res = {}
    for h, t in output.items():
      if h in plan:
        perm, sign = plan[h]
        L.check(L.lib().ct_flip_merge(L.ptr(t), L.ptr(merged[h]), t.shape[1], t.shape[2], t.shape[3], L.ptr(perm),
                                      L.ptr(sign), L.stream_ptr()), 'ct_flip_merge')
        res[h] = merged[h]
      else:
        res[h] = t[0:1]
    return res

  def _process_plan(self, B, H, W, device, has_pre, has_hm):
    """Everything `process` launches for one input signature, built once: engine plan, flip-merge buffers, decode
    buffers, and a CUDA graph of the lot (CTB_NO_GRAPH=1 keeps it eager)."""
    key = (B, H, W, str(device), has_pre, has_hm, bool(self.opt.flip_test))
    if not hasattr(self, '_graphs'):
      self._graphs = {}
    p = self._graphs.get(key)
    if p is not None and p['eng'] is self.model.engine_for(B, H, W, device):
      return p
    eng = self.model.engine_for(B, H, W, device)
    if not eng.fused_act:
      eng.set_fused_activations(True)
    p = {'eng': eng, 'graph': None, 'rec': None, 'ws': None, 'res': None, 'out': None}
    if self.opt.flip_test:
      assert B == 2, 'flip_test runs the frame and its mirror image as a batch of 2'
      p['plan'] = self._flip_plan(eng)
      p['merged'] = {h: torch.empty((1,) + tuple(eng.outputs[h].shape[1:]), dtype=torch.float32, device=device)
                     for h in p['plan']}
    img = eng.in_img
    pre = eng.in_pre if has_pre else None
    hm = eng.in_hm if has_hm else None

    def launch():
      out = dict(eng.forward(img, pre, hm))
      if self.opt.flip_test:
        out = self._flip_output(out, p['plan'], p['merged'])
      if p['ws'] is None:
        cat = out['hm'].shape[1]
        J = out['hm_hp'].shape[1] if ('hm_hp' in out and 'hps' in out) else 0
        p['ws'] = torch.zeros(L.lib().ct_decode_workspace_bytes(out['hm'].shape[0], cat, J, self.opt.K),
                              dtype=torch.uint8, device=device)
      res = generic_decode(out, K=self.opt.K, opt=self.opt, records_out=p['rec'], workspace=p['ws'])
      p['rec'], p['res'], p['out'] = res.records, res, out

    p['launch'] = launch
    if not int(os.environ.get('CTB_NO_GRAPH', '0')):
      side = torch.cuda.Stream(device=device)
      side.wait_stream(torch.cuda.current_stream())
      with torch.cuda.stream(side):
        launch(); launch()
      torch.cuda.current_stream().wait_stream(side)
      g = torch.cuda.CUDAGraph()
      with torch.cuda.graph(g):
        launch()
      p['graph'] = g
    self._graphs[key] = p
    return p

  def process(self, images, pre_images=None, pre_hms=None, pre_inds=None, return_time=False):
    """detector.py:335-354: network + _sigmoid_output (+ _flip_output) + generic_decode + D2H.  One CUDA-graph replay
    (the 87 launches of the DLA-34 plan, the flip merge, the fused decode) and ONE device->host copy."""
    with torch.no_grad():
      torch.cuda.synchronize()
      B, _, H, W = images.shape
      has_hm = isinstance(pre_hms, torch.Tensor)
      p = self._process_plan(B, H, W, images.device, pre_images is not None, has_hm)
      eng = p['eng']
      eng.in_img.copy_(images)
      if pre_images is not None:
        eng.in_pre.copy_(pre_images)
      if has_hm:
        eng.in_hm.copy_(pre_hms)
      if p['graph'] is not None:
        p['graph'].replay()
      else:
        p['launch']()
      output = dict(p['out'])
      output.update({'pre_inds': pre_inds})
      torch.cuda.synchronize()
      forward_time = time.time()
      dets_dev = p['res']
      rec = dets_dev.records.cpu().numpy()          # the single device->host copy (synchronises)
      dets = {}
      if pre_inds is not None:                      # decode.py:173-180
        Wo = output['hm'].shape[3]
        dets['pre_cts'] = torch.stack([(pre_inds % Wo).float(), torch.div(pre_inds, Wo, rounding_mode='floor').float()],
                                      dim=2).cpu().numpy()
      dets.update(_numpy_views(rec, dets_dev))
    if return_time:
      return output, dets, forward_time
    return output, dets

  def post_process(self, dets, meta, scale=1):
    """detector.py:356-369."""
    dets = generic_post_process(self.opt, dets, [meta['c']], [meta['s']], meta['out_height'],
                                meta['out_width'], self.opt.num_classes, [meta['calib']],
                                meta['height'], meta['width'])
    self.this_calib = meta['calib']
    if scale != 1:
      for i in range(len(dets[0])):
        for k in ['bbox', 'hps']:
          if k in dets[0][i]:
            dets[0][i][k] = (np.array(dets[0][i][k], np.float32) / scale).tolist()
    return dets[0]

  def merge_outputs(self, detections):
    """detector.py:371-377."""
    assert len(self.opt.test_scales) == 1, 'multi_scale not supported!'
    return [d for d in detections[0] if d['score'] > self.opt.out_thresh]

  def reset_tracking(self):
    self.tracker.reset()
    self.pre_images = None
    self.pre_image_ori = None


def _numpy_views(rec, dets_dev):
  """Re-slice the host copy of the record buffer exactly like decode.views_from_records did on device."""
  from .decode import views_from_records
  t = torch.from_numpy(rec)
  out = views_from_records(t, dets_dev.layout)
  return {k: v.numpy() for k, v in out.items()}
