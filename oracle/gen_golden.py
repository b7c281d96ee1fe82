"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference, via oracle/ref_harness.py) on CPU in the build container:

    python oracle/gen_golden.py            # needs /root/reference; run here, commit the outputs

Inputs and weights are pure functions of seeds (oracle/weights.py, numpy RandomState) so the GPU box
regenerates them bit-identically without the reference; only the reference's OUTPUTS are stored.
"""
import hashlib
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness as rh          # noqa
sys.path.insert(0, os.path.join(HERE, '..'))
from centertrack_b200 import synthetic as wt   # noqa

OUT = os.environ.get('CT_GOLDEN_OUT') or os.path.join(HERE, '..', 'tests', 'golden')
SMALL_HW = (64, 96)
STAGES = ['base.level2', 'base.level3', 'base.level4', 'base.level5', 'dla_up.ida_0.proj_1',
          'dla_up.ida_0.node_1', 'dla_up.ida_1.node_2', 'dla_up.ida_2.node_3', 'ida_up.node_1', 'ida_up.node_2']


def decode_inputs(kind, B, C, H, W, seed):
  """Seeded decode-only inputs (SURVEY 8d): hm = sigmoid(2 N(0,1) - 4.6), heads ~ N(0,1)."""
  rng = np.random.RandomState(seed)
  out = {'hm': (1. / (1. + np.exp(-(2 * rng.randn(B, C, H, W) - 4.6)))).astype(np.float32),
         'reg': rng.rand(B, 2, H, W).astype(np.float32),
         'wh': (rng.randn(B, 2, H, W) * 6).astype(np.float32),
         'tracking': (rng.randn(B, 2, H, W) * 3).astype(np.float32)}
  if kind == 'ddd':
    out.update({'dep': (rng.rand(B, 1, H, W) * 60).astype(np.float32),
                'rot': rng.randn(B, 8, H, W).astype(np.float32),
                'dim': (rng.rand(B, 3, H, W) * 4).astype(np.float32),
                'amodel_offset': rng.randn(B, 2, H, W).astype(np.float32)})
  if kind == 'pose':
    out.update({'hps': (rng.randn(B, 34, H, W) * 6).astype(np.float32),
                'hm_hp': (1. / (1. + np.exp(-(2 * rng.randn(B, 17, H, W) - 3.0)))).astype(np.float32),
                'hp_offset': rng.rand(B, 2, H, W).astype(np.float32)})
  if kind == 'mot':
    out['ltrb_amodal'] = (rng.randn(B, 4, H, W) * 8).astype(np.float32)
  return out


DECODE_CASES = [('coco', 1, 80, 128, 128, 100, 11), ('mot', 1, 1, 136, 240, 100, 12),
                ('ddd', 1, 10, 112, 200, 100, 13), ('pose', 1, 1, 128, 128, 100, 14),
                ('coco', 2, 80, 32, 32, 50, 15)]


def gen_net():
  for cfg, node in [('coco_tracking', 'dcn'), ('mot', 'dcn'), ('nuscenes_ddd', 'dcn'), ('coco_pose', 'dcn'),
                    ('coco_tracking', 'conv'), ('coco_tracking', 'gcn')]:          # --dla_node (dla.py:588-592)
    opt, model = rh.build_reference_model(cfg, input_hw=SMALL_HW, extra=['--dla_node', node])
    sd = wt.make_state_dict(model.state_dict(), 317)
    model.load_state_dict(sd)
    img, pre, hm = wt.synthetic_inputs(1, *SMALL_HW)
    acts = {}
    hooks = []
    if cfg == 'coco_tracking':
      mods = dict(model.named_modules())
      for name in STAGES:
        hooks.append(mods[name].register_forward_hook(
            lambda m, i, o, name=name: acts.__setitem__(name, o.detach().clone())))
    with torch.no_grad():
      out = model(img, pre, hm)[-1]
    for h in hooks:
      h.remove()
    data = {'head.' + k: v.numpy() for k, v in out.items()}
    data.update({'stage.' + k: v.numpy() for k, v in acts.items()})
    data['keys'] = np.array(sorted(sd.keys()))
    stem = 'net_%s_64x96.npz' % cfg if node == 'dcn' else 'net_%s_%s_64x96.npz' % (cfg, node)
    np.savez_compressed(os.path.join(OUT, stem), **data)
    print('net', cfg, node, {k: v.shape for k, v in data.items() if k != 'keys'})


GENERIC_RENAME = (('backbone.', 'base.'), ('neck.dla_up.', 'dla_up.'), ('neck.ida_up.', 'ida_up.'))


def gen_generic():
  """--arch generic --backbone dla34 --neck dlaup (generic_network.py:29-107): the reference's GenericNetwork on the
  synthetic checkpoint (same tensors as the dla_34 goldens, generated under the DLASeg names), with its own default
  head width (64: opts.py:295) and with --head_conv 256, where its outputs must coincide with DLASeg's."""
  rh.no_pretrained_download()
  img, pre, hm = wt.synthetic_inputs(1, *SMALL_HW)
  inv = {b: a for a, b in GENERIC_RENAME}
  def generic_name(n):
    for b, a in inv.items():
      if n.startswith(b):
        return a + n[len(b):]
    return n
  data = {}
  for tag, extra in (('hc64', []), ('hc256', ['--head_conv', '256'])):
    opt, model = rh.build_reference_model('coco_tracking', input_hw=SMALL_HW, extra=['--arch', 'generic'] + extra)
    sd = wt.make_state_dict(model.state_dict(), 317, rename=GENERIC_RENAME)
    model.load_state_dict(sd)
    acts, hooks = {}, []
    mods = dict(model.named_modules())
    for name in STAGES:
      hooks.append(mods[generic_name(name)].register_forward_hook(
          lambda m, i, o, name=name: acts.__setitem__(name, o.detach().clone())))
    with torch.no_grad():
      out = model(img, pre, hm)[-1]
    for h in hooks:
      h.remove()
    data.update({'%s.head.%s' % (tag, k): v.numpy() for k, v in out.items()})
    data.update({'%s.stage.%s' % (tag, k): v.numpy() for k, v in acts.items()})
    data[tag + '.keys'] = np.array(sorted(sd.keys()))
    data[tag + '.head_conv'] = np.array([opt.head_conv[h][0] for h in opt.heads])
    if tag == 'hc256':       # same graph, same tensors as DLASeg(34): the two reference modules must agree
      opt2, dla = rh.build_reference_model('coco_tracking', input_hw=SMALL_HW)
      dla.load_state_dict(wt.make_state_dict(dla.state_dict(), 317))
      with torch.no_grad():
        ref = dla(img, pre, hm)[-1]
      data['hc256.max_abs_diff_vs_dla_34'] = np.array([float((out[k] - ref[k]).abs().max()) for k in out])
  np.savez_compressed(os.path.join(OUT, 'net_generic_coco_tracking_64x96.npz'), **data)
  print('generic', {k: v.shape for k, v in data.items() if 'head.' in k}, data['hc256.max_abs_diff_vs_dla_34'])


E2E_CASES = [  # (file stem, cfg, (H, W), batch the frame is cut from, frame index, input seed)
    ('e2e_coco_tracking_512', 'coco_tracking', (512, 512), 1, 0, 317),
    ('e2e_coco_tracking_512_b32f0', 'coco_tracking', (512, 512), 32, 0, 4242),      # the shape bench.py runs:
    ('e2e_coco_tracking_512_b32f31', 'coco_tracking', (512, 512), 32, 31, 4242),    # first / last frame of 32
    ('e2e_mot_544x960', 'mot', (544, 960), 1, 0, 317),
    ('e2e_coco_pose_512', 'coco_pose', (512, 512), 1, 0, 317)]
E2E_STAGE_POS = 128


def e2e_frame(hw, batch, frame, seed):
  """The (img, pre, hm) of one frame of a `batch`-frame synthetic step (bench.py builds the same batch)."""
  img, pre, hm = wt.synthetic_inputs(batch, hw[0], hw[1], seed=seed)
  return img[frame:frame + 1].clone(), pre[frame:frame + 1].clone(), hm[frame:frame + 1].clone()


def gen_e2e():
  """Full-size frames through the reference model + _sigmoid_output + generic_decode: head values at random
  positions, the decoded top-K, and every STAGES tensor at E2E_STAGE_POS random positions (all channels)."""
  from model.decode import generic_decode
  models = {}
  for stem, cfg, hw, batch, frame, seed in E2E_CASES:
    if cfg not in models:
      opt, model = rh.build_reference_model(cfg, input_hw=hw)
      sd = wt.make_state_dict(model.state_dict(), 317)
      model.load_state_dict(sd)
      models[cfg] = (opt, model)
    opt, model = models[cfg]
    img, pre, hm = e2e_frame(hw, batch, frame, seed)
    acts, hooks = {}, []
    mods = dict(model.named_modules())
    for name in STAGES:
      hooks.append(mods[name].register_forward_hook(
          lambda m, i, o, name=name: acts.__setitem__(name, o.detach().clone())))
    with torch.no_grad():
      out = model(img, pre, hm)[-1]
      for h in hooks:
        h.remove()
      out['hm'] = out['hm'].sigmoid_()
      if 'hm_hp' in out:
        out['hm_hp'] = out['hm_hp'].sigmoid_()
      out['pre_inds'] = None
      dets = generic_decode({k: (v.clone() if v is not None else None) for k, v in out.items()}, K=100, opt=opt)
    oh, ow = hw[0] // 4, hw[1] // 4
    rng = np.random.RandomState(3)
    pos = rng.randint(0, oh * ow, size=512)
    data = {'pos': pos}
    for k, v in out.items():
      if v is not None:
        data['sample.' + k] = v.numpy().reshape(v.shape[1], -1)[:, pos]
    data.update({'det.' + k: v.numpy() for k, v in dets.items()})
    data['hm_max_per_class'] = out['hm'].numpy().reshape(out['hm'].shape[1], -1).max(1)
    for name, t in acts.items():
      n = t.shape[2] * t.shape[3]
      sp = np.random.RandomState(5).randint(0, n, size=min(E2E_STAGE_POS, n))
      data['stagepos.' + name] = sp
      data['stage.' + name] = t.numpy().reshape(t.shape[1], -1)[:, sp]
    np.savez_compressed(os.path.join(OUT, stem + '.npz'), **data)
    print('e2e', stem, len(data), 'arrays', 'top score %.4f .. %.4f' % (float(dets['scores'][0, 0]), float(dets['scores'][0, -1])))


FLIP_CASES = ['coco_pose', 'nuscenes_ddd']


def flip_inputs(hw=SMALL_HW):
  img, pre, hm = wt.synthetic_inputs(1, hw[0], hw[1], seed=77)
  cat = lambda t: torch.cat((t, t.flip(3)), 0).contiguous()
  return cat(img), cat(pre), cat(hm)


def gen_flip():
  """--flip_test (detector.py:225-226,285-286,311-332): the (frame, mirrored frame) pair through the reference
  model, its _sigmoid_output and _flip_output, then generic_decode of the merged maps."""
  from detector import Detector as RefDetector
  from dataset.dataset_factory import get_dataset
  from model.decode import generic_decode
  data = {}
  for cfg in FLIP_CASES:
    opt, model = rh.build_reference_model(cfg, input_hw=SMALL_HW, extra=['--flip_test'])
    model.load_state_dict(wt.make_state_dict(model.state_dict(), 317))
    det = object.__new__(RefDetector)
    det.opt = opt
    det.flip_idx = get_dataset(opt.dataset).flip_idx
    img, pre, hm = flip_inputs()
    with torch.no_grad():
      out = model(img, pre, hm)[-1]
      out = det._sigmoid_output(out)
      out = det._flip_output(out)
      out['pre_inds'] = None
      dets = generic_decode({k: (v.clone() if v is not None else None) for k, v in out.items()}, K=50, opt=opt)
    for k, v in out.items():
      if v is not None:
        data['%s.head.%s' % (cfg, k)] = v.numpy()
    for k, v in dets.items():
      data['%s.det.%s' % (cfg, k)] = v.numpy()
  np.savez_compressed(os.path.join(OUT, 'flip_cases.npz'), **data)
  print('flip', len(data), 'arrays')


def gen_decode():
  from model.decode import generic_decode
  data = {}
  for i, (kind, B, C, H, W, K, seed) in enumerate(DECODE_CASES):
    inp = decode_inputs(kind, B, C, H, W, seed)
    opt = rh.make_opt('coco_tracking')
    t = {k: torch.from_numpy(v.copy()) for k, v in inp.items()}
    t['pre_inds'] = None
    with torch.no_grad():
      dets = generic_decode(t, K=K, opt=opt)
    for k, v in dets.items():
      data['%d.%s' % (i, k)] = v.numpy()
  np.savez_compressed(os.path.join(OUT, 'decode_cases.npz'), **data)
  print('decode', len(data), 'arrays')


def gen_post_track():
  """3 synthetic frames through the reference's generic_post_process + Tracker (greedy)."""
  from utils.post_process import generic_post_process
  from utils.tracker import Tracker
  from utils.image import get_affine_transform
  from model.decode import generic_decode
  data = {}
  for ci, (cfg, kind, C, H, W) in enumerate([('coco_tracking', 'coco', 80, 128, 128),
                                             ('nuscenes_ddd', 'ddd', 10, 112, 200),
                                             ('coco_pose', 'pose', 1, 128, 128)]):
    opt = rh.make_opt(cfg, extra=['--track_thresh', '0.05', '--new_thresh', '0.05'])
    tracker = Tracker(opt)
    height, width = 480, 640
    c = np.array([width / 2., height / 2.], dtype=np.float32)
    s = max(height, width) * 1.0
    calib = np.array([[1200, 0, width / 2, 0], [0, 1200, height / 2, 0], [0, 0, 1, 0]], dtype=np.float32)
    base = decode_inputs(kind, 1, C, H, W, 100 + ci)
    for frame in range(3):
      inp = {k: v.copy() for k, v in base.items()}
      rng = np.random.RandomState(1000 + frame)
      inp['tracking'] = (rng.randn(*inp['tracking'].shape) * 0.5).astype(np.float32)
      if 'dep' in inp:
        inp['dep'] = (1. / (1. / (1 + np.exp(-inp['dep'] / 30 + 1)) + 1e-6) - 1.).astype(np.float32)
      t = {k: torch.from_numpy(v) for k, v in inp.items()}
      t['pre_inds'] = None
      with torch.no_grad():
        dets = generic_decode(t, K=100, opt=opt)
      dets = {k: v.numpy() for k, v in dets.items()}
      res = generic_post_process(opt, dets, [c], [s], H, W, opt.num_classes, [calib], height, width)[0]
      res = [r for r in res if r['score'] > opt.out_thresh]
      if frame == 0:
        tracker.init_track([])
      out = tracker.step(res)
      for key in out[0].keys():
        arr = np.array([np.asarray(o[key], dtype=np.float64) for o in out])
        data['%s.f%d.%s' % (cfg, frame, key)] = arr
      data['%s.f%d.n' % (cfg, frame)] = np.array([len(out), tracker.id_count])
  np.savez_compressed(os.path.join(OUT, 'post_track.npz'), **data)
  print('post_track', len(data), 'arrays')


TRACK_MODES = [  # (name, extra opts argv)
    ('greedy_age2', ['--max_age', '2']),
    ('hungarian', ['--hungarian']),
    ('hungarian_age2', ['--hungarian', '--max_age', '2']),
    ('public', ['--public_det']),
    ('public_hungarian_age2', ['--public_det', '--hungarian', '--max_age', '2'])]


def gen_track_modes():
  """Crowded seeded streams (synthetic.synthetic_track_stream) through the reference's Tracker in its other modes:
  --hungarian (sklearn's removed linear_assignment is stood in for by scipy's linear_sum_assignment, ref_harness),
  --public_det, --max_age coasting."""
  import copy
  from utils.tracker import Tracker
  data = {}
  for name, extra in TRACK_MODES:
    for seed in range(4):
      opt = rh.make_opt('coco_tracking', extra=['--track_thresh', '0.2', '--new_thresh', '0.3'] + extra)
      tracker = Tracker(opt)
      for f, (dets, pub) in enumerate(wt.synthetic_track_stream(seed)):
        dets = copy.deepcopy(dets)
        for d in dets:                              # the reference adds lists: ct + tracking must be array-like
          d['ct'] = np.asarray(d['ct']); d['tracking'] = np.asarray(d['tracking'])
        if f == 0:
          tracker.init_track([])
        out = tracker.step(dets, pub)
        rows = [[o['tracking_id'], o['age'], o['active'], o['class'], o['score']] + list(map(float, o['bbox']))
                for o in out]
        data['%s.s%d.f%d' % (name, seed, f)] = np.array(rows, np.float64).reshape(-1, 9)
        data['%s.s%d.f%d.n' % (name, seed, f)] = np.array([len(out), tracker.id_count])
  np.savez_compressed(os.path.join(OUT, 'track_modes.npz'), **data)
  print('track_modes', len(data), 'arrays')


HOST_CASES = [  # (name, extra opts argv, image (h, w), input_meta has calib)
    ('fix_res', ['--input_h', '128', '--input_w', '160'], (120, 200), False),
    ('fix_res_tall', ['--input_h', '160', '--input_w', '128'], (333, 210), True),
    ('keep_res', ['--keep_res'], (97, 131), False),
    ('fix_short', ['--fix_short', '96'], (150, 260), False),
    ('fix_short_tall', ['--fix_short', '64'], (300, 170), True)]


def host_case_inputs(i, hw):
  rng = np.random.RandomState(900 + i)
  image = rng.randint(0, 256, size=(hw[0], hw[1], 3)).astype(np.uint8)
  n = 6
  x0 = rng.uniform(-10, hw[1] * 0.8, n); y0 = rng.uniform(-10, hw[0] * 0.8, n)
  w = rng.uniform(0, hw[1] * 0.5, n); h = rng.uniform(0, hw[0] * 0.5, n)
  w[0] = 0.0                                              # degenerate box: skipped by the reference
  tracks = [{'score': float(sc), 'active': int(ac), 'bbox': [float(a), float(b), float(a + c), float(b + d)]}
            for sc, ac, a, b, c, d in zip(rng.uniform(0.1, 1.0, n), [1, 1, 0, 1, 1, 1], x0, y0, w, h)]
  tracks[3]['score'] = 0.05                               # below pre_thresh
  calib = np.array([[700., 0, hw[1] / 2., 40.], [0, 700., hw[0] / 2., 1.], [0, 0, 1, 0.01]], dtype=np.float32)
  return image, tracks, calib


OPT_CASES = [['tracking'], ['tracking', '--pre_hm', '--track_thresh', '0.4', '--pre_thresh', '0.5'],
             ['tracking', '--num_classes', '1', '--input_h', '544', '--input_w', '960', '--ltrb_amodal', '--pre_hm'],
             ['tracking,ddd', '--pre_hm', '--nuscenes_att', '--velocity', '--input_res', '640'],
             ['tracking,multi_pose', '--keep_res', '--K', '50', '--num_head_conv', '2'],
             ['ctdet', '--head_conv', '128', '--test_scales', '1', '--fix_short', '512', '--out_thresh', '0.2'],
             ['tracking', '--no_pre_img', '--zero_pre_hm', '--zero_tracking', '--max_age', '3', '--new_thresh', '0.6'],
             ['tracking,multi_pose', '--hm_hp_weight', '0', '--hp_weight', '0', '--pre_hm'],      # zero-weight heads are not built
             ['tracking,ddd', '--dep_weight', '0', '--flip_test', '--dla_node', 'conv']]
OPT_FIELDS = ['task', 'dataset', 'test_dataset', 'arch', 'heads', 'head_conv', 'num_classes', 'input_h', 'input_w',
              'output_h', 'output_w', 'input_res', 'output_res', 'down_ratio', 'pad', 'num_stacks', 'fix_res', 'fix_short',
              'tracking', 'pre_img', 'pre_hm', 'zero_pre_hm', 'zero_tracking', 'out_thresh', 'pre_thresh', 'new_thresh',
              'track_thresh', 'max_age', 'K', 'test_scales', 'head_kernel', 'prior_bias', 'ltrb', 'ltrb_amodal',
              'nuscenes_att', 'velocity', 'depth_scale', 'flip_test', 'public_det', 'hungarian', 'model_output_list', 'weights',
              'dla_node']


def gen_opts():
  """Derived option fields of the reference's opts().init() (opts.py:257-403) for a set of command lines."""
  import io, contextlib, json
  from opts import opts
  out = []
  for argv in OPT_CASES:
    old = sys.argv
    sys.argv = ['demo.py'] + argv + ['--gpus', '-1']
    try:
      with contextlib.redirect_stdout(io.StringIO()):
        opt = opts().init()
    finally:
      sys.argv = old
    rec = {}
    for k in OPT_FIELDS:
      v = getattr(opt, k)
      rec[k] = [[n, c] for n, c in v.items()] if isinstance(v, dict) else v      # dicts keep their insertion order
    out.append(rec)
  with open(os.path.join(OUT, 'opts_cases.json'), 'w') as f:
    json.dump({'cases': OPT_CASES, 'fields': out}, f, indent=1)
  print('opts', len(out), 'cases')
  # every flag of the reference's parser with its default (opts.py:11-254): the product parser must agree wherever it
  # defines the same flag
  defaults = {}
  for a in opts().parser._actions:
    if a.dest != 'help':
      defaults[a.dest] = a.default
  with open(os.path.join(OUT, 'opts_defaults.json'), 'w') as f:
    json.dump(defaults, f, indent=1, sort_keys=True)
  print('opts defaults', len(defaults), 'flags')


def gen_dataset_info():
  """The class attributes Detector.__init__ / opts read off the reference's dataset classes (detector.py:38-47,
  opts.py:329-341): generic_dataset.py:21-52 and datasets/*.py."""
  import json
  from dataset.dataset_factory import dataset_factory
  out = {}
  for name, cls in sorted(dataset_factory.items()):
    out[name] = {'default_resolution': list(cls.default_resolution), 'num_categories': None if cls.num_categories is None else int(cls.num_categories),
                 'rest_focal_length': float(cls.rest_focal_length), 'num_joints': int(cls.num_joints),
                 'flip_idx': [list(map(int, e)) for e in cls.flip_idx],
                 'mean': np.asarray(cls.mean, np.float64).ravel().tolist(),
                 'std': np.asarray(cls.std, np.float64).ravel().tolist()}
  json.dump(out, open(os.path.join(OUT, 'dataset_info.json'), 'w'), indent=1, sort_keys=True)
  print('dataset_info', sorted(out))


def gen_host():
  """Detector.pre_process / _get_additional_inputs of the reference (detector.py:175-290), model-free: the
  methods are called on an instance built without __init__ (no checkpoint, no device)."""
  from detector import Detector as RefDetector
  from dataset.dataset_factory import get_dataset
  data = {}
  for i, (name, extra, hw, with_calib) in enumerate(HOST_CASES):
    opt = rh.make_opt('coco_tracking', extra=['--pre_thresh', '0.3'] + extra)
    det = object.__new__(RefDetector)
    ds = get_dataset(opt.dataset)
    opt.device = torch.device('cpu')                        # set by Detector.__init__ in the reference
    det.opt = opt
    det.mean = np.array(ds.mean, dtype=np.float32).reshape(1, 1, 3)
    det.std = np.array(ds.std, dtype=np.float32).reshape(1, 1, 3)
    det.rest_focal_length = ds.rest_focal_length
    image, tracks, calib = host_case_inputs(i, hw)
    images, meta = det.pre_process(image, 1.0, {'calib': calib} if with_calib else {})
    data[name + '.images'] = images.numpy()
    for k in ('c', 's', 'calib', 'trans_input', 'trans_output'):
      data[name + '.meta.' + k] = np.asarray(meta[k], dtype=np.float64)
    data[name + '.meta.ints'] = np.array([meta[k] for k in ('height', 'width', 'out_height', 'out_width',
                                                             'inp_height', 'inp_width')], dtype=np.int64)
    hm, inds = det._get_additional_inputs(tracks, meta, with_hm=True)
    data[name + '.pre_hm'] = hm.numpy()
    data[name + '.pre_inds'] = inds.numpy()
  np.savez_compressed(os.path.join(OUT, 'host_pre.npz'), **data)
  print('host_pre', len(data), 'arrays')


DIGESTS = 'reference_digests.json'


def golden_digest(path):
  """sha256 of a fixture's content: the parsed JSON, or every array's name, dtype, shape and bytes of an .npz."""
  h = hashlib.sha256()
  if path.endswith('.json'):
    h.update(json.dumps(json.load(open(path)), sort_keys=True).encode())
    return h.hexdigest()
  with np.load(path) as z:
    for k in sorted(z.files):
      a = np.ascontiguousarray(z[k])
      h.update(('%s|%s|%s|' % (k, a.dtype.str, a.shape)).encode())
      h.update(a.tobytes())
  return h.hexdigest()


def write_digests(names):
  """Record what the reference produced in DIGESTS, so that the committed fixtures can be checked against this run
  where the reference is not at hand (tests/test_golden_fresh.py)."""
  path = os.path.join(OUT, DIGESTS)
  d = json.load(open(path)) if os.path.exists(path) else {}
  d.update({n: golden_digest(os.path.join(OUT, n)) for n in names})
  with open(path, 'w') as f:
    json.dump(d, f, indent=1, sort_keys=True)


if __name__ == '__main__':
  os.makedirs(OUT, exist_ok=True)
  t0 = time.time()
  torch.manual_seed(0)
  which = sys.argv[1:] or ['net', 'generic', 'e2e', 'decode', 'post', 'track', 'host', 'opts', 'flip']
  rh.install()
  if 'net' in which:
    gen_net()
  if 'generic' in which:
    gen_generic()
  if 'decode' in which:
    gen_decode()
  if 'post' in which:
    gen_post_track()
  if 'track' in which:
    gen_track_modes()
  if 'e2e' in which:
    gen_e2e()
  if 'host' in which:
    gen_host()
  if 'opts' in which:
    gen_opts()
    gen_dataset_info()
  if 'flip' in which:
    gen_flip()
  write_digests(sorted(n for n in os.listdir(OUT) if n != DIGESTS and os.path.getmtime(os.path.join(OUT, n)) >= t0))
