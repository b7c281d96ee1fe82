"""Run in a SUBPROCESS by tests/test_shim.py (it rewires `sys.modules`): drives `centertrack_b200.shim.install()` the
way the REFERENCE's own `src/demo.py::demo(opt)` and `src/test.py::prefetch_test(opt)` do, in two modes.

  reference: runs those two scripts themselves, unmodified, from a CenterTrack checkout.  Everything but the device is
    the real thing: the reference's `opts`, `logger`, `utils.utils`, `utils.image`, `dataset.dataset_factory`,
    `torch.utils.data.DataLoader` worker calling `Detector.pre_process`, and the B200 package's `Detector.run` /
    `post_process` / `Tracker` / `model.model` / `model.decode` / DCN under the reference's names.  The per-frame
    results of the three runs (demo.py; test.py; test.py with --public_det --hungarian --load_results) are compared
    with tests/golden/shim_reference_run.npz, or written there with --write.
  replay: no checkout; the shim's stand-ins for the reference modules, driven call for call as the two scripts drive
    the detector (Detector(opt), run(frame) per frame; pre_process -> DataLoader collation of one item -> reset_tracking
    and pre_dets / cur_dets on the first frame -> run(batch)), must give the results recorded from the scripts.

CPU only: the one method that touches the GPU, `Detector.process`, is replaced by a stub that decodes seeded
synthetic maps with the oracle (exactly as tests/test_oracle_golden.py does), and the model constructor is skipped.

usage: python tests/shim_driver.py reference <reference root> <tmp dir> <record.npz> [--write]
       python tests/shim_driver.py replay <record.npz>
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'oracle'), os.path.join(ROOT, 'tests')):
  if p not in sys.path:
    sys.path.insert(0, p)

import numpy as np
import torch

DEMO_ARGS = ['tracking', '--gpus', '0', '--pre_hm', '--input_h', '128', '--input_w', '160', '--track_thresh', '0.05',
             '--new_thresh', '0.05', '--save_video', '--save_results', '--exp_id', 'shimtest']
TEST_ARGS = ['tracking', '--gpus', '0', '--pre_hm', '--track_thresh', '0.05', '--new_thresh', '0.05', '--exp_id',
             'shimtest', '--not_set_cuda_env']
PUBLIC_ARGS = ['--public_det', '--hungarian']


def stub_device_path():
  """Detector.process -> oracle decode of seeded maps (seed = 700 + call number); no model.  Returns the call log."""
  import ct_oracle as co
  from helpers import decode_inputs
  from centertrack_b200 import detector as D
  calls = []

  def fake_process(self, images, pre_images=None, pre_hms=None, pre_inds=None, return_time=False):
    calls.append((tuple(images.shape), pre_images is not None, pre_hms is not None))
    oh, ow = images.shape[2] // 4, images.shape[3] // 4
    maps = decode_inputs('coco', 1, 80, oh, ow, 700 + len(calls))
    dets = {k: v for k, v in co.generic_decode(maps, 100).items() if not k.startswith('_')}
    return ({}, dets, time.time()) if return_time else ({}, dets)

  def fake_device_model(opt):
    opt.device = torch.device('cpu')
    return None

  D.Detector.process = fake_process
  D.Detector._init_device_model = staticmethod(fake_device_model)
  torch.cuda.synchronize = lambda *a, **k: None
  return calls


def frames():
  """The three BGR frames of the one test video (written as PNG for the scripts: lossless)."""
  rng = np.random.RandomState(0)
  return [rng.randint(0, 255, (120, 160, 3)).astype(np.uint8) for _ in range(3)]


def public_dets():
  """--load_results file of the public-detection protocol: 12 detections on a grid in each of frames 1..3."""
  pts = [(20 + 40 * a, 20 + 40 * b) for a in range(4) for b in range(3)]
  return {str(i): [{'bbox': [x - 8., y - 8., x + 8., y + 8.], 'ct': [float(x), float(y)], 'score': 0.9, 'class': 1}
                   for x, y in pts] for i in (1, 2, 3)}


def record(runs):
  """{run: {frame id: [result dict]}} -> {'<run>.f<id>.<field>': float64 [n, width]}."""
  out = {}
  for run, res in runs.items():
    for fid, rows in res.items():
      fields = sorted(rows[0]) if rows else []
      assert all(sorted(r) == fields for r in rows), (run, fid)
      for f in fields:
        out['%s.f%d.%s' % (run, int(fid), f)] = np.array([np.asarray(r[f], np.float64).ravel() for r in rows])
      out['%s.f%d.n' % (run, int(fid))] = np.array([len(rows)], np.float64)
  return out


def check_or_write(rec, path, write=False):
  if write:
    np.savez_compressed(path, **rec)
    return
  g = np.load(path)
  assert sorted(rec) == sorted(g.files), sorted(set(rec) ^ set(g.files))
  for k in g.files:
    assert rec[k].shape == g[k].shape and np.allclose(rec[k], g[k], rtol=0, atol=1e-4), k


def replay(golden):
  import centertrack_b200.shim as shim
  from torch.utils.data import default_collate
  shim.install()
  calls = stub_device_path()
  from opts import opts
  from detector import Detector
  imgs = frames()
  det = Detector(opts().init(DEMO_ARGS))                             # demo.py: one detector, run() on every frame
  demo = {i + 1: det.run(img)['results'] for i, img in enumerate(imgs)}

  def prefetch(argv, loaded):                                        # test.py: prefetch_test on a 3-frame video
    opt = opts().init(argv + ['--input_h', '128', '--input_w', '160'])
    det = Detector(opt)
    out = {}
    for fid, img in enumerate(imgs, 1):
      images, meta = det.pre_process(img, 1, {'calib': det._get_default_calib(img.shape[1], img.shape[0])})
      item = {'images': {1: images}, 'image': img, 'meta': {1: meta}}
      if fid == 1:
        item.update(is_first_frame=1, video_id=1)
      _, batch = default_collate([(fid, item)])                      # the DataLoader's batch of one
      if 'is_first_frame' in batch:
        batch['meta']['pre_dets'] = loaded.get(str(fid), [])
        det.reset_tracking()
      if opt.public_det:
        batch['meta']['cur_dets'] = loaded.get(str(fid), [])
      out[fid] = det.run(batch)['results']
    return out

  private = prefetch(TEST_ARGS, {})
  public = prefetch(TEST_ARGS + PUBLIC_ARGS, json.loads(json.dumps(public_dets())))
  assert len(calls) == 9, calls
  check_or_write(record({'demo': demo, 'private': private, 'public': public}), golden)
  print('SHIM REPLAY OK: %d stubbed process() calls' % len(calls))


def main(ref_root, tmp, golden, write=False):
  import cv2
  import ref_harness as rh
  rh.install_third_party_stubs()                 # progress / pycocotools / ... are absent from this image

  import centertrack_b200.shim as shim
  aliases = shim.install()                       # BEFORE the reference's _init_paths puts src/lib on sys.path
  assert set(aliases) == {'detector', 'model.model', 'model.decode', 'utils.tracker', 'model.networks.DCNv2.dcn_v2'}

  # ---- the device path is stubbed (no GPU here) ------------------------------------------------
  from centertrack_b200 import detector as D
  calls = stub_device_path()

  # ---- the reference's scripts ------------------------------------------------------------------
  src = os.path.join(ref_root, 'src')
  os.makedirs(os.path.join(tmp, 'src'), exist_ok=True)
  os.makedirs(os.path.join(tmp, 'results'), exist_ok=True)
  os.chdir(os.path.join(tmp, 'src'))             # demo.py writes ../results/...
  sys.path.insert(0, src)
  import demo as ref_demo                         # runs `import _init_paths`, `from opts import opts`, `from detector import Detector`
  assert os.path.abspath(ref_demo.__file__).startswith(os.path.abspath(src))
  import detector, opts as ref_opts
  assert detector is D and ref_demo.Detector is D.Detector
  assert os.path.abspath(ref_opts.__file__).startswith(os.path.abspath(src)), 'opts must stay the reference\'s own'
  # the names round 1's shim shadowed stay importable from the reference
  from utils.utils import AverageMeter           # noqa: F401   (test.py:17)
  import utils.debugger, model.utils, logger     # noqa: F401,E401
  import utils.image as ref_image
  assert os.path.abspath(ref_image.__file__).startswith(os.path.abspath(src))
  import model.model as mm, model.decode as md, utils.tracker as ut
  from model.networks.DCNv2.dcn_v2 import DCN
  import centertrack_b200 as pkg
  assert mm is pkg.model and md is pkg.decode and ut is pkg.tracker and DCN is pkg.dcn.DCN

  # ---- demo.py on three written frames, with --save_video ------------------------------------------
  frames_dir = os.path.join(tmp, 'frames')
  os.makedirs(frames_dir, exist_ok=True)
  for i, img in enumerate(frames()):
    cv2.imwrite(os.path.join(frames_dir, '%03d.png' % i), img)
  written = []

  class FakeWriter(object):
    def __init__(self, *a, **k): pass
    def write(self, frame): written.append(frame)
    def release(self): pass

  ref_demo.cv2.imshow = lambda *a, **k: None
  ref_demo.cv2.waitKey = lambda *a, **k: 0
  ref_demo.cv2.VideoWriter = FakeWriter
  ref_demo.cv2.VideoWriter_fourcc = lambda *a: 0
  sys.argv = ['demo.py', '--demo', frames_dir] + DEMO_ARGS
  opt = ref_opts.opts().init()
  try:
    ref_demo.demo(opt)
    raise AssertionError('demo() must leave through save_and_exit -> sys.exit(0)')
  except SystemExit as e:
    assert e.code == 0
  assert len(calls) == 3 and all(c == ((1, 3, 128, 160), True, True) for c in calls), calls
  assert len(written) == 3 and all(f.shape == (120, 160, 3) and f.dtype == np.uint8 for f in written)
  import json
  res_files = [f for f in os.listdir(os.path.join(tmp, 'results')) if f.endswith('.json')]
  assert len(res_files) == 1, os.listdir(os.path.join(tmp, 'results'))
  saved = json.load(open(os.path.join(tmp, 'results', res_files[0])))
  assert sorted(saved) == ['1', '2', '3'] and all(len(v) > 0 and 'tracking_id' in v[0] for v in saved.values())
  n_demo = len(calls)

  # ---- test.py prefetch_test with a fake dataset --------------------------------------------------
  import test as ref_test
  assert os.path.abspath(ref_test.__file__).startswith(os.path.abspath(src))
  from dataset.dataset_factory import dataset_factory
  from dataset.generic_dataset import GenericDataset
  evaluated = {}

  class FakeCoco(object):
    def loadImgs(self, ids):
      return [{'file_name': '%03d.png' % (i - 1), 'frame_id': i, 'video_id': 1} for i in ids]

  class FakeDataset(GenericDataset):
    default_resolution = [128, 160]
    num_categories = 80
    class_name = ['c%d' % i for i in range(80)]

    def __init__(self, opt, split):
      self.images = [1, 2, 3]
      self.coco = FakeCoco()
      self.img_dir = frames_dir
      self.opt = opt

    def run_eval(self, results, save_dir):
      evaluated.update(results)

  dataset_factory['shimfake'] = FakeDataset
  sys.argv = ['test.py'] + TEST_ARGS + ['--test_dataset', 'shimfake']
  opt = ref_opts.opts().parse()
  opt.save_dir = os.path.join(tmp, 'exp')          # the reference checkout is read-only
  opt.debug_dir = os.path.join(tmp, 'exp', 'debug')
  logger.subprocess.check_output = lambda *a, **k: b'shimtest'   # Logger runs `git describe` in the cwd (logger.py:33)
  ref_test.opt = opt                                # PrefetchDataset.__getitem__ reads the module global (test.py:39)
  ref_test.prefetch_test(opt)
  assert sorted(evaluated) == [1, 2, 3], evaluated.keys()
  assert all(len(v) > 0 and {'bbox', 'score', 'class', 'tracking_id', 'ct', 'tracking'} <= set(v[0]) for v in evaluated.values())
  assert len(calls) == n_demo + 3
  ids = [sorted(r['tracking_id'] for r in evaluated[i]) for i in (1, 2, 3)]
  assert max(ids[2]) >= max(ids[0])                 # ids keep counting up through the video
  # ---- the same again in the MOT public-detection protocol: --public_det --hungarian --load_results ------------------
  # (test.py:64-70,90-108 -> meta['pre_dets'] / meta['cur_dets'] -> Tracker.init_track / Tracker.step(results, public_det))
  pub = public_dets()
  pub_path = os.path.join(tmp, 'public_dets.json')
  json.dump(pub, open(pub_path, 'w'))
  private = {k: list(v) for k, v in evaluated.items()}
  evaluated.clear()
  sys.argv = ['test.py'] + TEST_ARGS + PUBLIC_ARGS + ['--test_dataset', 'shimfake', '--load_results', pub_path]
  opt = ref_opts.opts().parse()
  opt.save_dir = os.path.join(tmp, 'exp')
  opt.debug_dir = os.path.join(tmp, 'exp', 'debug')
  ref_test.opt = opt
  n_before = len(calls)
  ref_test.prefetch_test(opt)
  assert sorted(evaluated) == [1, 2, 3] and len(calls) == n_before + 3
  seen = 12                                         # frame 1 starts from the 12 loaded pre_dets (ids 1..12)
  for i in (1, 2, 3):
    born = sorted(r['tracking_id'] for r in evaluated[i] if r['tracking_id'] > seen)
    assert len(born) <= 12, (i, born)               # a track may only start on a public detection
    assert born == list(range(seen + 1, seen + 1 + len(born)))
    seen += len(born)
  n_private = max(r['tracking_id'] for r in private[3])
  assert seen - 12 < n_private, (seen, n_private)    # far fewer births than the private protocol on the same frames
  check_or_write(record({'demo': saved, 'private': private, 'public': evaluated}), golden, write)
  print('SHIM OK: demo.py 3 frames (%d video frames written), test.py 3 frames, %d stubbed process() calls'
        % (len(written), len(calls)))


if __name__ == '__main__':
  if sys.argv[1] == 'replay':
    replay(sys.argv[2])
  else:
    main(sys.argv[2], sys.argv[3], sys.argv[4], write='--write' in sys.argv[5:])
