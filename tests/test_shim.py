"""Drop-in boundary (SURVEY 8b): `centertrack_b200.shim.install()` under the reference's own scripts.  CPU only."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('CT_REF_ROOT', '')


def test_reference_demo_and_test_scripts_run_unchanged_through_the_shim(tmp_path):
  """The reference's UNMODIFIED src/demo.py::demo(opt) (3 written frames, --save_video --save_results) and
  src/test.py::prefetch_test(opt) (fake dataset, real DataLoader worker calling Detector.pre_process; also with
  --public_det --hungarian --load_results) with the shim installed give the per-frame results recorded from them in
  tests/golden/shim_reference_run.npz.  Without a checkout the shim is driven the way those scripts drive it and must
  reproduce that record; when CT_REF_ROOT names one, the scripts themselves run too, see tests/shim_driver.py for what
  is asserted (which modules stay the reference's, which are replaced, ret['generic'] frames, saved results, tracking
  ids).  Runs in subprocesses because the shim rewires sys.modules."""
  driver = os.path.join(ROOT, 'tests', 'shim_driver.py')
  record = os.path.join(ROOT, 'tests', 'golden', 'shim_reference_run.npz')
  r = subprocess.run([sys.executable, driver, 'replay', record], capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
  assert r.returncode == 0 and 'SHIM REPLAY OK' in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
  if not (REF and os.path.isdir(os.path.join(REF, 'src', 'lib'))):
    return
  r = subprocess.run([sys.executable, driver, 'reference', REF, str(tmp_path), record], capture_output=True, text=True,
                     timeout=600)
  assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
  assert 'SHIM OK' in r.stdout


def test_shim_standalone_fallbacks_without_the_reference():
  """Without the reference on sys.path the replaced names still resolve, and the host-side mirrors stand in for
  `opts`, `utils.image`, `utils.post_process`, `dataset.dataset_factory`."""
  code = r'''
import sys
sys.path.insert(0, %r)
import centertrack_b200.shim as shim
shim.install()
from opts import opts
from detector import Detector
from model.model import create_model, load_model, save_model
from model.decode import generic_decode
from utils.tracker import Tracker
from utils.image import get_affine_transform, draw_umich_gaussian
from utils.post_process import generic_post_process
from dataset.dataset_factory import dataset_factory, get_dataset
from model.networks.DCNv2.dcn_v2 import DCN
import centertrack_b200 as pkg
assert Detector is pkg.detector.Detector and DCN is pkg.dcn.DCN and opts is pkg.opts.opts
opt = opts().init(['tracking', '--pre_hm'])
assert list(opt.heads) == ['hm', 'reg', 'wh', 'tracking']
try:
  import utils.utils
  raise SystemExit('utils.utils must not exist without the reference')
except ImportError:
  pass
shim.uninstall()
assert not [f for f in sys.meta_path if type(f).__name__ == 'B200Finder']
print('STANDALONE OK')
''' % ROOT
  r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=300, cwd='/tmp')
  assert r.returncode == 0 and 'STANDALONE OK' in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
