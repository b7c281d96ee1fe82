"""Golden freshness: the committed tests/golden fixtures must be what the UNMODIFIED reference produces.

Every run of oracle/gen_golden.py on the reference records a sha256 of each fixture it wrote in
tests/golden/reference_digests.json; the committed fixtures must hash to exactly that (no checkout needed).  When
CT_REF_ROOT names a CenterTrack checkout, the generator is also re-run on it into a scratch directory and its output
compared with the committed fixtures (same keys, integers exact, floats to 1e-5 -- CPU conv summation order may change
with the thread count)."""
import json
import os
import subprocess
import sys

import numpy as np

from gen_golden import DIGESTS, golden_digest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('CT_REF_ROOT', '')


SHIM_RECORD = 'shim_reference_run.npz'       # made by tests/shim_driver.py from the reference's scripts


def test_committed_goldens_are_what_the_reference_produces(tmp_path, golden_dir):
  want = json.load(open(os.path.join(golden_dir, DIGESTS)))
  assert sorted(want) == sorted(set(os.listdir(golden_dir)) - {DIGESTS, SHIM_RECORD})
  for name in sorted(want):
    assert golden_digest(os.path.join(golden_dir, name)) == want[name], name + ' is not what the reference produced'
  if not (REF and os.path.isdir(os.path.join(REF, 'src', 'lib'))):
    return
  env = dict(os.environ, CT_GOLDEN_OUT=str(tmp_path))
  r = subprocess.run([sys.executable, os.path.join(ROOT, 'oracle', 'gen_golden.py'), 'net', 'generic', 'decode', 'post', 'track', 'host',
                      'opts', 'e2e', 'flip'], capture_output=True, text=True, timeout=1500, env=env)
  assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
  fresh = sorted(set(os.listdir(str(tmp_path))) - {DIGESTS})
  assert fresh, 'generator wrote nothing'
  for name in fresh:
    a_path, b_path = os.path.join(str(tmp_path), name), os.path.join(golden_dir, name)
    assert os.path.exists(b_path), 'committed fixture missing: ' + name
    if name.endswith('.json'):
      assert json.load(open(a_path)) == json.load(open(b_path)), name
      continue
    a, b = np.load(a_path), np.load(b_path)
    assert sorted(a.files) == sorted(b.files), name
    for k in a.files:
      x, y = a[k], b[k]
      assert x.shape == y.shape and x.dtype == y.dtype, (name, k)
      if x.dtype.kind in 'fc':
        scale = max(1.0, float(np.abs(y).max())) if y.size else 1.0
        if k.startswith('det.') or '.f' in k:      # decoded lists: a near-tie may swap two rows; compare as sets of rows
          assert np.allclose(np.sort(x.ravel()), np.sort(y.ravel()), rtol=0, atol=2e-4 * scale), (name, k)
        else:
          assert np.allclose(x, y, rtol=0, atol=1e-5 * scale), (name, k, float(np.abs(x - y).max()))
      else:
        assert np.array_equal(x, y), (name, k)
