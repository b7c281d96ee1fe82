"""Kernel variants, tiles and stage counts follow from the layer shapes alone: the only environment variables the package
reads are the four that diagnose or time the code without changing what it computes."""
import glob
import os
import re

from conftest import ROOT

KEPT = {'CTB_DEBUG_SYNC', 'CTB_NO_GRAPH', 'CTB_PDL', 'CTB_DEC_DEBUG'}
READ = re.compile(r'''(?:getenv\(|environ\.get\(|environ\[)\s*["']([A-Za-z0-9_]+)["']''')


def test_package_reads_only_the_diagnostic_switches():
  pkg = os.path.join(ROOT, 'centertrack_b200')
  files = [f for ext in ('py', 'cu', 'cuh') for f in glob.glob(os.path.join(pkg, '**', '*.' + ext), recursive=True)]
  assert any(f.endswith('engine.py') for f in files) and any(f.endswith('conv_tc.cu') for f in files)
  names = set()
  for f in files:
    src = open(f).read()
    found = READ.findall(src)
    # every getenv / environ access must be a read of a literal name that the pattern above sees
    assert len(found) == len(re.findall(r'getenv\(|\benviron\b', src)), f
    names.update(found)
  assert names == KEPT
