"""
INTEGRATION.md section 2 applied to the reference's own classes.  The repository does not carry the reference's
code: this runs where build() compiled it into oracle/_ref/ (oracle/build_ref.py) and skips elsewhere.  CPU only:
it checks that the re-bound methods/properties sit correctly on dragonfly.gp.gp_core.GP and that, with no GPU, the
first numeric call fails loudly instead of silently using NumPy.
"""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, 'oracle', '_ref')

SCRIPT = r'''
import sys, warnings
warnings.simplefilter('ignore')
sys.path.insert(0, %(shim)r); sys.path.insert(0, %(ref)r); sys.path.insert(0, %(root)r)
import sitecustomize
import numpy as np
import dragonfly.gp.gp_core as ref_core
import dragonfly.opt.gpb_acquisitions as ref_acq
from dragonfly.gp.kernel import SEKernel
from dragonfly_b200 import gp_core as b200_core, gpb_acquisitions as b200_acq
for name in b200_core.REBIND_METHODS:      # every method of the device-backed GP the re-bound class needs
  setattr(ref_core.GP, name, getattr(b200_core.GP, name))
for prop in ['L', 'alpha', 'K_trtr_wo_noise']:
  setattr(ref_core.GP, prop, getattr(b200_core.GP, prop))
for ns in ('asy', 'syn', 'seq'):
  for acq in ('ucb', 'ei', 'pi', 'ttei', 'ts', 'add_ucb'):
    setattr(getattr(ref_acq, ns), acq, getattr(getattr(b200_acq, ns), acq))
import dragonfly.opt.multiobjective_gpb_acquisitions as ref_moo
from dragonfly_b200 import multiobjective_gpb_acquisitions as b200_moo
for ns in ('asy', 'seq'):
  for acq in ('lin_ucb', 'tch_ucb', 'lin_ts', 'tch_ts'):
    assert hasattr(getattr(ref_moo, ns), acq)
    setattr(getattr(ref_moo, ns), acq, getattr(getattr(b200_moo, ns), acq))
assert ref_moo.asy.lin_ucb is b200_moo.mo_lin_asy_ucb and vars(ref_moo.syn) == vars(b200_moo.syn) == {}
X = np.random.rand(6, 2); Y = np.random.rand(6)
gp = ref_core.GP(X, Y, SEKernel(2, 1.0, [0.5, 0.5]), lambda x: np.zeros(len(x)), 0.1, build_posterior=False)
assert gp.L is None and gp.alpha is None and gp.num_tr_data == 6
assert gp._train_matrix().shape == (6, 2)
import torch
if not torch.cuda.is_available():
  try:
    gp.build_posterior()
    raise SystemExit('build_posterior did not fail without a GPU')
  except RuntimeError as e:
    assert 'no CPU fallback' in str(e)
assert ref_acq.asy.ei is b200_acq.asy_ei
print('REBIND_OK')
'''


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, 'dragonfly')),
                    reason='needs the reference package that build() compiles into oracle/_ref/ from its sources')
def test_rebinding_recipe_on_reference_classes():
  code = SCRIPT % dict(shim=os.path.join(ROOT, 'oracle', 'ref_shim'), ref=REF, root=ROOT)
  env = dict(os.environ, PYTHONDONTWRITEBYTECODE='1')
  out = subprocess.run([sys.executable, '-W', 'ignore', '-c', code], capture_output=True, text=True, env=env,
                       timeout=300)
  assert 'REBIND_OK' in out.stdout, out.stdout + out.stderr
