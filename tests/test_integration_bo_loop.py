"""
The drop-in inside the reference's OWN Bayesian-optimisation loop.  The repository does not carry the reference's
code: this runs where build() compiled it into oracle/_ref/ (oracle/build_ref.py) and skips elsewhere.

INTEGRATION.md section 2 is applied to the reference's classes (GP numerics re-bound, acquisition tables replaced)
and `dragonfly.maximise_function` (plus `maximise_multifidelity_function` and `multiobjective_maximise_functions`) -- GPBandit, the hyper-parameter fitter, ask/tell, the multi-armed choice of
acquisitions, hallucinations for pending points: all the reference's control plane, untouched -- is run twice under
the same seed: once unmodified, once re-bound.  There is no GPU here, so the ONE thing substituted below the host
mirror is DevicePosterior, by a NumPy stand-in that answers with the oracle's arithmetic (the CUDA path's parity
with that arithmetic is what the -m gpu tests establish).  Everything above it is the product's host code: kernel
descriptors, centring, jitter ladder, lazy L / alpha, incremental add_data, hallucinated extensions, candidate
generation and RNG consumption, acquisition descriptors, TTEI's reference arm and coin flips.

Pass criterion: the re-bound run queries EXACTLY the points the unmodified reference queries, evaluation by
evaluation, and returns the same optimum.
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
sys.path.insert(0, %(ref)r); sys.path.insert(0, %(root)r)
exec(open(%(shim)r + '/sitecustomize.py').read())     # NumPy-2 aliases the reference needs (np.math, ...)
import numpy as np
from dragonfly import maximise_function, maximise_multifidelity_function
from dragonfly.utils.option_handler import load_options
from dragonfly.opt.gp_bandit import get_all_euc_gp_bandit_args
import dragonfly.gp.gp_core as ref_core
import dragonfly.opt.gpb_acquisitions as ref_acq
from oracle import gp_oracle as O


def objective(x):
  x = np.asarray(x)
  return float(-((x[0] - 0.3) ** 2 + (x[1] - 0.7) ** 2) + 0.1 * np.sin(8 * x[0]) + 0.05 * x[2])


CONFIGS = {
  'rand_ucb_ei_ttei_pi': dict(acq_opt_method='rand', acq='ucb-ei-ttei-pi', capital=16),
  'rand_ts_ucb': dict(acq_opt_method='rand', acq='ts-ucb', capital=12),
  # the reference's DEFAULT hyper-parameter tuning ('ml-post_sampling': marginal likelihood + slice sampling of
  # the posterior over hps, gp_bandit.py) and default acquisition portfolio
  'default_hp_tuning': dict(acq_opt_method='rand', acq='default', capital=10, default_hp_tune=True),
  'pdoo_ei_ucb': dict(acq_opt_method='pdoo', acq='ei-ucb', capital=11),
  # three workers: pending evaluations are hallucinated (gp_bandit.py:45, gpb_acquisitions.py:43-64) -- in the
  # re-bound run through the temporary in-place extension of the posterior
  'rand_3_workers': dict(acq_opt_method='rand', acq='ucb-ei', capital=14, num_workers=3),
  # additive GP + Add-UCB (gpb_acquisitions.py:139-189): per-group test kernels against the full model's L, alpha
  'additive_add_ucb': dict(acq_opt_method='rand', acq='add_ucb-ucb', capital=11),
  # multi-fidelity: EuclideanMFGP (product kernel on [z || x] rows) + BOCA (gpb_acquisitions.py:399-439)
  'mf_boca': dict(acq='ucb-ei', capital=9, mf=True),
  # two objectives, MOORS scalarisations (multiobjective_gpb_acquisitions.py:19-107)
  'moo_ucb_ts': dict(acq='ucb-ts', capital=11, moo=True),
}


def mf_objective(z, x):
  z, x = np.asarray(z), np.asarray(x)
  return objective(x) - 0.3 * (1.0 - z[0]) ** 2 * (1 + np.sin(5 * x[1]))


def run_mf(cfg):
  from dragonfly.opt.gp_bandit import get_all_mf_euc_gp_bandit_args
  opts = load_options(get_all_mf_euc_gp_bandit_args())
  opts.acq_opt_method = 'rand'
  opts.acq = cfg['acq']
  opts.gpb_hp_tune_criterion = 'ml'
  opts.gpb_ml_hp_tune_opt = 'rand'
  opts.build_new_model_every = 4
  np.random.seed(3)
  val, pt, hist = maximise_multifidelity_function(
      mf_objective, [[0, 1]], [[0, 1], [0, 1], [0, 2]], [1.0], lambda z: 0.2 + 0.8 * np.asarray(z)[0],
      cfg['capital'], options=opts)
  return val, np.asarray(pt), np.array([np.concatenate((np.ravel(f), np.ravel(p))) for f, p in
                                        zip(hist.query_fidels, hist.query_points)]), np.array(hist.query_vals)


def run_moo(cfg):
  from dragonfly import multiobjective_maximise_functions
  from dragonfly.opt.multiobjective_gp_bandit import get_all_euc_moo_gp_bandit_args
  opts = load_options(get_all_euc_moo_gp_bandit_args())
  opts.acq_opt_method = 'rand'
  opts.acq = cfg['acq']
  opts.gpb_hp_tune_criterion = 'ml'
  opts.gpb_ml_hp_tune_opt = 'rand'
  opts.build_new_model_every = 4
  np.random.seed(3)
  funcs = [objective, lambda x: float(-np.sum((np.asarray(x) - 0.6) ** 2))]
  pareto_vals, pareto_pts, hist = multiobjective_maximise_functions(funcs, [[0, 1], [0, 1], [0, 2]],
                                                                    cfg['capital'], options=opts)
  return (np.array(pareto_vals).sum(), np.array(pareto_pts).ravel(), np.array(hist.query_points),
          np.array(hist.query_vals))


def run(cfg):
  if cfg.get('mf'):
    return run_mf(cfg)
  if cfg.get('moo'):
    return run_moo(cfg)
  opts = load_options(get_all_euc_gp_bandit_args())
  opts.acq_opt_method = cfg['acq_opt_method']
  opts.acq = cfg['acq']
  if not cfg.get('default_hp_tune'):
    opts.gpb_hp_tune_criterion = 'ml'
    opts.gpb_ml_hp_tune_opt = 'rand'
  opts.build_new_model_every = 4
  np.random.seed(3)
  val, pt, hist = maximise_function(objective, [[0, 1], [0, 1], [0, 2]], cfg['capital'], options=opts,
                                    num_workers=cfg.get('num_workers', 1))
  return val, np.asarray(pt), np.array(hist.query_points), np.array(hist.query_vals)

reference_runs = dict((name, run(cfg)) for name, cfg in CONFIGS.items())

# ---- re-bind (INTEGRATION.md 2a, 2b) --------------------------------------------------------------------------
from dragonfly_b200 import gp_core as b200_core, gpb_acquisitions as b200_acq, device as b200_device, _lib
for name in b200_core.REBIND_METHODS:      # every method of the device-backed GP the re-bound class needs
  setattr(ref_core.GP, name, getattr(b200_core.GP, name))
for prop in ['L', 'alpha', 'K_trtr_wo_noise']:
  setattr(ref_core.GP, prop, getattr(b200_core.GP, prop))
for ns in ('asy', 'syn', 'seq'):
  for acq in ('ucb', 'ei', 'pi', 'ttei', 'ts', 'add_ucb'):
    setattr(getattr(ref_acq, ns), acq, getattr(getattr(b200_acq, ns), acq))
# multi-fidelity (INTEGRATION.md 2c): BOCA and the [z || x] packing it needs on the reference's MF class
import dragonfly.gp.euclidean_gp as ref_egp
from dragonfly_b200 import mf_gp as b200_mf
ref_acq.boca = b200_acq.boca
import dragonfly.opt.multiobjective_gpb_acquisitions as ref_moo
from dragonfly_b200 import multiobjective_gpb_acquisitions as b200_moo
for ns in ('asy', 'seq'):
  for acq in ('lin_ucb', 'tch_ucb', 'lin_ts', 'tch_ts'):
    setattr(getattr(ref_moo, ns), acq, getattr(getattr(b200_moo, ns), acq))
ref_egp.EuclideanMFGP.get_ZX_matrix = b200_mf.EuclideanMFGP.get_ZX_matrix

# ---- the stand-in for the device: the oracle's arithmetic behind DevicePosterior's interface -----------------------
calls = dict(build=0, extend=0, restore=0, score=0, eval=0)


def numpy_kernel(kern):
  """ Kernel objects of the host mirror (hp_grid's layout builds those) evaluate on the device; the stand-in needs
      the same kernel as a NumPy object: the reference's own class with the same hyper-parameters. """
  import dragonfly.gp.kernel as ref_kernel
  if not type(kern).__module__.startswith('dragonfly_b200'):
    return kern
  hp = kern.hyperparams
  if type(kern).__name__ == 'SEKernel':
    return ref_kernel.SEKernel(kern.dim, hp['scale'], hp['dim_bandwidths'])
  if type(kern).__name__ == 'MaternKernel':
    return ref_kernel.MaternKernel(kern.dim, hp['nu'], hp['scale'], hp['dim_bandwidths'])
  if type(kern).__name__ == 'AdditiveKernel':
    return ref_kernel.AdditiveKernel(hp['scale'], [numpy_kernel(k) for k in kern.kernel_list], kern.groupings)
  if type(kern).__name__ == 'CoordinateProductKernel':
    return ref_kernel.CoordinateProductKernel(kern.dim, hp['scale'], [numpy_kernel(k) for k in kern.kernel_list],
                                              kern.coordinate_list)
  raise NotImplementedError(type(kern).__name__)


class NumpyDevice(object):
  TS_BLOCK = 4096

  def __init__(self, n_max, device=None, chunk=0):
    import torch
    self.n, self.dim, self.saved, self.n_max = 0, 0, None, n_max
    self.device = torch.device('cpu')

  def query(self, name):
    return {'chunk': 6528.0}[name]

  def bind_current_stream(self):
    pass

  def moo_score_argmax(self, kind, a_list, b_list, weights, refs=None, beta=0.0, want_scores=False):
    calls['moo'] = calls.get('moo', 0) + 1
    a = [np.asarray(v, dtype=np.float64) for v in a_list]
    b = None if b_list is None else [np.asarray(v, dtype=np.float64) for v in b_list]
    if kind == _lib.DFB_MOO_LIN_UCB:
      sc = O.moo_lin_ucb(a, b, weights, beta)
    elif kind == _lib.DFB_MOO_TCH_UCB:
      sc = O.moo_tch_ucb(a, b, weights, refs, beta)
    elif kind == _lib.DFB_MOO_LIN_VAL:
      sc = O.moo_lin_vals(a, weights)
    else:
      sc = O.moo_tch_vals(a, weights, refs)
    i = O.np_argmax_first(sc)
    return float(sc[i]), i, sc

  def set_kernel(self, kern):            # build_descriptor is patched to pass Dragonfly's own kernel object through
    self.kern = numpy_kernel(kern)

  def set_train(self, X, yc):
    self.X, self.yc = np.array(X, dtype=np.float64), np.array(yc, dtype=np.float64)
    self.n, self.dim = self.X.shape

  def capacity(self):
    return (self.n + 127) // 128 * 128

  def max_diag(self):
    return float(np.diag(self.kern(self.X, self.X)).max() + self.noise)

  def _factor(self):
    K = self.kern(self.X, self.X) + self.noise * np.eye(self.n)
    try:
      self.L = np.linalg.cholesky(K)
    except np.linalg.LinAlgError:
      return 1, None
    self.alpha = O.solve_upper_triangular(self.L.T, O.solve_lower_triangular(self.L, self.yc))
    return 0, -0.5 * self.yc.dot(self.alpha) - np.log(np.diag(self.L)).sum() - 0.5 * self.n * np.log(2 * np.pi)

  def build(self, noise_var, jitter=0.0, flags=0):
    calls['build'] += 1
    self.noise = noise_var + jitter
    return self._factor()

  def extend(self, X_new, yc_new, flags=0, save=False):
    calls['extend'] += 1
    if save:
      self.saved = (self.X, self.yc, self.L, self.alpha, self.n)
    self.X = np.concatenate((self.X, np.asarray(X_new, dtype=np.float64)), axis=0)
    self.yc = np.concatenate((self.yc, np.asarray(yc_new, dtype=np.float64)))
    self.n = len(self.X)
    info, lml = self._factor()
    if save and info == 0:
      self.alpha = np.concatenate((self.saved[3], np.zeros(len(X_new))))
    if info != 0 and save:
      self.X, self.yc, self.L, self.alpha, self.n = self.saved
    return info, lml

  def restore(self, n_before):
    calls['restore'] += 1
    self.X, self.yc, self.L, self.alpha, self.n = self.saved
    self.saved = None

  def set_alpha(self, alpha):
    a = np.zeros(self.n); a[:len(alpha)] = alpha
    self.alpha = a

  def get_state(self, want_L=False, want_alpha=False, want_K=False):
    import torch
    t = lambda a: torch.from_numpy(np.array(a))
    return (t(self.L) if want_L else None, t(self.alpha) if want_alpha else None,
            t(self.kern(self.X, self.X)) if want_K else None)

  def _mu_sd(self, Xc, mean_const):
    """ gp_core.py:165-190 as the reference evaluates it: full covariance, then the diagonal.  With a test kernel
        set (Add-UCB, gpb_acquisitions.py:160-176): K_*j = scale k_j(X*_j, X[:, g_j]) against the full L, alpha. """
    Xc = np.asarray(Xc, dtype=np.float64)
    test = getattr(self, 'test', None)
    if test is None:
      Ks, Kcc = self.kern(Xc, self.X), self.kern(Xc, Xc)
    else:
      single, kw = test
      calls['group_score'] = calls.get('group_score', 0) + 1
      scale, k_j = single.hyperparams['scale'], single.kernel_list[0]
      Ks, Kcc = scale * k_j(Xc, self.X[:, kw['train_coords']]), scale * k_j(Xc, Xc)
    mu = mean_const + Ks.dot(self.alpha)
    V = O.solve_lower_triangular(self.L, Ks.T)
    covar = Kcc - V.T.dot(V)
    return mu, np.sqrt(np.diag(covar))

  def eval(self, Xc, mean_const=0.0, want_std=True):
    calls['eval'] += 1
    Xc = np.asarray(Xc, dtype=np.float64)
    if len(Xc) <= 16:
      # like the device's row-streaming path, a point's result must not depend on its batch-mates (NumPy's BLAS
      # kernels round differently for different shapes): one point at a time
      parts = [self._mu_sd(Xc[i:i + 1], mean_const) for i in range(len(Xc))]
      mu, sd = np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
    else:
      mu, sd = self._mu_sd(Xc, mean_const)
    return mu, (sd if want_std else None)

  def score_argmax(self, acq, Xc, mean_const=0.0, want_scores=False):
    calls['score'] += 1
    mu, sd = self._mu_sd(Xc, mean_const)
    if acq.kind == _lib.DFB_ACQ_UCB:
      sc = O.acq_ucb(mu, sd, acq.beta)
    elif acq.kind == _lib.DFB_ACQ_EI:
      sc = O.acq_ei(mu, sd, acq.best)
    elif acq.kind == _lib.DFB_ACQ_PI:
      sc = O.acq_pi(mu, sd, acq.best)
    elif acq.kind == _lib.DFB_ACQ_TTEI:
      sc = O.acq_ttei(mu, sd, acq.ref_mean, acq.ref_std)
    else:
      sc = mu
    i = O.np_argmax_first(sc)
    return float(sc[i]), i, (sc if want_scores else None)

  def set_test_kernel(self, desc):
    self.test = desc

  def ts_draws(self, Xc, Ut, mean_const=0.0, jitter=0.0):
    """ One attempt of draw_gaussian_samples (general_utils.py:224-232) on the posterior of gp_core.py:165-187. """
    import torch
    calls['ts'] = calls.get('ts', 0) + 1
    Xc = np.asarray(Xc, dtype=np.float64)
    Ks = self.kern(Xc, self.X)
    mu = mean_const + Ks.dot(self.alpha)
    V = O.solve_lower_triangular(self.L, Ks.T)
    covar = self.kern(Xc, Xc) - V.T.dot(V)
    try:
      Lp = np.linalg.cholesky(covar + jitter * np.eye(len(Xc)))
    except np.linalg.LinAlgError:
      return 1, None, float(np.diag(covar).max())
    U = np.asarray(Ut, dtype=np.float64).T                      # (m, S)
    return 0, torch.from_numpy(Lp.dot(U).T + mu), float(np.diag(covar).max())


b200_device.DevicePosterior = NumpyDevice
b200_core.build_descriptor = lambda kern, **kw: (kern, kw) if kw.get('train_coords') is not None else kern
for name, cfg in CONFIGS.items():
  ref_val, ref_pt, ref_q, ref_v = reference_runs[name]
  new_val, new_pt, new_q, new_v = run(cfg)
  assert new_q.shape == ref_q.shape, (name, new_q.shape, ref_q.shape)
  assert (new_q == ref_q).all(), (name, np.abs(new_q - ref_q).max())
  assert (new_v == ref_v).all() and new_val == ref_val and (new_pt == ref_pt).all(), name
  print('same trajectory:', name, len(ref_q), 'queries')
assert calls['build'] > 0 and calls['score'] > 0 and calls['extend'] > 0 and calls.get('ts', 0) > 0, calls
assert calls.get('moo', 0) > 0, calls             # the multi-objective scalarisations ran
assert calls.get('group_score', 0) > 0, calls     # Add-UCB's per-group test kernels were scored
assert calls['restore'] > 0, calls        # hallucinated (N + q)-point posteriors were extensions, undone afterwards

# ---- phase 2: the hyper-parameter fitter's fit_gp re-bound as well (INTEGRATION.md 2e): every batch of marginal
# likelihoods is one hp_grid.lml_for_hyperparams call (concurrent lanes; threads here, CUDA streams stubbed) --------
import contextlib
import torch
from dragonfly_b200 import hp_grid
batches = []
real_lmls = hp_grid.lml_for_hyperparams


def counting_lmls(X, Y, hps, layout, **kw):
  batches.append(len(hps))
  return real_lmls(X, Y, hps, layout, **kw)


class FakeStream(object):
  def __init__(self, *a, **k):
    pass

  def wait_stream(self, other):
    pass
torch.cuda.current_stream = lambda *a, **k: FakeStream()
torch.cuda.Stream = FakeStream
torch.cuda.device = lambda *a, **k: contextlib.nullcontext()
torch.cuda.stream = lambda *a, **k: contextlib.nullcontext()
hp_grid.lml_for_hyperparams = counting_lmls
hp_grid.build_descriptor = lambda kern, **kw: kern
hp_grid.bind_fit_gp(ref_core.GPFitter)
for name in ['rand_ucb_ei_ttei_pi', 'default_hp_tuning', 'additive_add_ucb', 'mf_boca']:
  ref_val, ref_pt, ref_q, ref_v = reference_runs[name]
  del batches[:]
  new_val, new_pt, new_q, new_v = run(CONFIGS[name])
  assert new_q.shape == ref_q.shape and (new_q == ref_q).all(), (name, 'fit_gp re-bound')
  assert (new_v == ref_v).all() and new_val == ref_val, name
  assert len(batches) > 0, name              # (the MF fitter goes through EuclideanMFHPLayout)
  if True:
    if name == 'default_hp_tuning':          # ml_hp_tune_opt 'default' -> 'direct' -> PDOO: a round of all passes per batch
      assert 2 < max(batches) <= 32 and len(batches) > 20, (name, len(batches), max(batches))
    else:                                    # 'rand': all candidates of a discrete setting in one batch
      assert max(batches) >= 100, (name, batches[:5])
  print('same trajectory with fit_gp re-bound:', name, 'batches', len(batches), 'largest', max(batches or [0]))
print('BO_LOOP_OK', calls)
'''


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, 'dragonfly')),
                    reason='needs the reference package that build() compiles into oracle/_ref/ from its sources')
def test_rebound_bo_loop_queries_exactly_what_the_reference_queries():
  code = SCRIPT % dict(shim=os.path.join(ROOT, 'oracle', 'ref_shim'), ref=REF, root=ROOT)
  # single-threaded BLAS: both runs must see bit-identical NumPy reductions (and tiny matrices gain nothing from threads)
  env = dict(os.environ, PYTHONDONTWRITEBYTECODE='1', OMP_NUM_THREADS='1', OPENBLAS_NUM_THREADS='1',
             MKL_NUM_THREADS='1')
  out = subprocess.run([sys.executable, '-W', 'ignore', '-c', code], capture_output=True, text=True, env=env,
                       timeout=1500)
  assert 'BO_LOOP_OK' in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
