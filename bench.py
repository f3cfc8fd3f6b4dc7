"""
bench.py -- the headline metric of BASELINE.json: posterior + acquisition candidates / second at
N = 5000 training points, fp64 (SURVEY.md 8d "headline": Hartmann-6, Matern-2.5, EI).

One "step" = one BO inner-loop iteration over one batch of synthetic candidates:
    GP.build_posterior (K, Cholesky, L^-1, alpha, LML)  +  K_* rows + mu  +  |L^-1 k_*|^2 -> sigma
    +  EI  +  running arg-max                         for M candidates per GPU.
  value : candidates / s with the candidate matrix already resident in HBM (device tensor).
  e2e   : the same step through the reference-facing operator `gpb_acquisitions.asy.ei(gp, anc_data)` on a GP built
          from HOST training data: candidates drawn from NumPy's global MT19937 stream exactly as the reference's
          random_maximise does (oper_utils.py:59-80), uploaded, scored; the arg-max point comes back.
Multi-GPU (torchrun, one rank per GPU): every rank builds the (tiny, replicated) posterior and scores its own M
candidates -- weak scaling, no data-path collective; the single collective is the (score, index[, point]) all-gather
of the final arg-max (dragonfly_b200/dist.py).

`--config c2|c3|c4|c5` runs BASELINE.json's other configurations through the public operators (asy.ucb, asy.add_ucb,
the BOCA step-1 slice, GP.draw_samples_argmax) with the GLOBAL candidate count of the config fixed and sharded over
the ranks by the operators themselves ("scaling": "strong").

`--impl reference` times the CPU restatement of the reference algorithm (oracle/gp_oracle.py, the faithful chunked
gp.eval(.., 'std') driver of SURVEY 8d) on the host cores, rank 0 only.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step of each leg handed its caller as
DIR/<name>.npy (float64, rank 0): the arg-max (score, index or point) of every leg and, of the `value` leg's
posterior, the log marginal likelihood, alpha and a fixed sample of L.  The inputs are seeded, so two builds run
with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

METRIC = 'posterior+acq candidates/sec at N=5000 fp64'
UNIT = 'candidates/s'
CPU_CHUNK = 2000          # SURVEY 8d: the reference's eval('std') builds chunk x chunk covariances

CONFIGS = {
  # name: (synth_data workload, default global candidates, description)
  'headline': ('headline_hartmann6_matern_ei', None,
               'headline: Hartmann-6 (d=6) Matern-2.5, N=%d train, EI over %d candidates per GPU '
               '(BASELINE.json metric N=5000; configs[1] geometry at the metric\'s N)'),
  'c2': ('c2_hartmann6_matern_ucb', 1000000, 'configs[1]: Hartmann-6 Matern-2.5, N=%d, UCB over %d candidates'),
  'c3': ('c3_additive40_add_ucb', 4000000, 'configs[2]: 40-D additive GP (7 groups) add_ucb, N=%d, %d candidates in total'),
  'c4': ('c4_borehole_mf_ucb', 1000000, 'configs[3]: Borehole MF-GP (SE x SE product kernel) UCB on the fidel_to_opt slice, N=%d, %d candidates'),
  'c5': ('c5_park1_20_ts', 1000000, 'configs[4]: Park1-20 Thompson sampling, 256 joint posterior draws x %d candidates (N=%d)'),
}


def parse_args():
  p = argparse.ArgumentParser()
  p.add_argument('--gpus', type=int, default=1)
  p.add_argument('--steps', type=int, default=5)
  p.add_argument('--warmup', type=int, default=3)
  p.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  p.add_argument('--config', default='headline', choices=sorted(CONFIGS))
  p.add_argument('--n-train', type=int, default=0, help='0 = the configuration\'s own N')
  p.add_argument('--cands-per-gpu', type=int, default=1000000, help='headline: candidates per GPU (weak scaling)')
  p.add_argument('--global-cands', type=int, default=0, help='c2..c5: total candidates (0 = the configuration\'s own)')
  p.add_argument('--cpu-sample', type=int, default=24000)
  p.add_argument('--no-cpu-baseline', action='store_true')
  p.add_argument('--no-extras', action='store_true', help='skip the fp64-only / K_* / update side measurements')
  p.add_argument('--dump-outputs', metavar='DIR', default=None,
                 help='write the outputs of the last timed step of every leg to DIR/<name>.npy')
  args = p.parse_args()
  if args.steps < 1:
    p.error('--steps must be at least 1')
  return args


def dist_env():
  rank = int(os.environ.get('RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  return rank, world, local


def n_train_of(args):
  if args.n_train > 0:
    return args.n_train
  return {'headline': 5000, 'c2': 2000, 'c3': 5000, 'c4': 4000, 'c5': 5000}[args.config]


# ---------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port of the reference algorithm)
# ---------------------------------------------------------------------------------------------------
def use_all_host_threads():
  """ torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm is meant to run on all the host
      cores, so lift the BLAS / OpenMP pools back to the core count (threadpoolctl works after import). """
  try:
    from threadpoolctl import threadpool_limits
    threadpool_limits(limits=os.cpu_count())
  except Exception:  # pylint: disable=broad-except
    pass


def cpu_threads():
  try:
    from threadpoolctl import threadpool_info
    infos = [i for i in threadpool_info() if i.get('user_api') == 'blas']
    if infos:
      return max(i['num_threads'] for i in infos)
  except Exception:  # pylint: disable=broad-except
    pass
  return os.cpu_count()


def oracle_kernel(O, spec):
  t = spec['type']
  if t == 'se':
    return O.OSEKernel(spec['dim'], spec['scale'], spec['dim_bandwidths'])
  if t == 'matern':
    return O.OMaternKernel(spec['dim'], spec['nu'], spec['scale'], spec['dim_bandwidths'])
  if t == 'additive':
    return O.OAdditiveKernel(spec['scale'], [oracle_kernel(O, k) for k in spec['kernels']], spec['groupings'])
  if t == 'coordinate_product':
    return O.OCoordinateProductKernel(spec['dim'], spec['scale'], [oracle_kernel(O, k) for k in spec['kernels']],
                                      spec['coordinate_list'])
  raise ValueError(t)


class CpuArm(object):
  """ One configuration on the host cores through the oracle's faithful restatement: build() = GP(...) as
      gp_core.py:155-163, score(sample) = the reference's chunked eval + acquisition + arg-max. """

  def __init__(self, config, n_train, sample):
    from dragonfly_b200 import synth_data
    from oracle import gp_oracle as O
    self.O, self.config, self.sample = O, config, int(sample)
    self.w = synth_data.make_workload(CONFIGS[config][0], n_train=n_train, n_cand=max(self.sample, 16))
    self.kern = oracle_kernel(O, self.w['kernel'])
    self.gp = None

  def build(self):
    w, mc = self.w, self.w['mean_const']
    t0 = time.perf_counter()
    self.gp = self.O.OGP(w['X'], w['Y'], self.kern, lambda x: np.array([mc] * len(x)), w['noise_var'])
    return time.perf_counter() - t0

  def score(self):
    O, w, gp = self.O, self.w, self.gp
    C = w['candidates'][:self.sample]
    t0 = time.perf_counter()
    if self.config == 'headline':
      O.chunked_scores(gp, C, 'ei', chunk=CPU_CHUNK, curr_best=float(w['Y'].max()))
    elif self.config == 'c2':
      O.chunked_scores(gp, C, 'ucb', chunk=CPU_CHUNK, beta_th=O.ucb_beta_th(6, len(w['Y'])))
    elif self.config == 'c3':
      groups = self.kern.groupings
      per = max(1, self.sample // len(groups))
      for j, g in enumerate(groups):
        for s in range(0, per, CPU_CHUNK):
          O.add_ucb_group_scores(gp, self.kern, j, C[s:min(per, s + CPU_CHUNK)][:, :len(g)], len(w['Y']))
    elif self.config == 'c4':
      zx = O.mf_zx([1.0], C)
      O.chunked_scores(gp, zx, 'ucb', chunk=CPU_CHUNK, beta_th=O.ucb_beta_th(8, len(w['Y'])))
    else:   # c5: one exact joint block of 256 draws (the reference's own algorithm cannot go beyond a block)
      blk = C[:min(self.sample, 2048)]
      U = np.random.RandomState(2).standard_normal((len(blk), 256))
      gp.draw_samples_with_normals(blk, U)
      return time.perf_counter() - t0, len(blk)
    return time.perf_counter() - t0, len(C) if self.config != 'c3' else per * len(self.kern.groupings)


def cpu_measure(config, n_train, sample, steps, warmup, full_m):
  """ K timed steps of (posterior build + scoring of a bounded sample); best and mean.  `value` projects the two
      measured parts to the GPU arm's full step: full_m / (build + full_m / scoring_rate) -- the build is paid once per
      step whatever the number of candidates, so charging it to the small sample alone would understate the CPU. """
  use_all_host_threads()
  arm = CpuArm(config, n_train, sample)
  for _ in range(max(warmup, 0)):
    arm.build()
    arm.score()
  builds, scores, n_scored = [], [], 0
  for _ in range(steps):
    builds.append(arm.build())
    dt, n_scored = arm.score()
    scores.append(dt)
  b, s = float(np.mean(builds)), float(np.mean(scores))
  rate = n_scored / s
  value = full_m / (b + full_m / rate)
  return dict(value=value, build_s=b, score_s=s, scored=n_scored, rate=rate, best_rate=n_scored / min(scores),
              step_ms=1e3 * (b + s), builds=builds, scores=scores)


def cpu_block(m, config, cores):
  return {'value': m['value'], 'unit': UNIT, 'cores': cores, 'kind': 'port',
          'sample': '%d candidates per step in chunks of %d through the faithful gp.eval(chunk, "std") restatement '
                    '(chunk x chunk covariance + TRSM) + acquisition + running arg-max: %.0f cand/s (best step %.0f); '
                    'posterior build %.2f s per step INCLUDED, projected to the full step as '
                    'M / (build + M / scoring rate)' % (m['scored'], CPU_CHUNK, m['rate'], m['best_rate'], m['build_s']),
          'scoring_only_value': m['rate'], 'posterior_build_s': m['build_s']}


def run_reference(args):
  rank, world, _ = dist_env()
  if rank != 0:
    return
  n_train = n_train_of(args)
  full_m = args.cands_per_gpu if args.config == 'headline' else (args.global_cands or CONFIGS[args.config][1])
  m = cpu_measure(args.config, n_train, args.cpu_sample, args.steps, args.warmup, full_m)
  cores = cpu_threads()
  line = {
    'impl': 'reference', 'metric': METRIC, 'value': m['value'], 'unit': UNIT, 'n_gpus': args.gpus,
    'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': m['step_ms'],
    'higher_is_better': True, 'scaling': 'weak' if args.config == 'headline' else 'strong', 'vs_baseline': None,
    'dtype': 'f64', 'data': 'synthetic',
    'config': workload_config(args, 1),
    'cpu_baseline': cpu_block(m, args.config, cores),
    'e2e': {'value': m['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    'gpu_launches': 0,
  }
  print(json.dumps(line))


def workload_config(args, world):
  n = n_train_of(args)
  if args.config == 'headline':
    return {'workload': CONFIGS['headline'][2] % (n, args.cands_per_gpu),
            'n_train': n, 'dim': 6, 'kernel': 'matern-2.5', 'acquisition': 'ei',
            'candidates_per_gpu': args.cands_per_gpu, 'global_candidates': args.cands_per_gpu * world,
            'parallelism': 'candidate-sharded x%d (posterior replicated)' % world,
            'step': 'build_posterior + score + arg-max',
            'l2': 'explicit L2 flush (512 MB write) before every timed step; per-step working set '
                  '(W 210 MB + K_* chunk 267 MB) also exceeds the 126 MB L2'}
  gm = args.global_cands or CONFIGS[args.config][1]
  desc = CONFIGS[args.config][2] % ((gm, n) if args.config == 'c5' else (n, gm))
  return {'workload': desc, 'n_train': n, 'global_candidates': gm,
          'parallelism': 'candidate-sharded x%d inside the operator (posterior replicated)' % world,
          'step': 'build_posterior + the public operator (score + arg-max)',
          'l2': 'explicit L2 flush (512 MB write) before every timed step'}


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
class ClockSampler(object):
  Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
       'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
       'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, gpu_index):
    self.path = '/tmp/dfb_clocks_%d_%d.csv' % (os.getpid(), gpu_index)
    self.proc = None
    self.gpu_index = gpu_index

  def start(self):
    try:
      self.f = open(self.path, 'w')
      self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu_index), '--query-gpu=' + self.Q,
                                    '--format=csv,noheader,nounits', '-lms', '200'],
                                   stdout=self.f, stderr=subprocess.DEVNULL)
    except Exception:  # pylint: disable=broad-except
      self.proc = None

  def stop(self):
    out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
    if self.proc is None:
      return out
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except Exception:  # pylint: disable=broad-except
      self.proc.kill()
    self.f.close()
    sm, mx, pw, reasons = [], [], [], set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for row in open(self.path):
      parts = [p.strip() for p in row.split(',')]
      if len(parts) < 9:
        continue
      try:
        sm.append(float(parts[1])); mx.append(float(parts[2]))
      except ValueError:
        continue
      try:
        pw.append(float(parts[3]))
      except ValueError:
        pass
      for name, val in zip(names, parts[5:9]):
        if val.lower().startswith('active'):
          reasons.add(name)
    if sm:
      out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                 samples=len(sm), power_w=float(np.median(pw)) if pw else None)
    try:
      os.remove(self.path)
    except OSError:
      pass
    return out


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def measure_dgemm_peak(torch, dev):
  """ Live roofline denominator for the fp64 contraction: cuBLAS DGEMM 8192^3, best of 5
      (MEASURED_PEAKS.json holds no fp64 figure).  Not part of the product path. """
  n = 8192
  a = torch.randn(n, n, dtype=torch.float64, device=dev)
  b = torch.randn(n, n, dtype=torch.float64, device=dev)
  for _ in range(2):
    c = a @ b
  torch.cuda.synchronize(dev)
  best = 1e30
  for _ in range(5):
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(); c = a @ b; e1.record(); torch.cuda.synchronize(dev)
    best = min(best, e0.elapsed_time(e1))
  del a, b, c
  torch.cuda.empty_cache()
  return 2.0 * n ** 3 / best * 1e-9


def measure_issue_peaks(local):
  """ tcgen05 kind::i8 and fp64 DMMA issue rates measured in THIS process on THIS GPU (dfb_measure_peak,
      csrc/ubench.cu): the roofline denominators MEASURED_PEAKS.json does not carry. """
  import ctypes as C
  from dragonfly_b200 import _lib
  lib = _lib.load()
  out = {}
  for name, what in [('tcgen05_i8_tops', _lib.DFB_PEAK_TCGEN05_I8), ('dmma_f64_tflops', _lib.DFB_PEAK_DMMA_F64)]:
    v = C.c_double(0.0)
    st = lib.dfb_measure_peak(int(local), int(what), C.byref(v))
    out[name] = float(v.value) if st == 0 else None
  return out


def kstar_build_line(prof, n_train, peaks):
  """ The standalone materialising K_* build (fp64 rows written to HBM) against the HBM roofline: 8 N bytes written
      per candidate (SURVEY 8d; the padded row is 8 npad bytes, reported beside it). """
  ms, launches, cands = prof
  npad = (n_train + 127) // 128 * 128
  if ms <= 0:
    return None
  gbs = cands * n_train * 8.0 / (ms * 1e-3) * 1e-9
  hbm = float(peaks.get('hbm_gbs', 6564.2))
  return {'kernel': 'kstar_seg_kernel<Matern, p=2, d=6, ROWS64> (+ cand_prep, mu_reduce) writing fp64 K_* rows', 'achieved_gbs': gbs,
          'achieved_gbs_incl_padding': gbs * npad / n_train,
          'hbm_peak_gbs': hbm, 'frac_of_hbm': gbs / hbm, 'candidates_per_s': cands / (ms * 1e-3),
          'entries_per_s': cands * n_train / (ms * 1e-3), 'launch_ms_avg': ms / max(launches, 1),
          'bound': 'fp64 pipe / issue slots (sqrt + exp per entry), not HBM: see DESIGN.md 5.1'}


class Workload(object):
  """ Builds the GP of one configuration from HOST arrays and runs its step in two flavours. """

  def __init__(self, args, rank, world, local, torch):
    from dragonfly_b200 import synth_data, kernel, gp_core, mf_gp, device
    from dragonfly_b200 import gpb_acquisitions as A
    self.args, self.rank, self.world, self.local, self.torch = args, rank, world, local, torch
    self.A, self.gp_core, self.device, self.kernel, self.mf_gp = A, gp_core, device, kernel, mf_gp
    self.cfg = args.config
    self.n = n_train_of(args)
    self.w = synth_data.make_workload(CONFIGS[self.cfg][0], n_train=self.n, n_cand=16)
    self.mean = gp_core.ConstantMean(self.w['mean_const'])
    self.Xh, self.Yh = np.ascontiguousarray(self.w['X']), np.ascontiguousarray(self.w['Y'])
    self.dev = torch.device('cuda', local)
    if self.cfg == 'headline':
      self.M = args.cands_per_gpu
      self.global_m = self.M * world
      rs = np.random.RandomState(1000 + rank)
      host = torch.empty((self.M, 6), dtype=torch.float64, pin_memory=True)
      host.numpy()[:] = rs.random_sample((self.M, 6))
      self.cands_dev = host.to(self.dev)
      del host
      self.acq = device.make_acq_desc('ei', best=float(self.Yh.max()))
    else:
      self.global_m = args.global_cands or CONFIGS[self.cfg][1]
      self.M = self.global_m
      if self.cfg == 'c5':
        self.c5_cands = None
    self.d = self.w['dim']
    self.local_ms = []

  # -- model -------------------------------------------------------------------------------------
  def make_gp(self):
    w, k = self.w, self.w['kernel']
    if self.cfg == 'c4':
      kF = self.kernel.kernel_from_spec(k['kernels'][0]); kD = self.kernel.kernel_from_spec(k['kernels'][1])
      return self.mf_gp.EuclideanMFGP(list(self.Xh[:, :1]), list(self.Xh[:, 1:]), list(self.Yh), None, k['scale'], kF, kD,
                                      self.mean, w['noise_var'])
    return self.gp_core.GP(self.Xh, self.Yh, self.kernel.kernel_from_spec(k), self.mean, w['noise_var'], device=self.local)

  def anc(self, rng):
    from argparse import Namespace
    dom = self.A.EuclideanDomain([[0, 1]] * self.d)
    return Namespace(curr_acq='x', max_evals=self.global_m, t=self.n, domain=dom, curr_max_val=float(self.Yh.max()),
                     eval_points_in_progress=[], acq_opt_method='rand', handle_parallel='halluc', is_mf=False,
                     mf_strategy=None, domain_bounds=np.array(dom.bounds), candidate_rng=rng)

  def post_of(self, gp):
    return gp._post

  # -- steps -------------------------------------------------------------------------------------
  def step_device(self):
    """ Candidates resident in (or generated in) HBM: the `value` leg. """
    from dragonfly_b200 import dist as dfb_dist
    t0 = time.perf_counter()
    gp = self.make_gp()
    if self.cfg == 'headline':
      best, idx, _ = gp._fused_score(self.acq, self.cands_dev)      # returns after the device is done (16-byte read-back)
      self.local_ms.append(1e3 * (time.perf_counter() - t0))        # this rank's own work, before the collective
      idx += self.rank * self.M
      if self.world > 1:
        best, idx = dfb_dist.all_reduce_argmax(best, idx, self.dev)
      self.last_ret = (best, idx)
    else:
      self.last_ret = self.operator(gp, 'device')
    return gp

  def step_e2e(self):
    """ The reference-facing operator with the reference's own host-side candidate draw (NumPy global stream): every
        rank consumes the whole stream, uploads and scores its shard.  The `e2e` leg. """
    gp = self.make_gp()
    np.random.seed(7)
    if self.cfg == 'headline':
      self.last_ret = self.A.asy.ei(gp, self.anc('numpy'))
    else:
      self.last_ret = self.operator(gp, 'numpy')
    return gp

  def step_e2e_device_rng(self):
    """ The same operator in its throughput mode (anc_data.candidate_rng = 'device'): candidates generated on the GPU by
        global row index, so a rank neither draws nor uploads anything proportional to max_evals. """
    gp = self.make_gp()
    np.random.seed(7)
    if self.cfg == 'headline':
      self.last_ret = self.A.asy.ei(gp, self.anc('device'))
    else:
      self.last_ret = self.operator(gp, 'device')
    return gp

  def outputs(self, leg, gp, with_posterior):
    """ What the step just run handed its caller, as float64 arrays named <leg>_<what>: the arg-max of the leg and,
        with `with_posterior`, the posterior the step built (L as a fixed sample of 2^16 lower-triangle entries). """
    ret = self.last_ret
    if self.cfg == 'headline' and leg == 'device':
      out = {'best_score': ret[0], 'best_index': ret[1]}
    elif self.cfg == 'c5':
      out = {'draw_max_values': ret[0], 'draw_argmax_indices': ret[1]}
    else:
      out = {'point': ret}
    out = dict((leg + '_' + k, np.asarray(v, dtype=np.float64)) for k, v in out.items())
    if with_posterior:
      L = gp.L
      rs = np.random.RandomState(0)
      a, b = rs.randint(0, len(L), 1 << 16), rs.randint(0, len(L), 1 << 16)
      out.update(posterior_lml=np.float64(gp.compute_log_marginal_likelihood()),
                 posterior_alpha=np.asarray(gp.alpha, dtype=np.float64),
                 posterior_L_sample=np.asarray(L[np.maximum(a, b), np.minimum(a, b)], dtype=np.float64))
    return out

  def operator(self, gp, rng):
    A = self.A
    if self.cfg == 'c2':
      return A.asy.ucb(gp, self.anc(rng))
    if self.cfg == 'c3':
      return A.asy.add_ucb(gp, self.anc(rng))
    if self.cfg == 'c4':
      return A.asy.ucb(A._get_fidel_to_opt_gp(gp, [1.0]), self.anc(rng))
    # c5: 256 joint draws over the global candidate matrix, blocks shared out over the ranks by the method
    if rng == 'device':
      if self.c5_cands is None:
        self.c5_cands = gp._post.fill_candidates(12345, 0, self.global_m, [[0, 1]] * self.d)
      return gp.draw_samples_argmax(256, self.c5_cands, seed=2)
    cands = np.random.random((self.global_m, self.d))
    return gp.draw_samples_argmax(256, cands, seed=2)

  def h2d_bytes(self):
    train = self.Xh.nbytes + self.Yh.nbytes
    if self.cfg == 'c3':
      per_group = self.global_m // 7
      cand = sum(per_group * len(g) * 8 for g in self.w['kernel']['groupings'])
    else:
      cand = self.global_m * self.d * 8
    return int(cand + train * self.world)


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(out_dir, arrays):
  """ --dump-outputs: one float64 .npy per output, 64 MB at most in all. """
  total = sum(a.nbytes for a in arrays.values())
  if total > DUMP_LIMIT_BYTES:
    raise ValueError('outputs to dump take %d bytes, more than %d' % (total, DUMP_LIMIT_BYTES))
  os.makedirs(out_dir, exist_ok=True)
  for name, a in sorted(arrays.items()):
    np.save(os.path.join(out_dir, name + '.npy'), a)


def run_ours(args):
  import torch
  import torch.distributed as dist
  from dragonfly_b200 import device, gp_core
  rank, world, local = dist_env()
  assert torch.cuda.is_available(), 'bench.py needs a CUDA device: there is no CPU fallback'
  torch.cuda.set_device(local)
  dev = torch.device('cuda', local)
  # stdout carries exactly one JSON line: native libraries that write to fd 1 (NCCL prints its version banner
  # there) are pointed at stderr for the duration; the line itself goes to the saved descriptor.
  sys.stdout.flush()
  json_fd = os.dup(1)
  os.dup2(2, 1)
  if world > 1:
    dist.init_process_group('nccl', device_id=dev)
  wl = Workload(args, rank, world, local, torch)
  headline = args.config == 'headline'
  M, N = wl.M, wl.n
  flush = torch.empty(512 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)
  launches = [0]

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize(dev)

  dump = {} if args.dump_outputs and rank == 0 else None

  def timed(step, steps, leg=None):
    """ K steps; per step the larger of the device-event time and the host wall time of the same region (the
        host view includes Python + ctypes + the candidate draw), so nothing is hidden.  With --dump-outputs, the
        outputs of the last step of the named leg are kept, read back after its timed region. """
    times = []
    for s in range(steps):
      flush.fill_(1.0)
      e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
      torch.cuda.synchronize(dev)
      t0 = time.perf_counter()
      e0.record()
      gp = step()
      e1.record()
      torch.cuda.synchronize(dev)
      wall_ms = 1e3 * (time.perf_counter() - t0)
      times.append(max(e0.elapsed_time(e1), wall_ms))
      launches[0] += wl.post_of(gp).launch_count()
      if dump is not None and leg is not None and s == steps - 1:
        dump.update(wl.outputs(leg, gp, with_posterior=(leg == 'device')))
      del gp
    return times

  for _ in range(args.warmup):
    wl.step_device()
  barrier()
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  try:
    launches[0] = 0
    wl.local_ms = []
    t_dev = timed(wl.step_device, args.steps, 'device')
    local_ms = float(np.mean(wl.local_ms)) if wl.local_ms else 0.0
    n_launch = launches[0]
    barrier()
    wl.step_e2e()                                  # warm-up of the host path (pinned staging, thread start)
    barrier()
    t_e2e = timed(wl.step_e2e, args.steps, 'e2e')
    barrier()
    t_e2e_dev = []
    if headline:
      wl.step_e2e_device_rng()
      barrier()
      t_e2e_dev = timed(wl.step_e2e_device_rng, args.steps, 'e2e_device_candidates')
      barrier()
  finally:
    clocks = sampler.stop() if rank == 0 else None
  ms_dev, ms_e2e = float(np.sum(t_dev)), float(np.sum(t_e2e))
  ms_e2e_dev = float(np.mean(t_e2e_dev)) if t_e2e_dev else 0.0

  extras = {}
  prof, used_i8, shortlist, i8_bound, i8_impl, i8_r256 = {}, False, 0, 0.0, 2, 1
  dsig = None
  ms_fp64 = 0.0
  if headline:
    # per-kernel device timing for the roofline: same step, event pairs around every launch of the
    # dominant kernel on the launching stream (libdfb200's own profiling hooks).
    gp = wl.make_gp()
    gp._post.profile_enable(True)
    for _ in range(2):
      flush.fill_(1.0)
      gp._fused_score(wl.acq, wl.cands_dev)
    for name, cls in [('kstar', 0), ('gemm', 1), ('acq', 2)]:
      prof[name] = gp._post.profile_read(cls)
    gp._post.profile_enable(False)
    used_i8 = bool(gp._post.query('last_used_i8'))
    shortlist = int(gp._post.query('last_shortlist'))
    i8_bound = gp._post.query('i8_sigma2_bound')
    i8_impl = int(gp._post.query('i8_impl'))
    i8_r256 = int(gp._post.query('i8_radix256'))
    if used_i8 and rank == 0:
      # LIVE accuracy of the int8 screen on this posterior: sigma^2 of the same candidates through the int8-slice
      # contraction (score_impl 1 makes dfb_eval use it) and through fp64 DMMA (score_impl 0)
      sub = wl.cands_dev[:4 * int(gp._post.query('chunk'))]
      gp._post.set_option('score_impl', 1)
      _, sd8 = gp._post.eval(sub, mean_const=wl.w['mean_const'], want_std=True)
      gp._post.set_option('score_impl', 0)
      _, sd64 = gp._post.eval(sub, mean_const=wl.w['mean_const'], want_std=True)
      dsig = float((sd8 * sd8 - sd64 * sd64).abs().max())
      extras['int8_screen_check'] = {'max_abs_dsigma2': dsig, 'candidates': int(len(sub)), 'a_priori_bound': i8_bound,
                                     'contract': 1e-8}
    del gp
  if headline and not args.no_extras:
    # the same step with the int8 path disabled: pure fp64 DMMA contraction, for reference
    device.DEFAULT_OPTIONS['score_impl'] = 0
    wl.step_device()
    barrier()
    ms_fp64 = float(np.sum(timed(wl.step_device, args.steps)))
    # the materialising K_* build of the fp64 path (the north-star's "K_* build vs HBM" figure), timed per
    # launch with the same event hooks
    gp = wl.make_gp()
    gp._post.profile_enable(True)
    for _ in range(2):
      flush.fill_(1.0)
      gp._fused_score(wl.acq, wl.cands_dev[:200000])
    kstar64 = gp._post.profile_read(0)
    gp._post.profile_enable(False)
    del gp
    device.DEFAULT_OPTIONS.pop('score_impl')
    extras['kstar64'] = kstar64
    # incremental posterior update (dfb_extend_posterior) against the full rebuild the reference does on every
    # new observation: N-1 -> N points
    if rank == 0:
      upd = {}
      Xh, Yh = wl.Xh, wl.Yh
      kern = wl.kernel.kernel_from_spec(wl.w['kernel'])
      gp = gp_core.GP(Xh[:-1], Yh[:-1], kern, wl.mean, wl.w['noise_var'], device=local)
      post0 = gp._post
      torch.cuda.synchronize(dev)
      t0 = time.perf_counter()
      gp.add_data_multiple([Xh[-1]], [Yh[-1]])
      torch.cuda.synchronize(dev)
      upd['extend_1_point_ms'] = 1e3 * (time.perf_counter() - t0)
      upd['in_place'] = bool(gp._post is post0)
      lml_ext = gp.compute_log_marginal_likelihood()
      del gp, post0
      t0 = time.perf_counter()
      gp = gp_core.GP(Xh, Yh, kern, wl.mean, wl.w['noise_var'], device=local)
      torch.cuda.synchronize(dev)
      upd['full_build_ms'] = 1e3 * (time.perf_counter() - t0)
      upd['lml_rel_diff'] = abs(lml_ext - gp.compute_log_marginal_likelihood()) / abs(gp.compute_log_marginal_likelihood())
      t0 = time.perf_counter()
      grads = [gp.compute_grad_log_marginal_likelihood(p) for p in ('scale', 'noise_var', 'noise_mean')]
      torch.cuda.synchronize(dev)
      upd['lml_gradients_all_params_ms'] = 1e3 * (time.perf_counter() - t0)
      upd['lml_gradients_head'] = [float(g) for g in grads]
      upd['note'] = ('GP.add_data_multiple of one observation at N-1 -> N: in-place extension of the factorisation '
                     '(last row block of L / L^-1 only) vs GP(...) from scratch, host wall-clock incl. uploads; '
                     'lml_gradients: one dfb_lml_gradients call (all 4 + d gradients)')
      extras['posterior_update'] = upd
      del gp

  # max over ranks of every rank's own K-step time; per-rank figures kept
  mine = torch.tensor([ms_dev, ms_e2e, ms_fp64, local_ms, ms_e2e_dev], dtype=torch.float64, device=dev)
  per_rank = [mine.clone() for _ in range(world)]
  if world > 1:
    dist.all_gather(per_rank, mine)
  per_rank = torch.stack(per_rank).cpu().numpy()
  ms_dev, ms_e2e, ms_fp64 = [float(v) for v in per_rank.max(axis=0)[:3]]
  value = wl.global_m * args.steps / (ms_dev * 1e-3)
  e2e_value = wl.global_m * args.steps / (ms_e2e * 1e-3)

  if dump is not None:
    write_outputs(args.dump_outputs, dump)
  if rank == 0:
    peaks = {}
    try:
      peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:  # pylint: disable=broad-except
      pass
    step_ms = ms_dev / args.steps
    line = {
      'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': step_ms, 'higher_is_better': True,
      'scaling': 'weak' if headline else 'strong', 'vs_baseline': None,
      'dtype': 'f64', 'data': 'synthetic', 'config': workload_config(args, world),
      'clocks': clocks,
      'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': wl.h2d_bytes(),
              'd2h_bytes_per_step': 16 * world,
              'call': ('gpb_acquisitions.asy.ei(gp, anc_data) on GP(X_host, Y_host, ...): candidates from NumPy\'s global '
                       'MT19937 stream (the reference\'s random_maximise draw, streamed in slabs against the scoring), '
                       'H2D, score, arg-max point back') if headline else
                      'the configuration\'s public operator with the reference\'s host-side NumPy candidate draw',
              'ms_per_step': ms_e2e / args.steps},
      'gpu_launches': int(n_launch),
      'e2e_device_candidates': ({'value': wl.global_m / (float(per_rank[:, 4].max()) * 1e-3), 'unit': UNIT,
                                 'ms_per_step': float(per_rank[:, 4].max()),
                                 'call': 'the same asy.ei(gp, anc_data) with anc_data.candidate_rng = \'device\': candidates generated on the '
                                         'GPU by global row index (Philox), host inputs = the training data only'}
                                if float(per_rank[:, 4].max()) > 0 else None),
      'per_rank_ms_per_step': {'device': [float(v) / args.steps for v in per_rank[:, 0]],
                               'e2e': [float(v) / args.steps for v in per_rank[:, 1]],
                               'device_before_the_collective': [float(v) for v in per_rank[:, 3]]},
      'step_ms_each': {'device': t_dev, 'e2e': t_e2e},
      'collectives_per_step': {'headline': 1, 'c2': 1, 'c3': 7, 'c4': 1, 'c5': 1}[args.config] if world > 1 else 0,
    }
    if headline:
      N = wl.n
      issue = measure_issue_peaks(local)
      dgemm_peak = measure_dgemm_peak(torch, dev)
      gemm_ms, gemm_launches, gemm_cands = prof['gemm']
      flops_per_cand = float(N) * float(N + 1)       # triangular W: sum_i 2(i+1) = N(N+1) flops
      fp64_equiv = gemm_cands * flops_per_cand / (gemm_ms * 1e-3) * 1e-12 if gemm_ms > 0 else 0.0
      traffic = None
      tpath = os.path.join(ROOT, 'profiles', 'gemm_traffic.json')
      if os.path.exists(tpath):
        try:
          tj = json.load(open(tpath))
          traffic = tj.get({2: 'dram_bytes_per_launch_i8c2', 1: 'dram_bytes_per_launch_i8x2'}.get(i8_impl, 'dram_bytes_per_launch_i8')
                           if used_i8 else 'dram_bytes_per_launch')
        except Exception:  # pylint: disable=broad-except
          traffic = None
      share = {kname: prof[kname][0] / max(sum(p[0] for p in prof.values()), 1e-9) for kname in prof}
      if used_i8:
        # dominant kernel: the tcgen05 int8 contraction.  Algorithmic work: one int8 digit product per kept (s, t)
        # pair for every fp64 multiply-add of the triangular contraction -- 15 with five radix-256 digits, 21 with
        # six radix-128 digits.
        n_products = 15.0 if i8_r256 else 21.0
        ops_per_cand = n_products * flops_per_cand
        achieved = gemm_cands * ops_per_cand / (gemm_ms * 1e-3) * 1e-12
        peak = issue.get('tcgen05_i8_tops') or 4577.2
        digits = ('five radix-256 digits, 15 exact int8 products' if i8_r256
                  else 'six radix-128 digits, 21 exact int8 products')
        kname = {2: 'score_i8c2_kernel (persistent 2-CTA clusters; tcgen05.mma.cta_group::2 kind::i8 M256 N128 K32 / '
                    'UTCIMMA.2CTA, TMEM accumulators, TMA ring)',
                 1: 'score_i8x2_kernel (persistent, one CTA per SM; tcgen05.mma kind::i8 M128 N128 K32)',
                 0: 'score_i8_kernel (tcgen05.mma kind::i8 M128 N64 K32)'}[i8_impl]
        line['roofline'] = {
          'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TOP/s (int8)',
          'frac': achieved / peak, 'traffic': traffic, 'kernel': kname + ': V = L^-1 K_*^T as %s, fused |v|^2' % digits,
          'int8_products_per_fp64_fma': n_products, 'ops_per_candidate': ops_per_cand,
          'launch_ms_avg': gemm_ms / max(gemm_launches, 1), 'launches_timed': int(gemm_launches),
          'peak_source': 'tcgen05.mma kind::i8 issue rate (M128 N256 K32 from shared memory) measured live in this run '
                         'by dfb_measure_peak on this GPU; r01 ubench on this pool: 4577 TOP/s; MEASURED_PEAKS.json bf16 '
                         'burst = %s TF/s for comparison' % peaks.get('bf16_tflops', 'n/a'),
          'frac_at_sampled_clock': (achieved / (peak * clocks['sm_mhz'] / clocks['sm_max_mhz'])
                                    if clocks and clocks.get('sm_mhz') else None),
          'fp64_equivalent_tflops': fp64_equiv,
          'fp64_equivalent_vs_cublas_dgemm': fp64_equiv / dgemm_peak if dgemm_peak > 0 else None,
          'cublas_dgemm_tflops_live': dgemm_peak, 'dmma_issue_peak_tflops_live': issue.get('dmma_f64_tflops'),
          'share_of_scoring': share,
          'i8_sigma2_error_bound': i8_bound, 'argmax_shortlist_rescored_fp64': shortlist}
        line['dtype'] = ('f64 (sigma^2 contraction screened by an int8 digit expansion of the fp64 operands on tcgen05: '
                         'a-priori |d sigma^2| <= %.1e, measured in this run %s over %d candidates; arg-max re-scored in '
                         'fp64 DMMA)' % (i8_bound, ('%.1e' % dsig) if dsig is not None else 'n/a',
                                         extras.get('int8_screen_check', {}).get('candidates', 0)))
        line['int8_screen_check'] = extras.get('int8_screen_check')
      else:
        line['roofline'] = {
          'bound': 'tensor', 'achieved': fp64_equiv, 'peak': dgemm_peak, 'unit': 'TFLOP/s',
          'frac': fp64_equiv / dgemm_peak if dgemm_peak > 0 else None, 'traffic': traffic,
          'kernel': 'score_tma_kernel (fp64 DMMA, TMA + mbarrier ring: V = L^-1 K_*^T fused with |v|^2)',
          'flops_per_candidate': flops_per_cand, 'launch_ms_avg': gemm_ms / max(gemm_launches, 1),
          'launches_timed': int(gemm_launches),
          'peak_source': 'live cuBLAS DGEMM 8192^3 burst on this GPU; DMMA issue peak measured live: %s TFLOP/s'
                         % issue.get('dmma_f64_tflops'), 'share_of_scoring': share}
      if not args.no_extras:
        line['fp64_dmma_only'] = {'value': M * world * args.steps / (ms_fp64 * 1e-3), 'unit': UNIT,
                                  'note': 'same step with DFB200_SCORE=fp64 (no int8 path), %d timed steps' % args.steps}
        line['kstar_build_fp64'] = kstar_build_line(extras['kstar64'], N, peaks)
        line['posterior_update'] = extras.get('posterior_update')
    if not args.no_cpu_baseline and world == 1:
      full_m = wl.global_m
      m = cpu_measure(args.config, wl.n, args.cpu_sample, 1, 1, full_m)
      line['cpu_baseline'] = cpu_block(m, args.config, cpu_threads())
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + '\n').encode())
  os.close(json_fd)
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


def main():
  args = parse_args()
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_ours(args)


if __name__ == '__main__':
  main()
