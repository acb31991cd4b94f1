#!/usr/bin/env python3
"""bench.py -- UIS-RNN predict() throughput on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
  python bench.py --impl reference --gpus N --steps K ...  # reference CPU arm (host cores)

A "step" is one predict() pass over one batch of synthetic utterances (BASELINE config 2:
500-frame 256-d utterances, hidden 512, beam_size 10, look_ahead 1, test_iteration 2).
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definitions.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

METRIC = 'predict_frames_per_sec_beam10_256d'
UNIT = 'frames/s'
N_FRAMES, DIM, HIDDEN, BEAM, LOOK_AHEAD, TEST_ITER = 500, 256, 512, 10, 1, 2
WORKLOAD = ('configs[1]: predict() synthetic 256-d d-vectors, 500-frame utterances, hidden=512, '
            'beam_size=10, look_ahead=1, test_iteration=2')
MODEL_FIXTURE = os.path.join(ROOT, 'tests', 'golden', 'model_toy100.npz')
FIRST_SEED = 100000          # utterance i of the workload = synth_utt(FIRST_SEED + i)
STRONG_UTTS = 888            # fixed list of the strong-scaling side measurement (utterances 0..887 of the job)
MMA_FLOOR_CYCLES = 86.4      # measured: cycles per 128 x N x 16 kind::f16 MMA fed from shared memory, N <= 128
                             # (tools/tc/tc_chain_probe.cu, profiles/r2_tc_chain_probe_uniform_issue.txt)
DUMP_LIMIT_BYTES = 64 << 20  # --dump-outputs writes at most this much


def synth_batch(first_seed, n_utt, pinned=False):
  from uisrnn_b200.synth import synth_utt
  seqs = []
  for u in range(n_utt):
    x = synth_utt(first_seed + u, n_frames=N_FRAMES, dim=DIM)[0]
    if pinned:
      import torch
      t = torch.from_numpy(x).pin_memory()
      seqs.append((t.numpy(), t))  # keep the pinned tensor alive next to its numpy view
    else:
      seqs.append((x, None))
  return seqs


class ClockSampler:
  """Samples nvidia-smi SM clocks / throttle reasons while the timed region runs."""
  Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
       'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
       'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, gpu_index=0):
    self.gpu = gpu_index
    self.lines = []
    self.proc = None

  def start(self):
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
           '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thr = threading.Thread(target=self._pump, daemon=True)
      self.thr.start()
    except Exception:  # pylint: disable=broad-except
      self.proc = None

  def _pump(self):
    for line in self.proc.stdout:
      self.lines.append(line.strip())

  def stop(self):
    if not self.proc:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except Exception:  # pylint: disable=broad-except
      self.proc.kill()
    sm, smax, reasons, power = [], [], set(), []
    for ln in self.lines:
      f = [s.strip() for s in ln.split(',')]
      if len(f) < 9:
        continue
      try:
        sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
      except ValueError:
        continue
      for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
        if v.lower().startswith('active'):
          reasons.add(name)
    if not sm:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
    busy = [c for c, p in zip(sm, power) if p > 0.5 * max(power)] or sm
    return {'sm_mhz': float(np.median(busy)), 'sm_max_mhz': float(max(smax)), 'reasons': sorted(reasons),
            'samples': len(sm), 'power_w_max': float(max(power))}


def load_peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      d = json.load(f)
    return {'hbm_gbs': float(d['hbm_gbs']), 'tensor_tflops': float(d['bf16_tflops']),
            'tensor_tflops_sustained': float(d.get('bf16_tflops_sustained', d['bf16_tflops'])),
            'sm_max_mhz': float(d.get('sm_max_mhz', 1965.0)), 'source': 'measured (MEASURED_PEAKS.json)'}
  return {'hbm_gbs': 6650.0, 'tensor_tflops': 1590.0, 'tensor_tflops_sustained': 1400.0, 'sm_max_mhz': 1965.0,
          'source': 'fallback (B200_PROFILING.md)'}


def measured_traffic(utts, engine):
  """DRAM bytes per launch of the beam kernel from the committed ncu capture of THIS build's kernel on THIS
  workload size (profiles/r3_traffic.json); None when the capture does not match what was just run."""
  path = os.path.join(ROOT, 'profiles', 'r3_traffic.json')
  try:
    with open(path) as f:
      d = json.load(f)
    if d['utterances'] == utts and d['frames_per_utterance'] == N_FRAMES and d['engine'] == engine:
      return d['dram_bytes_read'] + d['dram_bytes_write'], d.get('l2_to_sm_bytes')
  except Exception:  # pylint: disable=broad-except
    pass
  return None, None


def host_info():
  """Usable host cores: scheduler affinity and the cgroup CPU quota, not os.cpu_count()."""
  info = {'os_cpu_count': os.cpu_count()}
  try:
    info['affinity'] = len(os.sched_getaffinity(0))
  except Exception:  # pylint: disable=broad-except
    info['affinity'] = os.cpu_count() or 1
  quota = None
  try:
    with open('/sys/fs/cgroup/cpu.max') as f:
      q, per = f.read().split()
    if q != 'max':
      quota = float(q) / float(per)
  except Exception:  # pylint: disable=broad-except
    try:
      with open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us') as f:
        q = float(f.read())
      with open('/sys/fs/cgroup/cpu/cpu.cfs_period_us') as f:
        per = float(f.read())
      if q > 0:
        quota = q / per
    except Exception:  # pylint: disable=broad-except
      pass
  info['cgroup_cpu_quota'] = quota
  usable = info['affinity']
  if quota:
    usable = max(1, min(usable, int(quota)))
  info['usable_cores'] = usable
  try:
    with open('/proc/cpuinfo') as f:
      for ln in f:
        if ln.startswith('model name'):
          info['cpu_model'] = ln.split(':', 1)[1].strip()
          break
  except Exception:  # pylint: disable=broad-except
    pass
  return info


def secondary_metrics(model, torch):
  """Best-effort extra numbers for the other BASELINE configs (never allowed to break the headline line)."""
  out = {}
  try:  # config 4: fit() iteration on 50k concatenated frames, batch_size=32 (device trainer, csrc/uis_train.cu)
    import random
    from uisrnn_b200 import native, utils
    from uisrnn_b200.synth import synth_training_set
    np.random.seed(0); random.seed(0)
    seqs, ids = synth_training_set(2000, 500, n_frames=100, dim=DIM, n_spk=3)
    xcat, ycat = utils.concatenate_training_data(seqs, ids, True, True)
    index_lists, lens = utils.resize_indices(np.array(ycat), 10)
    w = dict(np.load(MODEL_FIXTURE))
    params = {'gru.weight_ih_l0': w['weight_ih_l0'], 'gru.weight_hh_l0': w['weight_hh_l0'], 'gru.bias_ih_l0': w['bias_ih_l0'],
              'gru.bias_hh_l0': w['bias_hh_l0'], 'linear_mean1.weight': w['w1'], 'linear_mean1.bias': w['b1'],
              'linear_mean2.weight': w['w2'], 'linear_mean2.bias': w['b2'], 'rnn_init_hidden': w['h0'].reshape(-1),
              'sigma2': w['sigma2']}
    hp = {'learning_rate': 1e-3, 'sigma_alpha': 1.0, 'sigma_beta': 1.0, 'regularization_weight': 1e-5,
          'grad_max_norm': 5.0, 'train_sigma2': True}
    tr = native.NativeTrainer(params, hp)
    tr.set_corpus(xcat, index_lists)             # as UISRNN.fit does: training set resident on the device
    sampler = utils.BatchSampler(lens, 32)
    iters, rows = 100, 0
    fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(5 + iters):
      if i == 5:
        tr.losses(1); t0 = time.perf_counter(); fe0.record()
      chosen, li = sampler.draw()
      if i >= 5:
        rows += int(li.sum())
      tr.step_corpus(chosen)                     # asynchronous; the batch is gathered on the device
    fe1.record()
    tr.losses(1)                                 # synchronises
    dt = time.perf_counter() - t0
    out['config4_fit_batch32'] = {'ms_per_iteration': 1e3 * dt / iters, 'device_ms_per_iteration': fe0.elapsed_time(fe1) / iters,
                                  'packed_rows_per_s': rows / dt,
                                  'includes': 'batch draw (host RNG) + device gather + forward/backward/clip/Adam kernels'}
    tr.close()
  except Exception as err:  # pylint: disable=broad-except
    out['config4_fit_batch32'] = {'error': str(err)[:200]}
  try:  # config 3: beam_size=30, look_ahead=2 (wide-beam stress), device-resident, 148 x 100 frames
    from uisrnn_b200.synth import synth_utt
    U3, N3 = 148, 100
    x3 = torch.from_numpy(np.concatenate([synth_utt(1000 + u, n_frames=N3, dim=DIM)[0] for u in range(U3)]).astype(np.float32)).cuda()
    lab3 = torch.empty(U3 * N3, dtype=torch.int32, device='cuda')
    off3 = np.arange(U3 + 1, dtype=np.int64) * N3
    for _ in range(2):
      model.predict_device(x3.data_ptr(), off3, lab3.data_ptr(), beam_size=30, look_ahead=2, test_iteration=TEST_ITER)
      st3 = model.stats()
    out['config3_beam30_lookahead2'] = {'frames_per_s': U3 * N3 / (st3['beam_ms'] / 1e3), 'kernel_ms': st3['beam_ms'],
                                        'gru_columns_per_step': st3['gru_columns'] / max(1, st3['beam_steps'])}
  except Exception as err:  # pylint: disable=broad-except
    out['config3_beam30_lookahead2'] = {'error': str(err)[:200]}
  try:  # SURVEY 8(d): latency mode (U=1), small batches and the FFMA engine on the bench batch, device-resident
    from uisrnn_b200.synth import synth_utt
    for U1, engine in ((1, 0), (64, 0), (296, 1)):
      xs = torch.from_numpy(np.concatenate([synth_utt(1000 + u, n_frames=N_FRAMES, dim=DIM)[0] for u in range(U1)]).astype(np.float32)).cuda()
      lab = torch.empty(U1 * N_FRAMES, dtype=torch.int32, device='cuda')
      offs = np.arange(U1 + 1, dtype=np.int64) * N_FRAMES
      for _ in range(2):
        model.predict_device(xs.data_ptr(), offs, lab.data_ptr(), beam_size=BEAM, look_ahead=LOOK_AHEAD,
                             test_iteration=TEST_ITER, engine=engine)
        stu = model.stats()
      key = 'config2_U%d' % U1 + ('_ffma_engine' if engine == 1 else '')
      out[key] = {'frames_per_s': U1 * N_FRAMES / ((stu['beam_ms'] + stu['prepass_ms']) / 1e3),
                  'ms': stu['beam_ms'] + stu['prepass_ms'], 'ctas': stu['ctas'], 'lanes': stu['lanes'],
                  'cluster': stu['cluster'], 'engine': stu['engine']}
  except Exception as err:  # pylint: disable=broad-except
    out['config2_small_batches'] = {'error': str(err)[:200]}
  return out


def partition_secondary(api_model, iargs, rank, world, torch, dist, barrier):
  """Side measurements every rank takes part in (SURVEY 8(e)): (a) STRONG scaling of the partition -- one fixed list
  of STRONG_UTTS utterances (the first ones of the job's list) sharded over the ranks with predict_sharded, labels
  gathered to rank 0, timed end to end; (b) data-parallel fit(): config-4 shapes, batch 32 sharded over the ranks,
  one NCCL all-reduce of [gradients | loss statistics] per iteration.  Returns a dict on rank 0 (else None)."""
  import random
  from uisrnn_b200 import native, utils
  from uisrnn_b200.distributed import my_shard, predict_sharded
  from uisrnn_b200.synth import synth_training_set, synth_utt
  from uisrnn_b200.uisrnn import shard_columns
  out = {}
  try:
    lengths = [N_FRAMES] * STRONG_UTTS
    own = set(my_shard(lengths))
    held = {i: torch.from_numpy(synth_utt(FIRST_SEED + i, n_frames=N_FRAMES, dim=DIM)[0]).pin_memory() for i in own}
    lazy = [held[i].numpy() if i in own else None for i in range(STRONG_UTTS)]
    run = lambda: predict_sharded(api_model, lazy, iargs, lengths=lengths, root=0, as_arrays=True)
    run(); run()
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
      res = run()
    torch.cuda.synchronize()
    t = torch.tensor([(time.perf_counter() - t0) / 3], dtype=torch.float64, device='cuda')
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    st = api_model._native_model().stats()  # pylint: disable=protected-access
    digest = int(np.concatenate([np.asarray(r, dtype=np.int64) for r in res]).sum()) if rank == 0 else 0
    out['strong_scaling_fixed_list'] = {
        'utterances_total': STRONG_UTTS, 'utterances_per_gpu': len(own), 'e2e_ms': float(t[0]) * 1e3,
        'frames_per_s': STRONG_UTTS * N_FRAMES / float(t[0]), 'label_checksum': digest,
        'rank0_kernel': {'engine': st['engine'], 'lanes': st['lanes'], 'ctas': st['ctas'], 'cluster': st['cluster'],
                         'beam_ms': st['beam_ms']},
        'note': 'fixed total work: with fewer than 2 utterances per SM a rank leaves the 6-lane tensor-core kernel for the '
                'one-utterance-per-CTA (or cluster) kernels, whose time is the latency of one 1000-step utterance -- the '
                'floor of strong scaling; label_checksum must be the same at every N'}
  except Exception as err:  # pylint: disable=broad-except
    out['strong_scaling_fixed_list'] = {'error': str(err)[:200]}
  try:
    np.random.seed(0); random.seed(0)
    seqs, ids = synth_training_set(2000, 200, n_frames=100, dim=DIM, n_spk=3)
    xcat, ycat = utils.concatenate_training_data(seqs, ids, True, True)
    index_lists, lens = utils.resize_indices(np.array(ycat), 10)
    w = dict(np.load(MODEL_FIXTURE))
    params = {'gru.weight_ih_l0': w['weight_ih_l0'], 'gru.weight_hh_l0': w['weight_hh_l0'], 'gru.bias_ih_l0': w['bias_ih_l0'],
              'gru.bias_hh_l0': w['bias_hh_l0'], 'linear_mean1.weight': w['w1'], 'linear_mean1.bias': w['b1'],
              'linear_mean2.weight': w['w2'], 'linear_mean2.bias': w['b2'], 'rnn_init_hidden': w['h0'].reshape(-1),
              'sigma2': w['sigma2']}
    hp = {'learning_rate': 1e-3, 'sigma_alpha': 1.0, 'sigma_beta': 1.0, 'regularization_weight': 1e-5,
          'grad_max_norm': 5.0, 'train_sigma2': True}
    tr = native.NativeTrainer(params, hp, device=torch.cuda.current_device())
    tr.set_corpus(xcat, index_lists)
    sampler = utils.BatchSampler(lens, 32)
    comm = torch.zeros(tr.comm_size(), dtype=torch.float32, device='cuda')
    iters = 60
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(5 + iters):
      if i == 5:
        tr.losses(1); barrier(); e0.record()
      chosen, _ = sampler.draw()                # same RNG state on every rank: the same batch
      if world == 1:
        tr.step_corpus(chosen)
      else:
        mine = shard_columns(len(chosen), rank, world)
        tr.step_corpus(chosen[mine], mode=2)
        tr.comm_export(comm.data_ptr())
        dist.all_reduce(comm, op=dist.ReduceOp.SUM)
        tr.comm_apply(comm.data_ptr())
    e1.record()
    last = tr.losses(1)
    t = torch.tensor([e0.elapsed_time(e1) / iters], dtype=torch.float64, device='cuda')
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out['fit_data_parallel_batch32'] = {
        'ms_per_iteration': float(t[0]), 'columns_per_rank': -(-32 // world), 'allreduce_floats': int(tr.comm_size()),
        'loss1_last': float(last[0, 0]),
        'note': 'device time, max over ranks; bounded by the ~100 sequential recurrence steps of the longest sequence '
                '(their cost barely depends on the number of live columns) plus one 6.3 MB all-reduce per iteration'}
    tr.close()
  except Exception as err:  # pylint: disable=broad-except
    out['fit_data_parallel_batch32'] = {'error': str(err)[:200]}
  return out if rank == 0 else None


# --------------------------------------------------------------------------- CPU legs (reference / oracle)

def _ref_worker(job):
  """One process of the CPU legs: decodes the first `n_frames` frames of workload utterance `seed` with the
  unmodified reference (kind 'reference': oracle/_ref through its public predict()), the reference on a CUDA
  device ('reference_cuda') or the oracle port; returns (seconds, labels)."""
  kind, weights_path, seed, n_frames, threads = job
  import torch
  if threads:
    torch.set_num_threads(threads)
  from uisrnn_b200.synth import synth_utt
  x = synth_utt(seed, n_frames=N_FRAMES, dim=DIM)[0][:n_frames]
  if kind in ('reference', 'reference_cuda'):
    sys.path[:0] = [os.path.join(ROOT, 'oracle', 'shims'), os.path.join(ROOT, 'oracle', '_ref')]
    import uisrnn as ref
    assert os.path.join('oracle', '_ref') in ref.__file__
    argv, sys.argv = sys.argv, [sys.argv[0]]
    try:
      margs, _, iargs = ref.parse_arguments()
    finally:
      sys.argv = argv
    margs.enable_cuda = (kind == 'reference_cuda')
    margs.verbosity = 0
    w = dict(np.load(weights_path))
    margs.transition_bias = float(w['transition_bias'])
    margs.crp_alpha = float(w['crp_alpha'])
    model = ref.UISRNN(margs)
    dev = model.device
    sd = {'gru.weight_ih_l0': w['weight_ih_l0'], 'gru.weight_hh_l0': w['weight_hh_l0'],
          'gru.bias_ih_l0': w['bias_ih_l0'], 'gru.bias_hh_l0': w['bias_hh_l0'],
          'linear_mean1.weight': w['w1'], 'linear_mean1.bias': w['b1'],
          'linear_mean2.weight': w['w2'], 'linear_mean2.bias': w['b2']}
    model.rnn_model.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
    model.rnn_init_hidden = torch.nn.Parameter(torch.from_numpy(np.array(w['h0'])).to(dev))
    model.sigma2 = torch.nn.Parameter(torch.from_numpy(np.array(w['sigma2'])).to(dev))
    if kind == 'reference_cuda':
      model.predict(x[:4], iargs)  # CUDA context / cuDNN start-up outside the timed call
      torch.cuda.synchronize()
    t0 = time.perf_counter()
    labels = model.predict(x, iargs)   # the reference's own public API, stock code path
    if kind == 'reference_cuda':
      torch.cuda.synchronize()
  else:
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import uis_oracle
    om = uis_oracle.OracleModel.load(weights_path)
    t0 = time.perf_counter()
    labels = uis_oracle.predict_single(om, x, beam_size=BEAM, look_ahead=LOOK_AHEAD, test_iteration=TEST_ITER)
  return time.perf_counter() - t0, [int(v) for v in labels]


def have_reference():
  return os.path.exists(os.path.join(ROOT, 'oracle', '_ref', 'uisrnn', 'uisrnn.py'))


def run_in_fresh_process(jobs, procs=1):
  """The reference package is also called `uisrnn`: it only ever runs in spawned processes of its own."""
  import multiprocessing as mp
  with mp.get_context('spawn').Pool(procs) as pool:
    return pool.map(_ref_worker, jobs, chunksize=1)


def cpu_baseline_and_parity(gpu_labels_of):
  """(a) cpu_baseline: SURVEY 8(d)(i), the unmodified reference in ONE process with the default torch threads on a
  bounded sample (2 slices x 40 frames of workload utterances; the oracle port if oracle/_ref is absent);
  (b) parity: full 500-frame utterances of the timed batch decoded by the oracle port -- the checker -- and compared
  with the labels the GPU produced for the same utterances."""
  import torch
  kind = 'reference' if have_reference() else 'port'
  n_slices, slice_frames = 1, 40
  # torch's default thread count is the machine's core count; inside a CPU-quota'd container that oversubscribes the
  # cores the process may use (measured: 0.8 frames/s with 64 threads on a 16-core quota), so the leg runs with
  # min(default, usable cores) threads -- the better number for the reference
  threads = max(1, min(torch.get_num_threads(), host_info()['usable_cores']))
  t0 = time.perf_counter()
  res = run_in_fresh_process([(kind, MODEL_FIXTURE, FIRST_SEED + i, slice_frames, threads) for i in range(n_slices)], 1)
  wall = time.perf_counter() - t0
  busy = sum(r[0] for r in res)
  cpu = {'value': n_slices * slice_frames / busy, 'unit': UNIT, 'cores': threads, 'kind': kind,
         'sample': '%d slice x %d frames of a workload utterance (seed %d), one process, %d torch threads (default %d, '
                   'usable cores %d), %s; %.1f s in predict(), %.1f s with start-up' % (
                       n_slices, slice_frames, FIRST_SEED, threads, torch.get_num_threads(), host_info()['usable_cores'],
                       'unmodified reference predict() from oracle/_ref' if kind == 'reference' else 'oracle/uis_oracle.py port',
                       busy, wall)}
  # parity: utterances of the batch at their whole length (the reference-decoded ones are checked separately)
  which = sorted(gpu_labels_of.keys())
  t0 = time.perf_counter()
  res = run_in_fresh_process([('port', MODEL_FIXTURE, FIRST_SEED + i, N_FRAMES, 1) for i in which], len(which))
  ok = sum(1 for i, r in zip(which, res) if r[1] == [int(v) for v in gpu_labels_of[i]])
  parity = {'checked': len(which), 'identical': ok, 'utterances': which, 'checker': 'oracle/uis_oracle.py (pinned to the '
            'reference by tests/test_oracle_golden.py), full %d-frame utterances' % N_FRAMES,
            'seconds': round(time.perf_counter() - t0, 1)}
  return cpu, parity


# --------------------------------------------------------------------------- reference arm

def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  import multiprocessing as mp
  kind = 'reference' if have_reference() else 'port'
  host = host_info()
  procs = max(1, min(host['usable_cores'], 256))
  # Slice length: as long as the time budget allows (the reference needs ~0.1-0.3 s per frame and process).  One
  # calibration step with 16-frame slices on every process, then frames = 16 * budget / t16 (cost is ~linear in the
  # slice length once the beam is full), capped at the workload's 500.
  budget_total = float(os.environ.get('UIS_BENCH_REF_SECONDS', '420'))
  budget_step = budget_total / max(1, args.steps + args.warmup)
  ctx = mp.get_context('spawn')
  times = []
  with ctx.Pool(procs) as pool:
    cal = pool.map(_ref_worker, [(kind, MODEL_FIXTURE, FIRST_SEED + i, 16, 1) for i in range(procs)], chunksize=1)
    t16 = max(r[0] for r in cal)  # slowest predict() of the calibration step (imports / model set-up not included)
    n_frames = int(max(16, min(N_FRAMES, 16 * 0.8 * budget_step / t16)))
    for step in range(args.warmup + args.steps):
      jobs = [(kind, MODEL_FIXTURE, FIRST_SEED + (step * procs + i) % 100000, n_frames, 1) for i in range(procs)]
      t0 = time.perf_counter()
      pool.map(_ref_worker, jobs, chunksize=1)
      dt = time.perf_counter() - t0
      if step >= args.warmup:
        times.append(dt)
  frames = procs * n_frames
  total = sum(times)
  value = frames * len(times) / total
  sample = ('%d processes x 1 utterance slice of %d frames per step (the workload generator and seeds of the GPU arm), '
            '%s, 1 torch thread per process; calibration step with 16-frame slices: %.1f s' % (
                procs, n_frames, 'unmodified reference predict() from oracle/_ref' if kind == 'reference'
                else 'oracle/uis_oracle.py port', t16))
  secondary = {}
  try:  # SURVEY 8(d)(i): one process, default torch threads
    r = run_in_fresh_process([(kind, MODEL_FIXTURE, FIRST_SEED, 40, 0)], 1)[0]
    secondary['single_process_default_threads'] = {'frames_per_s': 40 / r[0], 'sample': '1 slice x 40 frames'}
  except Exception as err:  # pylint: disable=broad-except
    secondary['single_process_default_threads'] = {'error': str(err)[:200]}
  if kind == 'reference':
    try:  # the "existing kernels on the same GPU" bar: the reference's own --enable_cuda=True path (eager cuDNN/cuBLAS)
      import torch
      if torch.cuda.is_available():
        rs = run_in_fresh_process([('reference_cuda', MODEL_FIXTURE, FIRST_SEED + i, 40, 0) for i in range(2)], 1)
        secondary['reference_enable_cuda_on_this_gpu'] = {
            'frames_per_s': 80 / sum(r[0] for r in rs), 'sample': '2 slices x 40 frames, one process, stock code path'}
    except Exception as err:  # pylint: disable=broad-except
      secondary['reference_enable_cuda_on_this_gpu'] = {'error': str(err)[:200]}
  out = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
         'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * total / len(times),
         'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
         'config': {'workload': WORKLOAD, 'sample_frames_per_step': frames, 'slice_frames': n_frames,
                    'same_config': n_frames == N_FRAMES,
                    'note': 'a step decodes the first slice_frames frames of `processes` workload utterances (the whole '
                            '500 frames do not fit the time limit of this arm); short slices favour the reference '
                            '(fewer clusters, the beam is still filling), so the ratio to the GPU arm is conservative',
                    'host': host},
         'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': procs, 'kind': kind, 'sample': sample},
         'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
         'secondary': secondary}
  print(json.dumps(out), flush=True)


# --------------------------------------------------------------------------- this repo's arm

def dump_outputs(path, out):
  """Writes the labels the timed path returned in its last step, one row per utterance of the job's list, as float32 to
  PATH/labels.npy, and the list index of each row to PATH/labels_utterances.npy (utterance i is synth_utt(FIRST_SEED
  + i), so two builds run with the same arguments can be compared output for output).  Where all rows would exceed
  DUMP_LIMIT_BYTES, a fixed seeded sample of the rows is written."""
  labels = np.asarray([np.asarray(o) for o in out], dtype=np.float32)
  rows = np.arange(len(labels))
  cap = (DUMP_LIMIT_BYTES - 4096) // (labels.shape[1] * 4 + 8)   # 4096: room for the two .npy headers
  if len(rows) > cap:
    rows = np.sort(np.random.default_rng(0).choice(len(rows), cap, replace=False))
  os.makedirs(path, exist_ok=True)
  np.save(os.path.join(path, 'labels.npy'), labels[rows])
  np.save(os.path.join(path, 'labels_utterances.npy'), rows.astype(np.float64))


def build_api_model(weights, local, torch):
  import uisrnn
  margs, _, iargs = uisrnn.parse_arguments([])
  margs.verbosity, margs.transition_bias, margs.crp_alpha = 0, float(weights['transition_bias']), float(weights['crp_alpha'])
  api_model = uisrnn.UISRNN(margs)
  assert api_model.device.type == 'cuda'
  if local != 0:
    api_model.device = torch.device('cuda', local)
  sd = {'gru.weight_ih_l0': weights['weight_ih_l0'], 'gru.weight_hh_l0': weights['weight_hh_l0'],
        'gru.bias_ih_l0': weights['bias_ih_l0'], 'gru.bias_hh_l0': weights['bias_hh_l0'],
        'linear_mean1.weight': weights['w1'], 'linear_mean1.bias': weights['b1'],
        'linear_mean2.weight': weights['w2'], 'linear_mean2.bias': weights['b2']}
  api_model.rnn_model.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
  api_model.rnn_init_hidden = torch.nn.Parameter(torch.from_numpy(np.array(weights['h0'])).to(api_model.device))
  api_model.sigma2 = torch.nn.Parameter(torch.from_numpy(np.array(weights['sigma2'])).to(api_model.device))
  iargs.beam_size, iargs.look_ahead, iargs.test_iteration = BEAM, LOOK_AHEAD, TEST_ITER
  return api_model, iargs


def run_b200(args):
  import torch
  import torch.distributed as dist
  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  if not torch.cuda.is_available():
    raise SystemExit('bench.py: no CUDA device; the sm_100a path cannot run (no CPU fallback by design)')
  torch.cuda.set_device(local)
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
  import __graft_entry__ as ge
  ge.build()
  from uisrnn_b200 import native
  from uisrnn_b200.distributed import my_shard, predict_sharded

  U = args.utts           # utterances per GPU per step (weak scaling: fixed per GPU)
  weights = dict(np.load(MODEL_FIXTURE))
  model = native.NativeModel(weights, device=local)
  # The job's utterance list: world * U utterances, utterance i = synth_utt(FIRST_SEED + i).  Rank r owns the shard
  # `shard_by_frames` gives it (the partition predict_sharded / parallel_predict use) and generates only that.
  lengths = [N_FRAMES] * (world * U)
  mine = my_shard(lengths)
  assert len(mine) == U
  from uisrnn_b200.synth import synth_utt
  held, seqs = [], []
  for i in mine:
    t = torch.from_numpy(synth_utt(FIRST_SEED + i, n_frames=N_FRAMES, dim=DIM)[0])
    if not args.pageable:
      t = t.pin_memory()
    held.append(t)
    seqs.append(t.numpy())
  frames = U * N_FRAMES
  stream = torch.cuda.current_stream().cuda_stream

  # ---- device-resident leg (`value`): fp32 inputs already in HBM
  x_dev = torch.from_numpy(np.concatenate(seqs).astype(np.float32)).cuda()
  labels_dev = torch.empty(frames, dtype=torch.int32, device='cuda')
  off = np.arange(U + 1, dtype=np.int64) * N_FRAMES

  def step_dev():
    model.predict_device(x_dev.data_ptr(), off, labels_dev.data_ptr(), beam_size=BEAM, look_ahead=LOOK_AHEAD,
                         test_iteration=TEST_ITER, stream=stream, engine=args.engine)

  def barrier():
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  for _ in range(args.warmup):
    step_dev()
  barrier()
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  beam_ms, prepass_ms = [], []
  ev0.record()
  for _ in range(args.steps):
    step_dev()
    # stats() synchronises on the step: device-side counters + per-kernel CUDA-event times
    st = model.stats()
    beam_ms.append(st['beam_ms']); prepass_ms.append(st['prepass_ms'])
  ev1.record()
  barrier()
  dev_ms = ev0.elapsed_time(ev1)
  labels_first = labels_dev.cpu().numpy().copy()

  # ---- end-to-end leg (`e2e`): the public API a user calls.  N = 1: uisrnn.UISRNN.predict(list of host float64
  #      arrays) -> list of label lists.  N > 1: uisrnn_b200.distributed.predict_sharded over the job's list (the
  #      partition by frame count; every rank decodes its shard, the labels are gathered to rank 0 as one int32
  #      tensor per rank over NCCL; rank 0 holds the whole ordered result as int32 arrays).  Pinned host inputs; H2D, cast, GEMM, beam search, D2H, the Python list
  #      conversion and (N > 1) the gather of the labels are all inside the timed region.
  sys.path.insert(0, os.path.join(ROOT, 'tests'))
  api_model, iargs = build_api_model(weights, local, torch)
  position = {i: k for k, i in enumerate(mine)}
  lazy = [seqs[position[i]] if i in position else None for i in range(world * U)]

  def step_e2e():
    if world > 1:  # rank 0 receives the merged result (int32 arrays); the other ranks keep their own shard
      return predict_sharded(api_model, lazy, iargs, lengths=lengths, root=0, as_arrays=True)
    return api_model.predict(seqs, iargs)

  for _ in range(max(1, args.warmup // 2)):
    out = step_e2e()
  barrier()
  t0 = time.perf_counter()
  for _ in range(args.steps):
    out = step_e2e()
  torch.cuda.synchronize()
  e2e_s = time.perf_counter() - t0
  clocks = sampler.stop() if rank == 0 else None
  got_mine = [out[i] for i in mine] if world > 1 else out
  assert np.array_equal(np.concatenate([np.asarray(o, dtype=np.int32) for o in got_mine]), labels_first), \
      'e2e and device-resident legs disagree'
  e2e_stats = api_model._native_model().stats()  # pylint: disable=protected-access

  t = torch.tensor([dev_ms, e2e_s * 1e3], dtype=torch.float64, device='cuda')
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  dev_ms, e2e_ms = float(t[0]), float(t[1])
  partition_extra = None
  if not args.no_secondary:
    partition_extra = partition_secondary(api_model, iargs, rank, world, torch, dist, barrier)
  if rank != 0:
    if world > 1:
      dist.destroy_process_group()
    return
  if args.dump_outputs:  # rank 0 holds the whole ordered result of the e2e leg, equal to the device-resident one
    dump_outputs(args.dump_outputs, out)

  # labels of the utterances the unmodified reference decoded (tests/golden/synth500_bench.npz): whichever rank
  # owned them, the merged result of the partitioned run must reproduce them
  golden_checked = golden_ok = 0
  try:
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'synth500_bench.npz'))
    for s, lab in zip(g['seeds'], g['labels']):
      i = int(s) - FIRST_SEED
      if 0 <= i < len(out) and out[i] is not None:
        golden_checked += 1
        golden_ok += int([int(v) for v in out[i]] == [int(v) for v in lab])
  except Exception:  # pylint: disable=broad-except
    pass

  total_frames = frames * world
  value = total_frames * args.steps / (dev_ms / 1e3)
  e2e_value = total_frames * args.steps / (e2e_ms / 1e3)
  H, D = HIDDEN, DIM
  peaks = load_peaks()
  beam_avg_ms = float(np.mean(beam_ms))
  beam_s = beam_avg_ms / 1e3
  sm_mhz = (clocks or {}).get('sm_mhz') or peaks['sm_max_mhz']
  flops = st['gru_columns'] * 2.0 * (3 * H * H + H * H + H * D)   # useful fp32-grade flops of the launch
  fp32_peak = st['ctas'] * 128 * 2 * sm_mhz * 1e6 / 1e12
  engine = st['engine']
  steps_per_launch = TEST_ITER * N_FRAMES
  # SURVEY 8(d): per beam-step "launch" over U utterances: the 6.3 MB weight set once + U * (4*D*L + 8*L) bytes
  hbm_alg = steps_per_launch * (4 * (3 * H * D + 3 * H * H + 6 * H + H * H + H + D * H + D) + U * (4 * D + 8))
  traffic, l2_to_sm = measured_traffic(U, engine)
  wbytes_pass = 4 * (3 * H * H + H * H + H * D)             # W_hh, W1, W2 (fp32, or fp16 hi + lo planes): streamed once per pass
  roof = {
      'kernel': 'uis_beam_kernel<512,256,tensor-core %d columns>' % st['tc_columns'] if engine == 2 else 'uis_beam_kernel<512,256> (FFMA)',
      'kernel_ms': beam_avg_ms,
      'peak_source': peaks['source'],
      'hbm': {'algorithmic_bytes': hbm_alg, 'achieved_gbs': hbm_alg / beam_s / 1e9, 'peak_gbs': peaks['hbm_gbs'],
              'frac': hbm_alg / beam_s / 1e9 / peaks['hbm_gbs'], 'traffic': traffic,
              'note': 'SURVEY 8(d): weights once per beam step + per-frame I/O; the weights stay L2-resident, so this is not '
                      'the binding resource (traffic = ncu dram bytes of the committed capture of this kernel and batch size, '
                      'profiles/r3_traffic.json; null if none matches)'},
      'l2_to_sm_bytes': st['weight_passes'] * wbytes_pass,
      'fp32_fma_equivalent': {'achieved_tflops': flops / beam_s / 1e12, 'peak_tflops': fp32_peak,
                              'frac': flops / beam_s / 1e12 / fp32_peak, 'sm_mhz_used': sm_mhz,
                              'note': 'useful flops (columns x 2.36 MFLOP) over the fp32 FFMA peak SMs*128*2*f: the round-1 '
                                      'yardstick; the tensor-core engine can exceed 1'},
  }
  if engine == 2:
    mma_per_pass = (3 * H + H + D) // 128 * (H // 64) * 2 * 4      # tiles x k atoms x planes x k steps
    np_cols = 2 * st['tc_columns']
    issued = st['weight_passes'] * mma_per_pass * 2.0 * 128 * np_cols * 16
    kernel_cycles = beam_s * sm_mhz * 1e6
    roof.update({
        'bound': 'tensor', 'unit': 'TFLOP/s', 'achieved': flops / beam_s / 1e12, 'peak': peaks['tensor_tflops'],
        'frac': flops / beam_s / 1e12 / peaks['tensor_tflops'], 'traffic': traffic,
        'issued_tflops': issued / beam_s / 1e12,
        'mma_slot': {'mma_per_pass': mma_per_pass, 'floor_cycles_per_mma': MMA_FLOOR_CYCLES,
                     'frac': st['weight_passes'] * mma_per_pass * MMA_FLOOR_CYCLES / (kernel_cycles * st['ctas']),
                     'issuer_us_per_pass': {k: v / (sm_mhz) / max(1, st['weight_passes']) for k, v in zip(
                         ('stall_tma', 'stall_epilogue', 'stall_operand', 'issue'), st['tc_cycles'])},
                     'note': 'share of the kernel the tensor pipe is busy at its measured per-instruction floor: a 128 x N x 16 '
                             'MMA fed from shared memory costs 86.4 cycles for ANY N <= 128 (tools/tc/tc_chain_probe.cu), '
                             'so with <= 48 live columns per pass the pipe is instruction-bound, not flop-bound: `frac` of '
                             'the dense fp16 peak stays small by construction'},
        'note': 'achieved = useful fp32-grade flops (each runs as 4 fp16 products: hi/lo split of both operands, see '
                'issued_tflops for what the pipe executes, padding included); peak = measured dense bf16/fp16 (burst)'})
  else:
    roof.update({'bound': 'fp32_fma', 'unit': 'TFLOP/s', 'achieved': flops / beam_s / 1e12, 'peak': fp32_peak,
                 'frac': flops / beam_s / 1e12 / fp32_peak, 'traffic': traffic})
  out_line = {
      'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': dev_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
      'dtype': 'f32', 'data': 'synthetic',
      'config': {'workload': WORKLOAD, 'utterances_per_gpu_per_step': U, 'frames_per_gpu_per_step': frames,
                 'model': 'D=256 H=512 depth=1, weights = reference fit() 100 it on toy data (tests/golden/model_toy100.npz)',
                 'engine': {1: 'fp32 FFMA kernels', 2: 'tcgen05 tensor-core pass (fp16 hi/lo split operands, fp32-grade)'}[engine],
                 'lanes_per_cta': st['lanes'],
                 'parallelism': 'utterance list of %d x %d sharded by frame count over %d rank(s) (shard_by_frames), '
                                'no data-path collective' % (world, U, world),
                 'l2': 'inputs larger than L2: x %.0f MB + gi %.0f MB rewritten every step' % (
                     frames * D * 4 / 1e6, frames * 3 * H * 4 / 1e6)},
      'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': frames * D * 8 * world, 'd2h_bytes_per_step': frames * 4 * world,
              'engine': e2e_stats['engine'], 'lanes_per_cta': e2e_stats['lanes'],
              'ms_per_step': e2e_ms / args.steps,
              'breakdown_ms_rank0_last_step': {
                  'uis_predict_wall': e2e_stats['host_ms'], 'h2d_copy_stream_span': e2e_stats['h2d_ms'],
                  'cast_and_input_projection_span_overlapped_with_h2d': e2e_stats['pipeline_ms'],
                  'beam_kernel': e2e_stats['beam_ms'], 'staging_chunks': e2e_stats['chunks'],
                  'pinned_staging_by_host_threads': bool(e2e_stats.get('staged', 0)),
                  'python_and_gather': max(0.0, e2e_ms / args.steps - e2e_stats['host_ms'])},
              'path': ('uisrnn_b200.distributed.predict_sharded(UISRNN, list, lengths, root=0, as_arrays=True) -> shard_by_frames -> '
                       'uis_predict() per rank -> dist.gather of one int32 label tensor per rank -> int32 arrays on rank 0'
                       if world > 1 else
                       'uisrnn.UISRNN.predict(list of %s float64 ndarrays) -> uis_predict() C ABI: chunked H2D on a copy stream || ' % ('pageable' if args.pageable else 'pinned') +
                       
                       'cast + input projection, beam kernel, one D2H copy of the int32 labels -> Python lists')},
      'gpu_launches': int(args.steps * 2),
      'clocks': clocks,
      'roofline': roof,
      'kernel_stats': {k: st[k] for k in ('beam_steps', 'gru_columns', 'weight_passes', 'candidates', 'max_k', 'ctas', 'lanes',
                                          'engine', 'tc_columns')},
      'prepass_ms': float(np.mean(prepass_ms)),
      'parity': {'reference_golden_utterances_checked': golden_checked, 'identical': golden_ok,
                 'source': 'tests/golden/synth500_bench.npz (labels of the unmodified reference), compared with the merged '
                           'result of the e2e leg'},
  }
  if world == 1 and not args.no_secondary:
    out_line['secondary'] = secondary_metrics(model, torch)
  if partition_extra:
    out_line.setdefault('secondary', {}).update(partition_extra)
  if world == 1 and not args.no_cpu_baseline:  # reported at N = 1 only (bounded CPU samples, ~1 min)
    try:
      cpu, parity = cpu_baseline_and_parity({U - 1: out[U - 1]})
      out_line['cpu_baseline'] = cpu
      out_line['parity']['oracle'] = parity
      out_line['parity_checked'] = parity['checked'] + golden_checked
    except Exception as err:  # pylint: disable=broad-except
      out_line['cpu_baseline'] = {'error': str(err)[:300]}
  print(json.dumps(out_line), flush=True)
  if world > 1:
    dist.destroy_process_group()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=5)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--utts', type=int, default=888, help='utterances per GPU per step (6 lanes x 148 CTAs)')
  ap.add_argument('--engine', type=int, default=0, help='0 auto (tensor cores), 1 FFMA kernels, 2 tensor cores')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--pageable', action='store_true', help='e2e leg from ordinary (pageable) numpy arrays instead of pinned ones')
  ap.add_argument('--no-secondary', action='store_true', help='skip the config-3 / config-4 side measurements')
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='after the timed steps, write the labels of the last step to DIR/*.npy (e.g. bench_outputs/)')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'b200':
    ap.error('--dump-outputs applies to --impl b200 (the reference arm decodes slices sized by a timing calibration)')
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_b200(args)


if __name__ == '__main__':
  main()
