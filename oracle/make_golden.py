#!/usr/bin/env python3
"""Generate the golden fixtures under tests/golden/ by RUNNING THE UNMODIFIED REFERENCE.

TEST INFRASTRUCTURE ONLY (see oracle/README.md).  This script runs only where a checkout of
the reference exists (located as in oracle/build_ref.py); the tests never run it.  It imports the
reference package from that checkout (plus the logging shim oracle/shims/colortimelog),
trains the fixture models with the reference's own fit(), runs the reference's own
predict_single() and, for a few utterances, drives the reference's own
`_calculate_score` / `_update_beam_state` (uisrnn/uisrnn.py:388-477) step by step to record
per-step ranked scores and winners.  Nothing here is a re-implementation of the arithmetic:
every number written to tests/golden/ was produced by reference code.

Fixtures written (all float32 where the reference computes in float32):
  model_toy100.npz   default-size model (D=256,H=512,depth=1): reference fit(), seeds 0,
                     100 iterations on data/toy_training_data.npz
  toy_test.npz       the 25 toy test utterances (as float32: the reference casts to float32
                     before any arithmetic, uisrnn.py:525-526) + reference labels
  toy_trace.npz      per-step trace of toy utterances 0 and 1
  synth500.npz       two 500-frame synthetic utterances (seeds 1000, 1001): reference labels
  model_small.npz    D=64,H=128 model trained by the reference on synthetic data
  model_small_d2.npz, depth2_cases.npz   the same with rnn_depth=2
  small_cases.npz    small-model cases: beam/look_ahead/test_iteration variants, traces
  ref_checkpoint.uisrnn, ref_checkpoint_cases.npz   a file written by the reference's save() (D=8, H=16)
                     and the reference's predictions with that model
  synth500_bench.npz reference labels of ten utterances of bench.py's workload (seeds 100000 + {0..5, 147, 148, 294, 295})
  small500.npz       reference labels of four 500-frame utterances with the D=64/H=128 model
  fit_traj.npz       the reference's fit(): three loss terms of 20 iterations + initial / final parameters
                     (depth 1 batch 16, depth 1 batch 48, depth 2 without dropout)
Usage:  python oracle/make_golden.py [--only NAME] [--jobs 8]
"""
import argparse
import importlib.util
import os
import random
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, HERE)
from build_ref import SOURCE as REF  # noqa: E402
GOLD = os.path.join(REPO, 'tests', 'golden')
CACHE = '/tmp/uis_golden_cache'

sys.path[:0] = [os.path.join(HERE, 'shims'), REF]
sys.argv_saved = sys.argv
import numpy as np  # noqa: E402
import torch  # noqa: E402
import uisrnn as ref  # noqa: E402  (the reference package)
from uisrnn import uisrnn as ref_mod  # noqa: E402

assert ref.__file__.startswith(REF), ref.__file__

_spec = importlib.util.spec_from_file_location(
    'synth', os.path.join(REPO, 'uisrnn_b200', 'synth.py'))
synth = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(synth)


def ref_args(**over):
  argv, sys.argv = sys.argv, [sys.argv[0]]
  try:
    m, t, i = ref.parse_arguments()
  finally:
    sys.argv = argv
  m.enable_cuda = False
  m.verbosity = 2
  for k, v in over.items():
    for ns in (m, t, i):
      if hasattr(ns, k):
        setattr(ns, k, v)
        break
    else:
      raise KeyError(k)
  return m, t, i


def seed_all(s):
  np.random.seed(s)
  random.seed(s)
  torch.manual_seed(s)


def model_to_dict(model):
  sd = model.rnn_model.state_dict()
  depth = model.rnn_init_hidden.shape[0]
  out = {
      'depth': np.int64(depth),
      'w1': sd['linear_mean1.weight'].numpy(), 'b1': sd['linear_mean1.bias'].numpy(),
      'w2': sd['linear_mean2.weight'].numpy(), 'b2': sd['linear_mean2.bias'].numpy(),
      'h0': model.rnn_init_hidden.detach().numpy(),
      'sigma2': model.sigma2.detach().numpy(),
      'transition_bias': np.float64(model.transition_bias),
      'transition_bias_denominator': np.float64(model.transition_bias_denominator),
      'crp_alpha': np.float64(model.crp_alpha),
  }
  for l in range(depth):
    for nm in ('weight_ih', 'weight_hh', 'bias_ih', 'bias_hh'):
      out['{}_l{}'.format(nm, l)] = sd['gru.{}_l{}'.format(nm, l)].numpy()
  return {k: (np.ascontiguousarray(v, dtype=np.float32)
              if isinstance(v, np.ndarray) and v.dtype.kind == 'f' and v.ndim > 0 else v)
          for k, v in out.items()}


def model_from_dict(d, **over):
  depth = int(d['depth'])
  H = d['w1'].shape[0]
  D = d['w2'].shape[0]
  m, _, _ = ref_args(observation_dim=D, rnn_hidden_size=H, rnn_depth=depth,
                     transition_bias=float(d['transition_bias']),
                     crp_alpha=float(d['crp_alpha']), **over)
  model = ref.UISRNN(m)
  sd = {'linear_mean1.weight': d['w1'], 'linear_mean1.bias': d['b1'],
        'linear_mean2.weight': d['w2'], 'linear_mean2.bias': d['b2']}
  for l in range(depth):
    for nm in ('weight_ih', 'weight_hh', 'bias_ih', 'bias_hh'):
      sd['gru.{}_l{}'.format(nm, l)] = d['{}_l{}'.format(nm, l)]
  model.rnn_model.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
  model.rnn_init_hidden = torch.nn.Parameter(torch.from_numpy(np.array(d['h0'])))
  model.sigma2 = torch.nn.Parameter(torch.from_numpy(np.array(d['sigma2'])))
  model.transition_bias = float(d['transition_bias'])
  model.transition_bias_denominator = float(d['transition_bias_denominator'])
  return model


def traced_predict(model, seq, iargs):
  """Drive the reference's own per-step methods and record what they return.

  The control flow mirrors predict_single (uisrnn.py:523-561); every score and state
  update comes from model._calculate_score / model._update_beam_state (reference code).
  """
  model.rnn_model.eval()
  n = seq.shape[0]
  tiled = torch.from_numpy(np.tile(seq, (iargs.test_iteration, 1))).float()
  beams = [ref_mod.BeamState()]
  rec = {'win': [], 'score': [], 'off': [0], 'ncand': [], 'nfinite': []}
  for t in range(0, iargs.test_iteration * n, iargs.look_ahead):
    chunk = tiled[t:t + iargs.look_ahead, :]
    la = chunk.shape[0]
    kmax = max(len(b.mean_set) for b in beams)
    table = np.full([iargs.beam_size] + [kmax + 1 + i for i in range(la)], np.inf)
    for r, b in enumerate(beams):
      s = model._calculate_score(b, chunk)
      table[r] = np.pad(s, [(0, kmax - len(b.mean_set))] * la, 'constant',
                        constant_values=np.inf)
    ranked = np.sort(table, axis=None)
    ranked[ranked == np.inf] = 0
    ranked = np.trim_zeros(ranked)
    order = np.argsort(table, axis=None)
    keep = min(len(ranked), iargs.beam_size)
    new_beams = []
    for r in range(keep):
      idx = np.unravel_index(order[r], table.shape)
      new_beams.append(model._update_beam_state(beams[idx[0].item()], chunk, idx[1:]))
      rec['win'].append([int(v) for v in idx] + [-1] * (iargs.look_ahead - la))
      rec['score'].append(float(new_beams[-1].neg_likelihood))
    rec['off'].append(len(rec['win']))
    rec['ncand'].append(int(np.isfinite(table).sum()))
    rec['nfinite'].append(len(ranked))
    beams = new_beams
  best = beams[0]
  out = {
      'labels': np.array(best.trace[-n:], dtype=np.int64),
      'win': np.array(rec['win'], dtype=np.int32),
      'score': np.array(rec['score'], dtype=np.float64),
      'off': np.array(rec['off'], dtype=np.int64),
      'nfinite': np.array(rec['nfinite'], dtype=np.int64),
      'final_scores': np.array([float(b.neg_likelihood) for b in beams], dtype=np.float64),
      'final_mean': np.stack([m.detach().numpy().reshape(-1) for m in best.mean_set]),
      'final_hidden': np.stack([h.detach().numpy().reshape(h.shape[0], -1)
                                for h in best.hidden_set]),
      'final_blocks': np.array(best.block_counts, dtype=np.int64),
      'full_trace': np.array(best.trace, dtype=np.int64),
  }
  return out


def _predict_worker(job):
  d, seq, ikw = job
  torch.set_num_threads(1)
  model = model_from_dict(d)
  _, _, ia = ref_args(**ikw)
  t0 = time.time()
  lab = model.predict_single(seq.astype(np.float64), ia)
  return np.array(lab, dtype=np.int64), time.time() - t0


def _trace_worker(job):
  d, seq, ikw = job
  torch.set_num_threads(1)
  model = model_from_dict(d)
  _, _, ia = ref_args(**ikw)
  return traced_predict(model, seq.astype(np.float64), ia)


def pmap(fn, jobs, nproc):
  import multiprocessing as mp
  ctx = mp.get_context('fork')
  with ctx.Pool(min(nproc, max(1, len(jobs)))) as pool:
    return pool.map(fn, jobs, chunksize=1)


def flatten_traces(prefix, traces, out):
  for i, tr in enumerate(traces):
    for k, v in tr.items():
      out['{}{}_{}'.format(prefix, i, k)] = v


# --------------------------------------------------------------------------- fixtures

def make_model_toy100():
  path = os.path.join(GOLD, 'model_toy100.npz')
  seed_all(0)
  m, t, _ = ref_args(train_iteration=100)
  train = np.load(os.path.join(REF, 'data', 'toy_training_data.npz'), allow_pickle=True)
  model = ref.UISRNN(m)
  t0 = time.time()
  model.fit(train['train_sequence'], train['train_cluster_id'], t)
  print('reference fit(toy, 100 it): %.1fs, transition_bias=%.6f sigma2[:3]=%s'
        % (time.time() - t0, model.transition_bias, model.sigma2.detach().numpy()[:3]))
  np.savez(path, **model_to_dict(model))
  return path


def make_toy_test(jobs):
  d = dict(np.load(os.path.join(GOLD, 'model_toy100.npz')))
  test = np.load(os.path.join(REF, 'data', 'toy_testing_data.npz'), allow_pickle=True)
  seqs = [np.asarray(s, dtype=np.float64) for s in test['test_sequences'].tolist()]
  truth = test['test_cluster_ids'].tolist()
  res = pmap(_predict_worker, [(d, s, {}) for s in seqs], jobs)
  out = {'n_utt': np.int64(len(seqs)),
         'lengths': np.array([len(s) for s in seqs], dtype=np.int64),
         'x': np.concatenate(seqs).astype(np.float32),
         'labels': np.concatenate([r[0] for r in res]),
         'ref_seconds': np.array([r[1] for r in res])}
  # ground-truth ids factorised to ints (for accuracy checks only)
  gt = []
  for ids in truth:
    m = {}
    gt.append(np.array([m.setdefault(s, len(m)) for s in ids], dtype=np.int64))
  out['truth'] = np.concatenate(gt)
  assert np.array_equal(out['x'].astype(np.float64).astype(np.float32), out['x'])
  np.savez_compressed(os.path.join(GOLD, 'toy_test.npz'), **out)
  print('toy_test: ref frames/s per process = %.2f'
        % (out['lengths'].sum() / out['ref_seconds'].sum()))
  # traces of utterances 0 and 1 (these also re-check traced_predict == predict_single)
  trs = pmap(_trace_worker, [(d, seqs[i], {}) for i in (0, 1)], jobs)
  off = np.concatenate([[0], np.cumsum(out['lengths'])])
  for i, tr in enumerate(trs):
    assert np.array_equal(tr['labels'], out['labels'][off[i]:off[i + 1]]), 'trace != predict'
  o = {}
  flatten_traces('u', trs, o)
  np.savez_compressed(os.path.join(GOLD, 'toy_trace.npz'), **o)


def make_synth500(jobs):
  d = dict(np.load(os.path.join(GOLD, 'model_toy100.npz')))
  seeds = [1000, 1001]
  seqs = [synth.synth_utt(s)[0] for s in seeds]
  res = pmap(_predict_worker, [(d, s, {}) for s in seqs], jobs)
  np.savez_compressed(
      os.path.join(GOLD, 'synth500.npz'), seeds=np.array(seeds),
      labels=np.stack([r[0] for r in res]), ref_seconds=np.array([r[1] for r in res]))
  print('synth500 ref seconds', [r[1] for r in res])


def make_model_small():
  seed_all(7)
  m, t, _ = ref_args(observation_dim=64, rnn_hidden_size=128, train_iteration=300,
                     learning_rate=2e-3, batch_size=16)
  seqs, ids = synth.synth_training_set(5000, 80, n_frames=80, dim=64, n_spk=3, noise=0.08)
  model = ref.UISRNN(m)
  model.fit(seqs, ids, t)
  print('small model: transition_bias=%.5f sigma2 mean=%.5f'
        % (model.transition_bias, float(model.sigma2.mean())))
  np.savez(os.path.join(GOLD, 'model_small.npz'), **model_to_dict(model))


SMALL_CASES = [
    # name, seed, n_frames, n_spk, inference kwargs
    ('b10', 6001, 90, 3, dict(beam_size=10, look_ahead=1, test_iteration=2)),
    ('b3', 6002, 70, 4, dict(beam_size=3, look_ahead=1, test_iteration=1)),
    ('b1', 6003, 50, 2, dict(beam_size=1, look_ahead=1, test_iteration=3)),
    ('b30', 6004, 60, 4, dict(beam_size=30, look_ahead=1, test_iteration=2)),
    ('one', 6005, 1, 1, dict(beam_size=10, look_ahead=1, test_iteration=2)),
    ('la2', 6006, 41, 3, dict(beam_size=5, look_ahead=2, test_iteration=1)),
    ('la2b', 6007, 30, 3, dict(beam_size=10, look_ahead=2, test_iteration=2)),
    ('la3', 6008, 20, 2, dict(beam_size=4, look_ahead=3, test_iteration=1)),
]


def make_small_cases(jobs):
  d = dict(np.load(os.path.join(GOLD, 'model_small.npz')))
  seqs = [synth.synth_utt(s, n_frames=n, dim=64, n_spk=k, noise=0.08)[0]
          for (_, s, n, k, _) in SMALL_CASES]
  trs = pmap(_trace_worker, [(d, x, kw) for x, (_, _, _, _, kw) in zip(seqs, SMALL_CASES)],
             jobs)
  o = {'names': np.array([c[0] for c in SMALL_CASES])}
  for (name, seed, n, k, kw), x, tr in zip(SMALL_CASES, seqs, trs):
    o[name + '_x'] = x.astype(np.float32)
    o[name + '_args'] = np.array([kw['beam_size'], kw['look_ahead'], kw['test_iteration']])
    for key, v in tr.items():
      o['{}_{}'.format(name, key)] = v
    print(name, 'labels', tr['labels'][:40])
  np.savez_compressed(os.path.join(GOLD, 'small_cases.npz'), **o)


def make_model_small_d2():
  """Depth-2 GRU (nn.GRU with inter-layer dropout in training), D=64, H=128."""
  seed_all(9)
  m, t, _ = ref_args(observation_dim=64, rnn_hidden_size=128, rnn_depth=2, train_iteration=300,
                     learning_rate=2e-3, batch_size=16)
  seqs, ids = synth.synth_training_set(5200, 80, n_frames=80, dim=64, n_spk=3, noise=0.08)
  model = ref.UISRNN(m)
  model.fit(seqs, ids, t)
  np.savez(os.path.join(GOLD, 'model_small_d2.npz'), **model_to_dict(model))


DEPTH2_CASES = [
    ('d2_b10', 6101, 70, 3, dict(beam_size=10, look_ahead=1, test_iteration=2)),
    ('d2_la2', 6102, 33, 3, dict(beam_size=5, look_ahead=2, test_iteration=1)),
]


def make_depth2_cases(jobs):
  d = dict(np.load(os.path.join(GOLD, 'model_small_d2.npz')))
  seqs = [synth.synth_utt(s, n_frames=n, dim=64, n_spk=k, noise=0.08)[0] for (_, s, n, k, _) in DEPTH2_CASES]
  trs = pmap(_trace_worker, [(d, x, kw) for x, (_, _, _, _, kw) in zip(seqs, DEPTH2_CASES)], jobs)
  o = {'names': np.array([c[0] for c in DEPTH2_CASES])}
  for (name, seed, n, k, kw), x, tr in zip(DEPTH2_CASES, seqs, trs):
    o[name + '_x'] = x.astype(np.float32)
    o[name + '_args'] = np.array([kw['beam_size'], kw['look_ahead'], kw['test_iteration']])
    for key, v in tr.items():
      o['{}_{}'.format(name, key)] = v
    print(name, 'labels', tr['labels'][:40])
  np.savez_compressed(os.path.join(GOLD, 'depth2_cases.npz'), **o)


def make_ref_checkpoint():
  """A checkpoint written by the reference's own save() (uisrnn.py:135-147) + what the reference predicts
  with that model: pins the file format both ways (SURVEY 8(f) f2)."""
  seed_all(11)
  m, t, i = ref_args(observation_dim=8, rnn_hidden_size=16, train_iteration=400, learning_rate=1e-2,
                     batch_size=8)
  seqs, ids = synth.synth_training_set(5400, 30, n_frames=40, dim=8, n_spk=2, noise=0.05)
  model = ref.UISRNN(m)
  model.fit(seqs, ids, t)
  model.save(os.path.join(GOLD, 'ref_checkpoint.uisrnn'))
  i.beam_size, i.look_ahead, i.test_iteration = 5, 1, 2
  xs = [synth.synth_utt(5500 + k, n_frames=30, dim=8, n_spk=2, noise=0.05)[0] for k in range(2)]
  labels = [np.array(model.predict_single(x, i)) for x in xs]
  np.savez(os.path.join(GOLD, 'ref_checkpoint_cases.npz'), x0=xs[0], x1=xs[1], labels0=labels[0],
           labels1=labels[1], transition_bias=model.transition_bias,
           transition_bias_denominator=model.transition_bias_denominator)
  print('ref checkpoint labels', labels[0][:20], labels[1][:20])


def make_synth500_bench(jobs):
  """Reference labels for the first utterances of bench.py's own workload (seeds 100000 + u, config 2 shape):
  pins the kernel variant the bench times (2 lanes, one CTA per lane group) at the full 1000 beam steps."""
  d = dict(np.load(os.path.join(GOLD, 'model_toy100.npz')))
  seeds = [100000 + u for u in (0, 1, 2, 3, 4, 5, 147, 148, 294, 295)]  # first / median / last of bench.py's 296
  seqs = [synth.synth_utt(s)[0] for s in seeds]
  res = pmap(_predict_worker, [(d, s, {}) for s in seqs], jobs)
  np.savez_compressed(
      os.path.join(GOLD, 'synth500_bench.npz'), seeds=np.array(seeds),
      labels=np.stack([r[0] for r in res]), ref_seconds=np.array([r[1] for r in res]))
  print('synth500_bench ref seconds', [r[1] for r in res])


def make_small500(jobs):
  """D=64 / H=128 model on four 500-frame utterances: the long-utterance pin for the small kernel shape."""
  d = dict(np.load(os.path.join(GOLD, 'model_small.npz')))
  seeds = [7000 + u for u in range(4)]
  seqs = [synth.synth_utt(s, n_frames=500, dim=64, n_spk=4, noise=0.08)[0] for s in seeds]
  res = pmap(_predict_worker, [(d, s, {}) for s in seqs], jobs)
  np.savez_compressed(
      os.path.join(GOLD, 'small500.npz'), seeds=np.array(seeds),
      labels=np.stack([r[0] for r in res]), ref_seconds=np.array([r[1] for r in res]))
  print('small500 ref seconds', [r[1] for r in res])


FIT_TRAJ_CASES = [
    # name, seed, model kwargs, training kwargs
    ('d1_b16', 21, dict(), dict(batch_size=16)),
    ('d1_b48', 22, dict(), dict(batch_size=48)),
    ('d2_b16', 23, dict(rnn_depth=2, rnn_dropout=0.0), dict(batch_size=16)),
]


def make_fit_traj():
  """Loss trajectory of the reference's own fit() (uisrnn.py:172-313, 315-386): 20 iterations, D=64 / H=128.
  The three loss terms of every iteration are recorded by wrapping (not replacing) the reference's
  loss_func functions; initial and final parameters are stored so that the repo's fit() can be started from
  the same point and compared (SURVEY 8(d) config 4: "loss1 trajectory vs oracle with identical RNG stream")."""
  from uisrnn import loss_func as ref_loss
  out = {'names': np.array([c[0] for c in FIT_TRAJ_CASES])}
  for name, seed, mkw, tkw in FIT_TRAJ_CASES:
    seed_all(seed)
    m, t, _ = ref_args(observation_dim=64, rnn_hidden_size=128, train_iteration=20, learning_rate=1e-3,
                       num_permutations=4, **mkw, **tkw)
    seqs, ids = synth.synth_training_set(7100 + seed, 40, n_frames=60, dim=64, n_spk=3, noise=0.08)
    model = ref.UISRNN(m)
    init = model_to_dict_partial(model)
    rec = {'l1': [], 'l2': [], 'l3': []}
    orig = (ref_loss.weighted_mse_loss, ref_loss.sigma2_prior_loss, ref_loss.regularization_loss)

    def wrap(fn, key):
      def inner(*a, **k):
        v = fn(*a, **k)
        rec[key].append(float(v.detach()))
        return v
      return inner
    ref_loss.weighted_mse_loss = wrap(orig[0], 'l1')
    ref_loss.sigma2_prior_loss = wrap(orig[1], 'l2')
    ref_loss.regularization_loss = wrap(orig[2], 'l3')
    try:
      seed_all(seed + 1000)   # the RNG state fit() starts from (shuffle, permutations, batch draws)
      model.fit(seqs, ids, t)
    finally:
      ref_loss.weighted_mse_loss, ref_loss.sigma2_prior_loss, ref_loss.regularization_loss = orig
    final = model_to_dict(model)
    assert len(rec['l1']) == 20
    out[name + '_args'] = np.array([seed, int(mkw.get('rnn_depth', 1)), tkw['batch_size']])
    out[name + '_losses'] = np.array([rec['l1'], rec['l2'], rec['l3']], dtype=np.float64).T
    for k, v in init.items():
      out['{}_init_{}'.format(name, k)] = v
    for k, v in final.items():
      out['{}_final_{}'.format(name, k)] = v
    print(name, 'loss1', rec['l1'][:3], '...', rec['l1'][-1], 'transition_bias', model.transition_bias)
  np.savez_compressed(os.path.join(GOLD, 'fit_traj.npz'), **out)


def model_to_dict_partial(model):
  """model_to_dict for a model whose transition_bias is still None (before fit)."""
  tb, model.transition_bias = model.transition_bias, 0.5
  try:
    d = model_to_dict(model)
  finally:
    model.transition_bias = tb
  d.pop('transition_bias')
  return {k: np.array(v) for k, v in d.items()}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--only', default=None)
  ap.add_argument('--jobs', type=int, default=8)
  a = ap.parse_args()
  os.makedirs(GOLD, exist_ok=True)
  steps = [('model_toy100', make_model_toy100), ('toy_test', lambda: make_toy_test(a.jobs)),
           ('synth500', lambda: make_synth500(a.jobs)), ('model_small', make_model_small),
           ('small_cases', lambda: make_small_cases(a.jobs)), ('model_small_d2', make_model_small_d2),
           ('depth2_cases', lambda: make_depth2_cases(a.jobs)), ('ref_checkpoint', make_ref_checkpoint),
           ('synth500_bench', lambda: make_synth500_bench(a.jobs)), ('small500', lambda: make_small500(a.jobs)),
           ('fit_traj', make_fit_traj)]
  for name, fn in steps:
    if a.only and name not in a.only.split(','):
      continue
    t0 = time.time()
    fn()
    print('== %s done in %.1fs' % (name, time.time() - t0), flush=True)


if __name__ == '__main__':
  main()
