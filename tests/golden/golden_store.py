"""Compact storage of the reference golden vectors (tests/golden/reference_*.npz), small enough to keep in git.

A golden set is a dict {key: ndarray} whose keys read '<case>/<kind>/...'.  `save` writes it as one .npz of three
members (a JSON index and a float64 and a float32 blob), where
  * the inputs the generator drew from a seeded torch generator are not stored: '<case>/rng_stream' lists the seed and
    the draws in order, and `load` replays them and checks each against its stored float64 sum;
  * large result tensors (gradients, end points, outputs) are stored as a `Sample`: max |x|, sum and L2 norm of the whole
    tensor and a fixed subset of its elements;
  * every other array (names, shapes, losses, normaliser state, ...) is stored whole.
`load` returns an object that is indexed like the np.load() of the full dict and has its `.files`.
"""
import json
import math

import numpy as np
import torch

SAMPLED_KINDS = ('grad', 'grad_in', 'ep', 'ep_s', 'gep_s', 'dep', 'out', 'infer')
SAMPLE_SIZE = 32


def sample_indices(n, m=SAMPLE_SIZE):
  """m distinct flat indices spread over a tensor of n elements (2654435761 is prime, so i * it mod n repeats no index)."""
  if n <= m:
    return np.arange(n, dtype=np.int64)
  return (np.arange(m, dtype=np.int64) * 2654435761) % n


def _stats(a):
  a = np.asarray(a, dtype=np.float64).ravel()
  return [float(np.abs(a).max()) if a.size else 0.0, float(a.sum()), float(np.sqrt((a * a).sum()))]


class Sample(object):
  """A golden tensor of which max |x|, sum and L2 norm and the elements at `sample_indices` were kept."""

  def __init__(self, shape, values, absmax, total, l2):
    self.shape, self.values = tuple(shape), np.asarray(values, dtype=np.float64)
    self.absmax, self.total, self.l2 = absmax, total, l2

  def rel(self, mine):
    """A lower bound of max |mine - ref| / max |ref| over the whole tensor: each of the four terms is at most that value,
    so `rel(mine) < tol` holds whenever the comparison with the full tensor would hold."""
    if isinstance(mine, torch.Tensor):
      mine = mine.detach().to('cpu', torch.float64).numpy()
    a = np.asarray(mine, dtype=np.float64)
    if tuple(a.shape) != self.shape:
      return math.inf
    a = a.ravel()
    n, d = a.size, max(self.absmax, 1e-300)
    absmax, total, l2 = _stats(a)
    return max(float(np.abs(a[sample_indices(n)] - self.values).max()) / d if n else 0.0,
               abs(absmax - self.absmax) / d,
               abs(l2 - self.l2) / (math.sqrt(n) * d),
               abs(total - self.total) / (n * d))


def _replay(stream):
  """{key: array} of the draws of one seeded generator, in the order the generator made them."""
  g = torch.Generator().manual_seed(int(stream['seed']))
  out = {}
  for key, kind, shape in stream['draws']:
    fn = {'rand': torch.rand, 'randn': torch.randn}[kind]
    out[key] = fn(tuple(shape), generator=g, dtype=torch.float64).numpy()
  return out


def save(path, arrays):
  """Write `arrays` (the full golden dict) to `path` in the compact form described above."""
  index, blobs = {}, {'f64': [], 'f32': []}
  offsets = {'f64': 0, 'f32': 0}
  replayed = {}
  for key in arrays:
    if key.endswith('/rng_stream'):
      for k, v in _replay(json.loads(str(arrays[key]))).items():
        assert k in arrays and np.array_equal(v, arrays[k]), ('the seeded draws do not reproduce', k)
        replayed[k] = key

  def put(blob, a):
    o = offsets[blob]
    blobs[blob].append(a.ravel())
    offsets[blob] += a.size
    return o

  for key, a in arrays.items():
    a = np.asarray(a)
    kind = key.split('/')[1] if key.count('/') >= 2 else ''
    if key in replayed:
      index[key] = {'rng': replayed[key], 'sum': float(a.sum())}
    elif a.dtype.kind != 'f':
      index[key] = {'json': a.tolist(), 'dtype': a.dtype.str, 'shape': list(a.shape)}
    else:
      blob = 'f32' if a.dtype == np.float32 else 'f64'
      if kind in SAMPLED_KINDS and a.size > SAMPLE_SIZE:
        vals = a.ravel()[sample_indices(a.size)].astype(np.float32 if blob == 'f32' else np.float64)
        index[key] = {'sample': put(blob, vals), 'blob': blob, 'shape': list(a.shape), 'stats': _stats(a)}
      else:
        index[key] = {'off': put(blob, a.astype(np.float32 if blob == 'f32' else np.float64)), 'blob': blob,
                      'shape': list(a.shape)}
  cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)
  np.savez_compressed(path, index=np.array(json.dumps(index)), f64=cat(blobs['f64'], np.float64),
                      f32=cat(blobs['f32'], np.float32))


class Golden(object):
  """The golden dict of one file: `z[key]` is an ndarray, or a `Sample` for the sampled result tensors."""

  def __init__(self, path):
    z = np.load(path)
    self._index = json.loads(str(z['index']))
    self._blobs = {'f64': z['f64'], 'f32': z['f32']}
    self.files = list(self._index)
    self._replayed = {}

  def __contains__(self, key):
    return key in self._index

  def __getitem__(self, key):
    e = self._index[key]
    if 'rng' in e:
      if e['rng'] not in self._replayed:
        self._replayed[e['rng']] = _replay(json.loads(str(self[e['rng']])))
      a = self._replayed[e['rng']][key]
      assert abs(float(a.sum()) - e['sum']) <= 1e-12 * max(1.0, abs(e['sum'])), \
          ('torch.Generator no longer reproduces the stored draw', key)
      return a
    if 'json' in e:
      return np.array(e['json'], dtype=np.dtype(e['dtype'])).reshape(e['shape'])
    blob = self._blobs[e['blob']]
    if 'sample' in e:
      o, n = e['sample'], len(sample_indices(math.prod(e['shape'])))
      return Sample(e['shape'], blob[o:o + n], *e['stats'])
    o = e['off']
    return blob[o:o + math.prod(e['shape'])].reshape(e['shape'])


def load(path):
  return Golden(path)
