"""Instance-by-instance parity of the convolution kernels: every case of tests/conv_coverage.py runs through its C-ABI entry
point on seeded operands, the kernel that actually launched (torch.profiler) must be the table's instance, and every output
is compared with an fp64 convolution computed on the GPU by torch (never through libtwg) at the per-kernel bar: rel_err
(max |a - b| / max |b|) < 1e-4 on the split-bf16 tensor-core path, < 2e-5 on the exact-fp32 kernels.

The operands carry per-image and per-channel offsets and the 3x3 weights a tap-dependent ramp, so an image swap, a
channel permutation, a tap flip or a lost edge row each move the result by far more than the bar; every case also checks
that against fp64 references with exactly those errors (sensitivity controls: >= 100x the bar).

test_step_convs_replayed_against_fp64 records the convolution calls of the benchmarked training step (BASELINE configs[3])
and of the 64-image inference (configs[4]) and replays every distinct one the same way."""
import math

import pytest
import torch
import torch.nn.functional as F

from tests.conv_coverage import COVERAGE, DEFAULT_OPTIONS, TOL, canonical

pytestmark = pytest.mark.gpu

DEV = 'cuda:0'
CONTROL_FACTOR = 100.0
REPORT = {}          # instance -> (cases, worst rel_err, worst control margin)


@pytest.fixture
def lib_options(built_lib):
  """Applies a case's twg_set_option overrides; the library defaults are restored afterwards whatever happens (the
  options are write-only, so the defaults are written back explicitly)."""
  def apply(opts):
    for k, v in DEFAULT_OPTIONS.items():
      built_lib.call('twg_set_option', k, opts.get(k, v))
  try:
    yield apply
  finally:
    for k, v in DEFAULT_OPTIONS.items():
      built_lib.call('twg_set_option', k, v)


# ---- fp64 references (torch on the GPU, NHWC <-> NCHW) --------------------------------------------------------------------

def _nchw(t):
  return t.permute(0, 3, 1, 2)


def _nhwc(t):
  return t.permute(0, 2, 3, 1).contiguous()


def ref_fwd(x, w, pad):
  return _nhwc(F.conv2d(_nchw(x), w.permute(3, 2, 0, 1), padding=pad))


def ref_dgrad(gy, w, x_shape, pad):
  N, H, W, Ci = x_shape
  return _nhwc(torch.nn.grad.conv2d_input((N, Ci, H, W), w.permute(3, 2, 0, 1), _nchw(gy), padding=pad))


def ref_wgrad(x, gy, k, pad):
  Ci, Co = x.shape[3], gy.shape[3]
  return torch.nn.grad.conv2d_weight(_nchw(x), (Co, Ci, k, k), _nchw(gy), padding=pad).permute(2, 3, 1, 0).contiguous()


def ref_epilogue(y, epi, bias, aff):
  """bias + leaky-ReLU (discriminator layer) or the evaluation-mode affine + leaky-ReLU + pixel norm (inference layer)."""
  lrelu, pix = epi.get('lrelu', 1), 0
  if aff is not None:
    t = aff * y + bias
    lrelu, pix = epi['flags'] & 1, epi['flags'] & 2
  else:
    t = y + bias
  if lrelu:
    t = torch.maximum(0.2 * t, t)
  if pix:
    t = t / torch.sqrt((t * t).mean(dim=3, keepdim=True) + 1e-6)
  return t


# ---- seeded operands ----------------------------------------------------------------------------------------------------

def _act(shape, g, offsets=True):
  t = torch.randn(shape, device=DEV, dtype=torch.float64, generator=g)
  if offsets:       # per-image and per-channel offsets: an image swap or a channel permutation changes the mean
    t = t + 0.5 * torch.randn((shape[0], 1, 1, 1), device=DEV, dtype=torch.float64, generator=g)
    t = t + 0.5 * torch.randn((1, 1, 1, shape[3]), device=DEV, dtype=torch.float64, generator=g)
  return t


def _weights(k, ci, co, g):
  s = 1.0 / math.sqrt(k * k * ci)
  w = torch.randn((k, k, ci, co), device=DEV, dtype=torch.float64, generator=g) * s
  ramp = torch.linspace(-1.0, 1.0, k * k, device=DEV, dtype=torch.float64).view(k, k, 1, 1)
  return w + 0.5 * s * ramp          # tap-dependent: a flipped or transposed kernel is visibly different


def _f32(t):
  return t.to(torch.float32).contiguous()


def _q(t):
  """The fp32 value the kernel sees, as fp64 for the reference."""
  return t.to(torch.float32).to(torch.float64)


def _split(L, x32):
  planes = torch.empty((2,) + tuple(x32.shape), device=DEV, dtype=torch.bfloat16)
  L.call('twg_split_act', x32.data_ptr(), planes.data_ptr(), x32.numel(), 0)
  return planes


def _wplanes(L, w32, dgrad):
  k, _, ci, co = w32.shape
  planes = torch.empty((2, k * k * ci * co), device=DEV, dtype=torch.bfloat16)
  L.call('twg_split_weights', w32.data_ptr(), planes.data_ptr(), k, ci, co, int(dgrad), 0)
  return planes


def _planes_value(p, shape):
  return (p[0].double() + p[1].double()).view(shape)


def rel_err(a, b):
  a, b = a.double(), b.double()
  d = float(b.abs().max())
  e = float((a - b).abs().max())
  return e / d if d > 0 else e


# ---- one case -------------------------------------------------------------------------------------------------------------

class Run:
  """Operands, the library call and the fp64 reference of one case."""

  def __init__(self, L, case, seed):
    self.L, self.case = L, case
    entry, (N, H, W, Ci, Co, k, pad), epi = case.entry, case.geom, case.epi
    self.Ho, self.Wo = H + 2 * pad - k + 1, W + 2 * pad - k + 1
    g = torch.Generator(device=DEV).manual_seed(seed)
    self.x = _q(_act((N, H, W, Ci), g) + epi.get('offset', 0.0))
    self.w = _q(_weights(k, Ci, Co, g) + (0.02 if epi.get('offset') else 0.0))
    wgrad = entry in ('wgrad', 'wgrad_planes')
    # the weight gradient's gy is zero-mean: offsets on both operands would make gw mostly a tap-symmetric sum
    self.gy = _q(_act((N, self.Ho, self.Wo, Co), g, offsets=not wgrad))
    self.bias = _q(0.1 * torch.randn(Co, device=DEV, dtype=torch.float64, generator=g))
    self.aff = _q(0.5 + torch.rand(Co, device=DEV, dtype=torch.float64, generator=g)) if entry == 'affine' else None
    self.prefill = _q(torch.randn((k, k, Ci, Co), device=DEV, dtype=torch.float64, generator=g)) \
        if wgrad and epi.get('accumulate') else None

  # the library call; returns {output name: tensor}
  def launch(self):
    L, c = self.L, self.case
    N, H, W, Ci, Co, k, pad = c.geom
    geom = (N, H, W, Ci, Co, k, pad)
    e, epi = c.entry, c.epi
    out = {}
    if e in ('fwd', 'dgrad', 'wgrad'):
      prec = epi['prec']
      nb = int(L.cdll.twg_conv_workspace_bytes(*geom, prec))
      ws = torch.empty(max(nb, 1), device=DEV, dtype=torch.uint8)
      if e == 'fwd':
        y = torch.empty((N, self.Ho, self.Wo, Co), device=DEV)
        L.call('twg_conv_fwd', self.x32.data_ptr(), self.w32.data_ptr(), y.data_ptr(), *geom, prec, ws.data_ptr(), nb, 0)
        return {'y': y}
      if e == 'dgrad':
        gx = torch.empty((N, H, W, Ci), device=DEV)
        L.call('twg_conv_dgrad', self.gy32.data_ptr(), self.w32.data_ptr(), gx.data_ptr(), *geom, prec, ws.data_ptr(), nb, 0)
        return {'gx': gx}
      gw = _f32(self.prefill) if self.prefill is not None else torch.full((k, k, Ci, Co), float('nan'), device=DEV)
      L.call('twg_conv_wgrad', self.x32.data_ptr(), self.gy32.data_ptr(), gw.data_ptr(), *geom,
             int(epi.get('accumulate', 0)), prec, ws.data_ptr(), nb, 0)
      return {'gw': gw}
    if e == 'wgrad_planes':
      gw = _f32(self.prefill) if self.prefill is not None else torch.full((k, k, Ci, Co), float('nan'), device=DEV)
      L.call('twg_conv_wgrad_planes', self.xp.data_ptr(), self.gp.data_ptr(), gw.data_ptr(), *geom, int(epi['accumulate']), 0)
      return {'gw': gw}
    if e == 'dgrad_planes':
      gx = torch.empty((N, H, W, Ci), device=DEV)
      L.call('twg_conv_dgrad_planes', self.gp.data_ptr(), self.wp.data_ptr(), gx.data_ptr(), *geom, 0)
      return {'gx': gx}
    y = torch.empty((N, H, W, Co), device=DEV)
    if e == 'fwd_planes':
      L.call('twg_conv_fwd_planes', self.xp.data_ptr(), self.wp.data_ptr(), y.data_ptr(), *geom, 0)
      return {'y': y}
    if e == 'stats':
      slots = int(L.cdll.twg_conv_stats_slots(*geom))
      assert slots > 0, 'a statistics case must run on a kernel with that epilogue'
      stats = torch.empty((N, slots, Co, 4), device=DEV)
      L.call('twg_conv_fwd_planes_stats', self.xp.data_ptr(), self.wp.data_ptr(), y.data_ptr(), stats.data_ptr(), *geom, 0)
      return {'y': y, 'stats': stats}
    zp = torch.empty((2, N, H, W, Co), device=DEV, dtype=torch.bfloat16)
    b = _f32(self.bias)
    if e == 'bias_act':
      L.call('twg_conv_bias_act_fwd_planes', self.xp.data_ptr(), self.wp.data_ptr(), b.data_ptr(), int(epi['lrelu']),
             y.data_ptr(), zp.data_ptr() if epi['planes'] else None, *geom, 0)
      return {'z': y, 'planes': zp} if epi['planes'] else {'z': y}
    if e == 'bias_act_mask':
      mask = torch.empty((N, H, W, Co // 4), device=DEV, dtype=torch.uint8)
      L.call('twg_conv_bias_act_fwd_planes_mask', self.xp.data_ptr(), self.wp.data_ptr(), b.data_ptr(), y.data_ptr(),
             zp.data_ptr() if epi['planes'] else None, mask.data_ptr(), *geom, 0)
      return {'z': y, 'planes': zp, 'mask': mask} if epi['planes'] else {'z': y, 'mask': mask}
    if e == 'affine':
      a = _f32(self.aff)
      want_z, want_p = epi['out'] in ('fp32', 'both'), epi['out'] in ('planes', 'both')
      L.call('twg_conv_affine_act_fwd_planes', self.xp.data_ptr(), self.wp.data_ptr(), a.data_ptr(), b.data_ptr(),
             int(epi['flags']), y.data_ptr() if want_z else None, zp.data_ptr() if want_p else None, *geom, 0)
      if want_z:
        out['z'] = y
      if want_p:
        out['planes'] = zp
      return out
    raise AssertionError('unknown entry %s' % e)

  def prepare(self):
    """fp32 and split-plane operands, made before the profiled launch and held until the case is done (the launches are
    asynchronous)."""
    e, L = self.case.entry, self.L
    self.x32, self.w32, self.gy32 = _f32(self.x), _f32(self.w), _f32(self.gy)
    if e in ('fwd_planes', 'stats', 'bias_act', 'bias_act_mask', 'affine', 'wgrad_planes'):
      self.xp = _split(L, self.x32)
    if e in ('dgrad_planes', 'wgrad_planes'):
      self.gp = _split(L, self.gy32)
    if e in ('fwd_planes', 'stats', 'bias_act', 'bias_act_mask', 'affine', 'dgrad_planes'):
      self.wp = _wplanes(L, self.w32, e == 'dgrad_planes')

  # fp64 reference of the primary output with (optionally) perturbed operands
  def reference(self, x=None, w=None, gy=None):
    x = self.x if x is None else x
    w = self.w if w is None else w
    gy = self.gy if gy is None else gy
    e, (N, H, W, Ci, Co, k, pad) = self.case.entry, self.case.geom
    if e in ('dgrad', 'dgrad_planes'):
      return ref_dgrad(gy, w, (N, H, W, Ci), pad)
    if e in ('wgrad', 'wgrad_planes'):
      gw = ref_wgrad(x, gy, k, pad)
      return gw + self.prefill if self.prefill is not None else gw
    y = ref_fwd(x, w, pad)
    if e in ('bias_act', 'bias_act_mask', 'affine'):
      return ref_epilogue(y, self.case.epi, self.bias, self.aff)
    return y

  def controls(self):
    """fp64 references of the same case with a tap flip (k = 1: an input-channel rotation), the images rolled by one,
    and the last rows of the image lost."""
    e, (N, H, W, Ci, Co, k, pad) = self.case.entry, self.case.geom
    wgrad = e in ('wgrad', 'wgrad_planes')
    src = 'gy' if e in ('dgrad', 'dgrad_planes') else 'x'
    t = getattr(self, src)
    out = {}
    if k > 1:
      if wgrad:
        ref = self.reference()
        out['tap flip'] = ref.flip(0, 1) if self.prefill is None else (ref - self.prefill).flip(0, 1) + self.prefill
      else:
        out['tap flip'] = self.reference(w=self.w.flip(0, 1))
    else:
      out['channel rotation'] = self.reference(**{src: t.roll(1, dims=3)})
    if N > 1:
      out['image roll'] = self.reference(**{src: t.roll(1, dims=0)})
    if t.shape[1] > 1:
      r = max(1, min(8, t.shape[1] // 2))
      cut = t.clone()
      cut[:, -r:] = 0
      out['lost rows'] = self.reference(**{src: cut})
    return out


def _stats_check(y_ref, stats, tol):
  """Merge the epilogue records {count, pivot, sum(y - pivot), sum(y - pivot)^2} per (image, channel) in fp64 and compare
  mean and variance with the fp64 moments of the fp64 y.  The kernel's y is within tol * max|y| of y_ref, which bounds
  its variance error by 2 * std * tol * max|y| + (tol * max|y|)^2; the records are held to that."""
  s = stats.double()

  cnt, piv, s1, s2 = s[..., 0], s[..., 1], s[..., 2], s[..., 3]
  n = cnt.sum(dim=1)
  safe = torch.where(cnt > 0, cnt, torch.ones_like(cnt))
  mean_r = torch.where(cnt > 0, piv + s1 / safe, torch.zeros_like(piv))
  mean = (cnt * mean_r).sum(dim=1) / n
  m2 = torch.where(cnt > 0, s2 - s1 * s1 / safe, torch.zeros_like(s2)) + cnt * (mean_r - mean[:, None]) ** 2
  var = m2.sum(dim=1) / n
  N, H, W, C = y_ref.shape
  assert torch.equal(n, torch.full_like(n, H * W)), 'records must count every pixel once'
  m_ref = y_ref.mean(dim=(1, 2))
  v_ref = y_ref.var(dim=(1, 2), unbiased=False)
  scale = float(y_ref.abs().max())
  e = tol * scale
  mean_err = float((mean - m_ref).abs().max()) / scale
  var_bound = 2 * v_ref.sqrt() * e + e * e + 1e-6 * v_ref
  var_excess = float(((var - v_ref).abs() / var_bound).max())
  assert mean_err < tol, ('stats mean', mean_err)
  assert var_excess < 1.0, ('stats variance', var_excess)
  return mean_err


def _launched(prof):
  """(conv / pointwise kernel instances, number of memsets) of a profiled region."""
  names, memsets = [], 0
  for ev in prof.events():
    if ev.device_type != torch.autograd.DeviceType.CUDA:
      continue
    if 'memset' in ev.name.lower():
      memsets += 1
    c = canonical(ev.name)
    if c is not None:
      names.append(c)
  return names, memsets


def run_case(L, case, seed, expect=None, controls=True):
  """Runs one case; returns (worst rel_err, smallest control ratio, launched instances)."""
  from torch.profiler import ProfilerActivity, profile
  r = Run(L, case, seed)
  r.prepare()
  torch.cuda.synchronize()
  with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    out = r.launch()
    torch.cuda.synchronize()
  names, memsets = _launched(prof)
  tag = (case, names)
  if expect is not None:
    assert names == [expect], tag
  split = case.epi.get('split')
  if split is not None:
    assert (memsets > 0) == split, tag + ('split-K memset', memsets)
  prec = case.epi.get('prec', 1)
  tol = TOL[prec]
  ref = r.reference()
  errs = []
  primary = None
  for name, t in out.items():
    if name == 'planes':
      got = _planes_value(t, ref.shape)
    elif name == 'mask':
      # bit j of byte i = z[4i + j] > 0; checked against the sign of the fp64 pre-activation away from the kink
      bits = ((t.unsqueeze(-1) >> torch.arange(4, device=DEV, dtype=torch.uint8)) & 1).reshape(ref.shape).bool()
      pre = ref_fwd(r.x, r.w, case.geom[6]) + r.bias
      clear = pre.abs() > 1e-3 * float(pre.abs().max())
      assert torch.equal(bits[clear], (pre > 0)[clear]), tag + ('mask',)
      continue
    elif name == 'stats':
      errs.append(_stats_check(ref_fwd(r.x, r.w, case.geom[6]), t, tol))
      continue
    else:
      got = t
    assert torch.isfinite(got).all(), tag + (name, 'non-finite')
    e = rel_err(got, ref)
    errs.append(e)
    assert e < tol, tag + (name, e, tol)
    if primary is None:
      primary = got
  ratio = math.inf
  # (with a large constant offset y is mostly a tap-symmetric sum: those cases test the statistics' cancellation only)
  if controls and primary is not None and not case.epi.get('offset'):
    for what, cref in r.controls().items():
      d = rel_err(primary, cref)
      ratio = min(ratio, d / tol)
      assert d >= CONTROL_FACTOR * tol, tag + ('control too close', what, d)
  return max(errs), ratio, names


def _record(key, n, err, ratio):
  REPORT[key] = (n, err, ratio)


@pytest.mark.parametrize('key', sorted(COVERAGE))
def test_instance_parity(built_lib, lib_options, key):
  worst, margin = 0.0, math.inf
  for i, case in enumerate(COVERAGE[key]):
    lib_options(case.opts)
    err, ratio, _ = run_case(built_lib, case, 1000 + i, expect=key)
    worst, margin = max(worst, err), min(margin, ratio)
  _record(key, len(COVERAGE[key]), worst, margin)


# ---- the benchmarked step's own convolutions -------------------------------------------------------------------------------

# C-ABI conv entry -> (case entry, index of N in the argument list)
_ENTRIES = {
    'twg_conv_fwd': ('fwd', 3), 'twg_conv_dgrad': ('dgrad', 3), 'twg_conv_wgrad': ('wgrad', 3),
    'twg_conv_fwd_planes': ('fwd_planes', 3), 'twg_conv_fwd_planes_stats': ('stats', 4),
    'twg_conv_bias_act_fwd_planes': ('bias_act', 6), 'twg_conv_bias_act_fwd_planes_mask': ('bias_act_mask', 6),
    'twg_conv_affine_act_fwd_planes': ('affine', 7), 'twg_conv_dgrad_planes': ('dgrad_planes', 3),
    'twg_conv_wgrad_planes': ('wgrad_planes', 3),
}


def _to_case(name, args):
  from tests.conv_coverage import Case
  entry, i = _ENTRIES[name]
  geom = tuple(int(a) for a in args[i:i + 7])
  rest = args[i + 7:]
  nonnull = lambda a: a is not None and a != 0
  if entry in ('fwd', 'dgrad'):
    epi = {'prec': int(rest[0])}
  elif entry == 'wgrad':
    epi = {'accumulate': int(rest[0]), 'prec': int(rest[1])}
  elif entry == 'wgrad_planes':
    epi = {'accumulate': int(rest[0])}
  elif entry == 'stats':
    epi = {'offset': 0.0}
  elif entry == 'bias_act':
    epi = {'lrelu': int(args[3]), 'planes': nonnull(args[5])}
  elif entry == 'bias_act_mask':
    epi = {'planes': nonnull(args[4])}
  elif entry == 'affine':
    z, zp = nonnull(args[5]), nonnull(args[6])
    epi = {'flags': int(args[4]), 'out': 'both' if z and zp else ('fp32' if z else 'planes')}
  else:
    epi = {}
  return Case(entry, geom, epi, {})


def _record_step_convs(fn):
  """Runs fn() with the library's call / try_call wrapped; returns the distinct conv cases it issued, in first-call order."""
  from twingan_b200 import _lib
  L = _lib.lib()
  seen = {}

  def wrap(orig):
    def inner(name, *args):
      rc = orig(name, *args)
      if name in _ENTRIES and not rc:       # a refused tensor-core call (the caller retries at prec 0) is not a conv
        c = _to_case(name, args)
        seen.setdefault((c.entry, c.geom, tuple(sorted(c.epi.items()))), c)
      return rc
    return inner

  L.call, L.try_call = wrap(L.call), wrap(L.try_call)
  try:
    fn()
    torch.cuda.synchronize()
  finally:
    del L.call, L.try_call           # back to the class methods
  return list(seen.values())


def test_step_convs_replayed_against_fp64(built_lib, lib_options, capsys):
  """Every distinct conv call of one compute_gradients at BASELINE configs[3] (256x256, 16 pairs, instance norm, batched
  passes) and of one 64-image inference at configs[4] (batch_renorm, moving statistics), replayed on fresh seeded operands
  through the same entry point with the same geometry and epilogue arguments, against fp64."""
  from twingan_b200 import ops, twingan
  lib_options({})
  ops.set_precision(1)
  gen = torch.Generator(device=DEV).manual_seed(3)
  model = twingan.GanModel(twingan.Flags(train_image_size=256), device=DEV, seed=1234)
  s = torch.rand((16, 256, 256, 3), device=DEV, generator=gen)
  t = torch.rand((16, 256, 256, 3), device=DEV, generator=gen)
  r = twingan.make_dragan_rand(16, 256, DEV, gen)
  train = _record_step_convs(lambda: model.compute_gradients(s, t, r))
  del model
  model = twingan.GanModel(twingan.Flags(train_image_size=256, generator_norm_type='batch_renorm'), device=DEV)
  x = torch.rand((64, 256, 256, 3), device=DEV, generator=gen)
  infer = _record_step_convs(lambda: model.infer(x))
  del model, s, t, r, x
  torch.cuda.empty_cache()
  cases = list({(c.entry, c.geom, tuple(sorted(c.epi.items()))): c for c in train + infer}.values())
  assert train and infer
  # the batched passes: encoder 2 x 16, discriminators 3 x 16, generator 4 x 16 images
  assert any(c.geom[0] == 64 for c in train) and any(c.geom[0] == 48 for c in train) and any(c.geom[0] == 32 for c in train)
  reached, worst = set(), 0.0
  for i, c in enumerate(cases):
    err, _, names = run_case(built_lib, c, 5000 + i, controls=False)
    assert len(names) == 1 and names[0] in COVERAGE, (c, names)   # every instance the step reaches has a parity case
    reached.add(names[0])
    worst = max(worst, err)
  with capsys.disabled():
    print('\n[step replay] %d distinct conv calls (%d training, %d inference), %d kernel instances, worst rel_err %.2e'
          % (len(cases), len(train), len(infer), len(reached), worst))


def test_zz_coverage_report(capsys):
  """Prints what test_instance_parity reached: each instance, its cases, worst rel_err and the smallest control ratio."""
  with capsys.disabled():
    print('\n[conv coverage] %d of %d instances verified' % (len(REPORT), len(COVERAGE)))
    for key in sorted(COVERAGE):
      if key in REPORT:
        n, err, ratio = REPORT[key]
        print('  %-34s cases %2d  worst rel_err %.2e  control / bar >= %.0f' % (key, n, err, ratio))
      else:
        print('  %-34s not run' % key)
