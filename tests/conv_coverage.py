"""Coverage table of the convolution kernels: for every conv / pointwise kernel instance compiled into libtwg.so, the
parity cases that must launch exactly that instance (tests/test_gpu_conv_matrix.py runs them against fp64 and checks the
launched kernel with the profiler; tests/test_cpu_conv_coverage.py checks that the table names every instance the
library contains).  Importable without a GPU.

A case is (entry, geom, epi, opts):
  entry  which C-ABI call runs it:
           'fwd' / 'dgrad' / 'wgrad'   twg_conv_fwd / _dgrad / _wgrad (epi 'prec', and 'accumulate' for wgrad)
           'fwd_planes' / 'dgrad_planes' / 'wgrad_planes'   the split-plane forms (wgrad: epi 'accumulate')
           'stats'          twg_conv_fwd_planes_stats (epi 'offset': constant added to x, large |mean| / std)
           'bias_act'       twg_conv_bias_act_fwd_planes (epi 'lrelu', 'planes')
           'bias_act_mask'  twg_conv_bias_act_fwd_planes_mask (epi 'planes')
           'affine'         twg_conv_affine_act_fwd_planes (epi 'flags', 'out' in fp32 / planes / both)
  geom   (N, H, W, Cin, Cout, k, pad) of the convolution; for dgrad it is the forward conv whose input gradient is taken,
         so the GEMM roles are swapped: a dgrad of Cin -> Cout runs the forward instance of Cout -> Cin
  epi    epilogue / call arguments as above, plus 'split' for the tap kernel: True = the launch must split the K loop
         (it zeroes y first, visible as a memset), False = it must not, absent = not checked
  opts   twg_set_option overrides for the case ({2: SUB} forces the halo kernel's sub-tile count; 6 / 7 / 9 = 0 reach the
         fallbacks); every other option has its library default (DEFAULT_OPTIONS)
"""
import math
import re
from collections import namedtuple

Case = namedtuple('Case', 'entry geom epi opts')

NUM_SMS = 148                   # B200: the persistent kernels launch min(work items, 148) CTAs
DEFAULT_OPTIONS = {1: 1, 2: 0, 3: 0, 4: 0, 6: 1, 7: 1, 8: 0, 9: 1}
TOL = {0: 2e-5, 1: 1e-4}        # rel_err bar per precision: exact fp32 (prec 0), split-bf16 tensor cores (prec 1)

# Compiled, but unreachable with the default options and kept out of the matrix on purpose.
EXCLUDED = {
    'k_conv_fwd_tc<64,128,1,1>': 'A operand staged in TMEM (option 3): a rejected experiment, measured slower',
    'k_conv_fwd_tc<64,128,0,2>': '2-CTA clusters with multicast weight tiles (option 4): a rejected experiment',
    'k_conv_fwd_tc<64,64,0,2>': '2-CTA clusters with multicast weight tiles (option 4): a rejected experiment',
    'k_conv_htap2_tc': 'CTA-pair wide-layer halo kernel (option 8): a rejected experiment, measured slower',
}

_DEMANGLED = re.compile(r'(k_(?:conv|pw)_[A-Za-z0-9_]+)(?:<([^<>]*)>)?')


def canonical(name: str):
  """'void twg::k_conv_fwd_tc<64, 128, false, 1>(CUtensorMap_st, ...)' -> 'k_conv_fwd_tc<64,128,0,1>'; None when the
  name is not a conv / pointwise kernel.  false / true and 0 / 1 compare alike."""
  m = _DEMANGLED.search(name)
  if not m:
    return None
  if m.group(2) is None:
    return m.group(1)
  args = [a.strip() for a in m.group(2).split(',')]
  args = [{'false': '0', 'true': '1'}.get(a, a) for a in args]
  return '%s<%s>' % (m.group(1), ','.join(args))


def instances_from_symbols(symbols):
  """Conv / pointwise kernel instances named by mangled symbols (`nm --defined-only` lines): a symbol such as
  _ZN3twg14k_conv_halo_tcILi16ELi32ELi4ELi0EEEv... or its __device_stub__ twin gives 'k_conv_halo_tc<16,32,4,0>'."""
  out = set()
  for sym in symbols:
    for m in re.finditer(r'ZN3twg(\d+)', sym):
      n = int(m.group(1))
      name = sym[m.end():m.end() + n]
      if not (name.startswith('k_conv_') or name.startswith('k_pw_')):
        continue
      rest = sym[m.end() + n:]
      t = re.match(r'I((?:L[a-z]\d+E)+)E', rest)
      if t:
        name += '<%s>' % ','.join(re.findall(r'L[a-z](\d+)E', t.group(1)))
      out.add(name)
  return out


def _cdiv(a, b):
  return -(-a // b)


def _wrap_n(per_image, per_cta=3):
  """Smallest batch whose persistent launch gives every one of the 148 CTAs at least `per_cta` work items, with a
  remainder (the last round is partial)."""
  n = 1
  while n * per_image < per_cta * NUM_SMS or (n * per_image) % NUM_SMS == 0:
    n += 1
  return n


COVERAGE = {}


def _add(key, *cases):
  COVERAGE.setdefault(key, []).extend(cases)


# ---- halo kernel k_conv_halo_tc<CIN, BN, SUB, EPI> (3x3, channels 16/32/64, CIN * BN <= 2048, H, W >= 16) -----------
# tile 16 rows x 8*SUB columns; geometries: several tiles per CTA with ragged rows and columns, H = W = 16 with more
# tiles than CTAs, and a small ragged one
HALO_TRIPLES = [(16, 16, 1), (16, 16, 2), (16, 16, 4), (16, 32, 1), (16, 32, 2), (16, 32, 4), (16, 64, 1), (16, 64, 2),
                (32, 16, 1), (32, 16, 2), (32, 32, 1), (32, 32, 2), (32, 64, 1), (32, 64, 2), (64, 16, 1), (64, 32, 1)]
_AFFINE_FLAGS = [0, 1, 2, 3]     # TWG_FLAG_LRELU | TWG_FLAG_PIXNORM combinations

for _i, (_ci, _bn, _sub) in enumerate(HALO_TRIPLES):
  _o = {2: _sub}
  _multi = (_wrap_n(3 * _cdiv(36, 8 * _sub)), 40, 36)          # H % 16 != 0, W % (8 SUB) != 0, >= 3 tiles per CTA
  _sq = (_wrap_n(_cdiv(16, 8 * _sub), 1), 16, 16)               # H = W = 16, more tiles than CTAs
  _small = (2, 20, 44)
  fwd = lambda g, ci=_ci, bn=_bn: g + (ci, bn, 3, 1)
  bwd = lambda g, ci=_ci, bn=_bn: g + (bn, ci, 3, 1)            # dgrad of BN -> CIN runs the CIN -> BN instance
  _add('k_conv_halo_tc<%d,%d,%d,0>' % (_ci, _bn, _sub),
       Case('fwd_planes', fwd(_multi), {}, _o),
       Case('dgrad_planes', bwd(_sq), {}, _o),
       Case('bias_act', fwd(_small), {'lrelu': 1, 'planes': False}, _o),
       Case('bias_act', fwd(_sq), {'lrelu': 0, 'planes': True}, _o),
       Case('bias_act_mask', fwd(_multi), {'planes': True}, _o))
  _add('k_conv_halo_tc<%d,%d,%d,1>' % (_ci, _bn, _sub),
       Case('stats', fwd(_multi), {'offset': 0.0}, _o),
       Case('stats', fwd(_small), {'offset': 40.0}, _o))
  _add('k_conv_halo_tc<%d,%d,%d,2>' % (_ci, _bn, _sub),
       Case('affine', fwd(_small), {'flags': _AFFINE_FLAGS[_i % 4], 'out': 'fp32'}, _o),
       Case('affine', fwd(_sq), {'flags': _AFFINE_FLAGS[(_i + 1) % 4], 'out': 'planes'}, _o),
       Case('affine', fwd(_multi), {'flags': _AFFINE_FLAGS[(_i + 2) % 4], 'out': 'both'}, _o))

# ---- wide-layer halo kernel k_conv_htap_tc<BN> (3x3, K % 64 == 0, Nc = 64 or a multiple of 128, >= 96 work items) ----
# work item = (16 x 8 tile, BN block); 40 x 36 images have 15 tiles each
for _k in (64, 128, 256, 512):
  _add('k_conv_htap_tc<64>', Case('fwd_planes', (_wrap_n(15), 40, 36, _k, 64, 3, 1), {}, {}))
  for _nc in (128, 256):
    _add('k_conv_htap_tc<128>', Case('fwd_planes', (_wrap_n(15 * _nc // 128), 40, 36, _k, _nc, 3, 1), {}, {}))
_add('k_conv_htap_tc<64>',
     Case('fwd_planes', (48, 16, 16, 64, 64, 3, 1), {}, {}),                       # exactly 96 items
     Case('bias_act', (17, 32, 24, 128, 64, 3, 1), {'lrelu': 1, 'planes': True}, {}),
     Case('dgrad_planes', (13, 32, 32, 64, 128, 3, 1), {}, {}))
_add('k_conv_htap_tc<128>',
     Case('fwd_planes', (48, 16, 16, 128, 128, 3, 1), {}, {}),                     # exactly 96 items
     Case('bias_act', (8, 32, 24, 256, 256, 3, 1), {'lrelu': 1, 'planes': True}, {}),
     Case('bias_act', (17, 16, 48, 128, 128, 3, 1), {'lrelu': 0, 'planes': False}, {}),
     Case('dgrad_planes', (13, 32, 32, 128, 256, 3, 1), {}, {}))

# ---- tap-per-TMA kernel k_conv_fwd_tc<CC, BN, false, 1>: everything the halo kernels do not take -----------------------
# CC = channel chunk of GEMM K (16 / 32 / 64), BN = min(GEMM N, 128); H or W < 16 keeps the halo kernels out.  Split-K
# sums y with atomics and cannot emit split planes; through the C ABI a plane output always comes with a bias, which keeps
# the K loop whole -- the second case pins that down at the shape where the first one splits.
for _cc in (16, 32, 64):
  for _bn in (16, 32, 64, 128):
    _kk = _cc if _cc < 64 else 128             # 128 input channels: two 64-channel chunks per tap
    _nc = _bn if _bn < 128 else 256            # 256 output channels: two BN blocks
    _add('k_conv_fwd_tc<%d,%d,0,1>' % (_cc, _bn),
         Case('fwd_planes', (2, 8, 12, _kk, _nc, 3, 1), {'split': True}, {}),      # under-filled grid: split-K
         Case('bias_act', (2, 8, 12, _kk, _nc, 3, 1), {'lrelu': 1, 'planes': True, 'split': False}, {}),
         Case('fwd_planes', (160, 12, 8, _kk, _nc, 3, 1), {'split': False}, {}),   # full grid, ragged rows
         Case('fwd_planes', (20, 4, 4, _kk, _nc, 1, 0), {'split': False}, {}),     # 1x1, 8 images per tile
         Case('dgrad_planes', (3, 8, 8, _nc, _kk, 3, 1), {}, {}))
# 95 work items: one short of the wide-layer halo kernel's threshold
_add('k_conv_fwd_tc<64,64,0,1>', Case('fwd_planes', (19, 16, 40, 64, 64, 3, 1), {'split': False}, {}))
_add('k_conv_fwd_tc<64,128,0,1>', Case('fwd_planes', (19, 16, 40, 128, 128, 3, 1), {'split': False}, {}))

# ---- weight gradients: row-shift kernel (default for the narrow layers), halo kernel (option 9 = 0), tap-stacked kernel
# (option 7 = 0, and every shape with W < 16 or H < 8 or k = 1); <CN, BNW> = (chunk of Cin, min(Cout, 64)) -------------
_WG_PAIRS = [(16, 16), (16, 32), (16, 64), (32, 16), (32, 32), (32, 64), (64, 16), (64, 32), (64, 64)]
for _cn, _bw in _WG_PAIRS:
  _many = (_wrap_n(9), 24, 40)                 # 16 x 8 tiles: 3 x 3 per image, ragged columns, several per CTA
  _min = (3, 8, 16)
  g = lambda s, cn=_cn, bw=_bw: s + (cn, bw, 3, 1)
  if (_cn, _bw) != (64, 64):
    _add('k_conv_wgrad_rows<%d,%d>' % (_cn, _bw),
         Case('wgrad_planes', g(_many), {'accumulate': 0}, {}),
         Case('wgrad_planes', g(_min), {'accumulate': 1}, {}))
    _halo_opts = {9: 0}
  else:
    _halo_opts = {}                            # no row-shift instance: the default path for 64 x 64
  _add('k_conv_wgrad_halo<%d,%d>' % (_cn, _bw),
       Case('wgrad_planes', g(_many), {'accumulate': 0}, _halo_opts),
       Case('wgrad_planes', g(_min), {'accumulate': 1}, _halo_opts))
  _add('k_conv_wgrad_tc2<%d,%d>' % (_cn, _bw),
       Case('wgrad_planes', g(_many), {'accumulate': 0}, {7: 0}),
       Case('wgrad_planes', (3, 8, 15, _cn, _bw, 3, 1), {'accumulate': 1}, {}),     # W = 15 goes to this kernel
       Case('wgrad_planes', (4, 8, 8, _cn, _bw, 1, 0), {'accumulate': 1}, {}))      # and so does k = 1
_add('k_conv_wgrad_rows<64,16>', Case('wgrad_planes', (20, 24, 40, 128, 16, 3, 1), {'accumulate': 1}, {}))   # 2 Cin chunks
_add('k_conv_wgrad_rows<32,64>', Case('wgrad_planes', (20, 24, 40, 32, 128, 3, 1), {'accumulate': 0}, {}))   # 2 Cout blocks
# 64 x 64 blocks need 5 tap groups x 128 TMEM columns: two CTA populations, sized from `want` = 148 / channel blocks
_add('k_conv_wgrad_halo<64,64>',
     Case('wgrad_planes', (4, 24, 40, 256, 256, 3, 1), {'accumulate': 1}, {}),     # 16 channel blocks: want = 9
     Case('wgrad_planes', (1, 8, 16, 128, 64, 3, 1), {'accumulate': 0}, {}))       # one pixel tile for both populations

# ---- exact-fp32 CUDA-core kernels (prec 0) ----------------------------------------------------------------------------
_P0, _P0A = {'prec': 0}, {'prec': 0, 'accumulate': 1}
_add('k_conv_fwd_simt<16,2,0>', Case('fwd', (2, 8, 8, 32, 16, 3, 1), _P0, {}), Case('fwd', (3, 12, 20, 3, 16, 3, 1), _P0, {}))
_add('k_conv_fwd_simt<16,2,1>', Case('dgrad', (2, 8, 8, 16, 32, 3, 1), _P0, {}), Case('dgrad', (2, 6, 10, 3, 64, 3, 1), _P0, {}))
_add('k_conv_fwd_simt<64,4,0>', Case('fwd', (4, 4, 4, 257, 256, 3, 1), _P0, {}), Case('fwd', (4, 4, 4, 256, 256, 4, 0), _P0, {}),
     Case('fwd', (2, 12, 20, 64, 32, 3, 1), _P0, {}), Case('fwd', (16, 32, 32, 32, 64, 3, 1), _P0, {}))
_add('k_conv_fwd_simt<64,4,1>', Case('dgrad', (4, 4, 4, 257, 256, 3, 1), _P0, {}), Case('dgrad', (4, 4, 4, 256, 256, 4, 0), _P0, {}),
     Case('dgrad', (16, 32, 32, 64, 32, 3, 1), _P0, {}))
_add('k_conv_wgrad_simt<16,16>', Case('wgrad', (2, 8, 8, 16, 16, 3, 1), _P0, {}), Case('wgrad', (3, 10, 14, 3, 16, 3, 1), _P0A, {}))
_add('k_conv_wgrad_simt<16,64>', Case('wgrad', (2, 8, 8, 3, 32, 3, 1), _P0, {}), Case('wgrad', (2, 8, 8, 16, 64, 3, 1), _P0A, {}))
_add('k_conv_wgrad_simt<64,16>', Case('wgrad', (2, 8, 8, 64, 16, 3, 1), _P0, {}), Case('wgrad', (2, 8, 8, 32, 3, 3, 1), _P0A, {}))
_add('k_conv_wgrad_simt<64,64>', Case('wgrad', (4, 4, 4, 257, 256, 3, 1), _P0, {}), Case('wgrad', (4, 4, 4, 256, 256, 4, 0), _P0A, {}))

# ---- pointwise kernels: fromRGB (Cin = 3) and toRGB (Cout = 3) at every channel width L, both directions ---------------
# the L-wide side is reduced by k_pw_reduce_px (L = 16, 32) or k_pw_reduce<V> (V float4 per lane); 420 pixels (ragged)
_PW_REDUCE = {16: 'k_pw_reduce_px<4>', 32: 'k_pw_reduce_px<8>', 64: 'k_pw_reduce<1>', 128: 'k_pw_reduce<1>',
              256: 'k_pw_reduce<2>', 512: 'k_pw_reduce<4>'}
_PW_WGRAD = {16: 'k_pw_wgrad<1>', 32: 'k_pw_wgrad<1>', 64: 'k_pw_wgrad<1>', 128: 'k_pw_wgrad<1>', 256: 'k_pw_wgrad<2>',
             512: 'k_pw_wgrad<4>'}
for _l in (16, 32, 64, 128, 256, 512):
  _from, _to = (3, 10, 14, 3, _l, 1, 0), (3, 10, 14, _l, 3, 1, 0)
  _add('k_pw_expand', Case('fwd', _from, _P0, {}), Case('dgrad', _to, _P0, {}))
  _add(_PW_REDUCE[_l], Case('fwd', _to, _P0, {}), Case('dgrad', _from, _P0, {}))
  _add(_PW_WGRAD[_l], Case('wgrad', _from, _P0, {}), Case('wgrad', _to, _P0A, {}))
_add('k_pw_reduce<4>', Case('fwd', (2, 8, 8, 512, 4, 1, 0), _P0, {}))        # four output channels
_add('k_pw_reduce<2>', Case('fwd', (4, 1, 1, 256, 1, 1, 0), _P0, {}))        # the discriminator's fully connected layer
