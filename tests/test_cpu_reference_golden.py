"""The oracle against golden vectors produced by THE REFERENCE'S OWN CODE.

tests/golden/reference_pggan.npz was written by tests/golden/make_reference_golden.py, which executes the reference's
nets/pggan.py, nets/pggan_utils.py, libs/batch_norm.py, libs/instance_norm.py and its leaky-ReLU (util_misc.py:68-86)
under a torch-backed stand-in for the TensorFlow-1.8 API (tests/golden/tf18_shim.py), wired like twingan.py:196-270.
That pins, against reference code rather than against a second reading of it: variable names and shapes (at the training
recipe's full 256x256 / 256-channel size too), layer order, which layers carry normaliser / bias / activation /
pixel-norm, the fade-in lerps, UNet end-point selection, minibatch-stddev, the normalisers' forward arithmetic, their
stop-gradients (through the gradients) and their moving-average pushes.  TensorFlow's own kernels (conv2d, avg_pool,
nearest-neighbour resize, moments, batch_normalization, slim's layer wrappers) are restated in the stand-in and stay
unpinned (DESIGN.md 4).  The files keep large result tensors as a sample plus whole-tensor statistics and the seeded inputs
as their seeds (tests/golden/golden_store.py)."""
import ast
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, 'golden'))
import golden_store  # noqa: E402
from golden_provider import stable_hash_provider  # noqa: E402
from oracle import twingan_oracle as O  # noqa: E402

GOLDEN = os.path.join(HERE, 'golden', 'reference_pggan.npz')
VALUE_CASES = ['in16', 'in16grow', 'renorm8grow', 'bn8', 'in4']
NAME_CASES = ['full256', 'full128grow']


@pytest.fixture(scope='module')
def golden():
  return golden_store.load(GOLDEN)


def _cfg(z, case):
  hw, growing, mc, batch, gs = [int(v) for v in z[case + '/meta']]
  return O.Config(hw=hw, is_growing=bool(growing), alpha_grow=float(z[case + '/alpha']), max_num_channels=mc,
                  generator_norm_type=str(z[case + '/norm']), global_step=gs), batch


def _rel(a, b):
  if isinstance(b, golden_store.Sample):
    return b.rel(a)
  a, b = torch.as_tensor(a, dtype=torch.float64), torch.as_tensor(b, dtype=torch.float64)
  return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


@pytest.mark.parametrize('case', VALUE_CASES + NAME_CASES)
def test_variable_names_and_shapes_match_the_reference(golden, case):
  z = golden
  cfg, _ = _cfg(z, case)
  names = [str(n) for n in z[case + '/var_order']]
  shapes = {n: ast.literal_eval(str(s)) for n, s in zip(names, z[case + '/var_shapes'])}
  trainable = {n: bool(t) for n, t in zip(names, z[case + '/var_trainable'])}
  params = O.init_params(cfg)
  state = O.init_norm_state(cfg)
  ref_train = {n for n in names if trainable[n]}
  ref_state = {n for n in names if not trainable[n]}
  # the golden run instantiates discriminator_s only; discriminator_t is the same network under another scope
  mine = {n for n in params if not n.startswith('discriminator_t/')}
  assert mine == ref_train, (sorted(mine - ref_train)[:5], sorted(ref_train - mine)[:5])
  assert {n.replace('discriminator_t/', 'discriminator_s/') for n in params if n.startswith('discriminator_t/')} == \
      {n for n in ref_train if n.startswith('discriminator_s/')}
  assert set(state) == ref_state, (sorted(set(state) - ref_state)[:5], sorted(ref_state - set(state))[:5])
  for n in ref_train:
    assert list(params[n].shape) == shapes[n], n
  for n in ref_state:
    assert list(state[n].shape) == shapes[n], n
  # the product's variable store declares exactly the same set (reference names are its public names)
  from twingan_b200 import pggan
  from twingan_b200.variables import VariableStore
  v = VariableStore('cpu')
  pggan.declare_variables(v, cfg.hw, cfg.is_growing, cfg.max_num_channels, True, cfg.generator_norm_type)
  v.materialize()
  assert {n for n in v.offsets if not n.startswith('discriminator_t/')} == ref_train
  for n in ref_train:
    assert list(v.offsets[n][1]) == shapes[n], n


@pytest.mark.parametrize('case', VALUE_CASES + NAME_CASES)
def test_end_point_keys_and_shapes_match_the_reference(golden, case):
  z = golden
  cfg, batch = _cfg(z, case)
  if cfg.hw > 64:
    pytest.skip('shapes of the full-size case follow from the variable shapes; running the fp64 oracle there is slow')
  provider = stable_hash_provider(1)
  params = {n: provider(n, list(p.shape)) for n, p in O.init_params(cfg).items()}
  state = {n: provider(n, list(s.shape)) for n, s in O.init_norm_state(cfg).items()}
  nets = O.Nets(cfg, params, state)
  x = torch.rand((batch, cfg.hw, cfg.hw, 3), dtype=torch.float64)
  code, ep = nets.encoder(x, '_s')
  img, gep = nets.generator(code, '_t', ep)
  _, dep = nets.discriminator(img, 'discriminator_s')
  for tag, mine in (('ep_s', ep), ('gep_t', gep), ('dep', dep)):
    ref = {str(k): ast.literal_eval(str(s)) for k, s in zip(z['%s/%s_keys' % (case, tag)], z['%s/%s_shapes' % (case, tag)])}
    for k, t in mine.items():
      assert k in ref, (tag, k, sorted(ref))
      assert list(t.shape) == ref[k], (tag, k)
    # everything the reference exposes per block is exposed by the oracle too
    missing = [k for k in ref if k not in mine and k.split('_')[0] in ('block', 'encoder', 'from', 'generator', 'before')]
    missing = [k for k in missing if not k.startswith('before_fc_1x1x') and not k.startswith('downsample_to')]
    assert not missing, (tag, missing)


@pytest.mark.parametrize('case', VALUE_CASES)
def test_forward_gradients_and_state_match_the_reference(golden, case):
  z = golden
  cfg, batch = _cfg(z, case)
  names = [str(n) for n in z[case + '/var_order']]
  trainable = {n: bool(t) for n, t in zip(names, z[case + '/var_trainable'])}
  provider = stable_hash_provider(1)
  params = {}
  for n, p in O.init_params(cfg).items():
    params[n] = provider(n, list(p.shape)).requires_grad_(True)
    if not n.startswith('discriminator_t/'):
      assert abs(float(params[n].detach().sum()) - float(z['%s/var_sum/%s' % (case, n)])) < 1e-9, n   # same values
  state = {n: torch.as_tensor(z['%s/state_before/%s' % (case, n)]) for n in names if not trainable[n]}
  src = torch.as_tensor(z[case + '/in/sources']).requires_grad_(True)
  tgt = torch.as_tensor(z[case + '/in/targets']).requires_grad_(True)

  nets = O.Nets(cfg, params, state)
  enc_s, ep_s = nets.encoder(src, '_s')                       # twingan.py:198-200
  enc_t, ep_t = nets.encoder(tgt, '_t')                       # :215-217
  s_prime, gep_s = nets.generator(enc_t, '_s', ep_t)          # :242-247
  t_prime, gep_t = nets.generator(enc_s, '_t', ep_s)          # :258-262
  pred_real, dep = nets.discriminator(src, 'discriminator_s')      # :370-371
  pred_fake, _ = nets.discriminator(s_prime, 'discriminator_s')    # :372-373
  outs = {'enc_s': enc_s, 'enc_t': enc_t, 's_prime': s_prime, 't_prime': t_prime, 'pred_real': pred_real,
          'pred_fake': pred_fake}
  for k, t in outs.items():
    assert _rel(t.detach(), z['%s/out/%s' % (case, k)]) < 1e-9, (case, k, _rel(t.detach(), z['%s/out/%s' % (case, k)]))
  for tag, mine in (('ep_s', ep_s), ('gep_s', gep_s), ('dep', dep)):
    for k, t in mine.items():
      key = '%s/%s/%s' % (case, tag, k)
      if key in z.files:
        assert _rel(t.detach(), z[key]) < 1e-6, key            # stored as float32

  L = sum((t * torch.as_tensor(z['%s/cot/%s' % (case, k)])).sum() for k, t in outs.items())
  gnames = [n for n in params if not n.startswith('discriminator_t/')]
  grads = torch.autograd.grad(L, [params[n] for n in gnames] + [src, tgt], allow_unused=True)
  for n, g in zip(gnames, grads):
    none_ref = bool(z['%s/grad_is_none/%s' % (case, n)])
    if none_ref:
      assert g is None or float(g.abs().max()) == 0.0, n
    else:
      assert g is not None, n
      assert _rel(g, z['%s/grad/%s' % (case, n)]) < 1e-5, (n, _rel(g, z['%s/grad/%s' % (case, n)]))   # float32 storage
  assert _rel(grads[-2], z[case + '/grad_in/sources']) < 1e-5
  assert _rel(grads[-1], z[case + '/grad_in/targets']) < 1e-5

  # the moving-average pushes of the reference's normalisers (libs/batch_norm.py:295-319, 359-393)
  O.apply_stat_updates(cfg, state, nets)
  for n in state:
    ref = z['%s/state_after/%s' % (case, n)]
    assert _rel(state[n].detach(), ref) < 1e-9 or float(np.abs(ref).max()) == 0.0, (n, _rel(state[n].detach(), ref))
  if state:
    moved = [n for n in state if not np.array_equal(z['%s/state_after/%s' % (case, n)], z['%s/state_before/%s' % (case, n)])]
    assert moved, 'the reference run should have pushed its moving averages'


CLONE_CASES = ['clone_in8', 'clone_in16grow', 'clone_renorm8', 'clone_in64']


F4_CASES = ['f4_wgan_gp8', 'f4_wgan8', 'f4_hinge16grow', 'f4_gan8', 'f4_eqlr_dragan8', 'f4_eqlr_hinge64', 'f4_res16grow',
            'f4_res_eqlr_renorm8']


@pytest.fixture(scope='module')
def golden_f4():
  return golden_store.load(os.path.join(HERE, 'golden', 'reference_f4.npz'))


@pytest.mark.parametrize('case', F4_CASES)
def test_optional_flags_match_the_reference(golden_f4, case):
  """SURVEY 8f-4 flags on the same wiring, again from the reference's own method sources (tests/golden/
  make_reference_golden.py --f4): loss_architecture wgan / wgan_gp (+ drift term) / hinge / gan (image_generation.py:
  330-439), --equalized_learning_rate (nets/pggan_utils.py:236-254) and --use_res_block (:257-264, 334-342)."""
  _check_whole_clone(golden_f4, case)


@pytest.mark.parametrize('case', ['f4_res16grow', 'f4_res_eqlr_renorm8', 'f4_wgan_gp8'])
def test_product_variable_store_matches_the_reference_under_optional_flags(golden_f4, case):
  """The product declares exactly the reference's variables (names, shapes) under --use_res_block too: the residual
  shortcuts add '<block>/shortcut/{weights,biases}' where a block changes its channel count (nets/pggan_utils.py:334-342)."""
  import json
  from twingan_b200 import pggan
  from twingan_b200.variables import VariableStore
  z = golden_f4
  hw, growing, mc, batch, gs, max_steps = [int(v) for v in z[case + '/meta']]
  extra = json.loads(str(z[case + '/extra_flags']))
  names = [str(n) for n in z[case + '/var_order']]
  trainable = {n: bool(t) for n, t in zip(names, z[case + '/var_trainable'])}
  shapes = {n: ast.literal_eval(str(s)) for n, s in zip(names, z[case + '/var_shapes'])}
  v = VariableStore('cpu')
  pggan.declare_variables(v, hw, bool(growing), mc, True, str(z[case + '/norm']), bool(extra.get('use_res_block', False)))
  v.materialize()
  ref_train = {n for n in names if trainable[n]}
  assert set(v.offsets) == ref_train, (sorted(set(v.offsets) - ref_train)[:5], sorted(ref_train - set(v.offsets))[:5])
  for n in ref_train:
    assert list(v.offsets[n][1]) == shapes[n], n
  if extra.get('use_res_block'):
    assert any(n.endswith('/shortcut/biases') for n in v.offsets)


@pytest.mark.parametrize('case', CLONE_CASES)
def test_whole_clone_losses_and_gradients_match_the_reference(golden, case):
  _check_whole_clone(golden, case)


def _check_whole_clone(z, case):
  """The reference's ENTIRE GanModel._clone_fn (twingan.py:146-445: 4 encoder, 4 generator, 6 discriminator passes with
  its scope / reuse / per-domain arg-scope wiring, fade-in of the inputs) followed by its add_loss / add_gan_loss /
  _add_dragan_loss (twingan.py:451-521, image_generation.py:317-476) was executed from the reference's own method
  sources; the oracle's twingan_losses / step_gradients must reproduce every named loss, the two totals and both
  gradient sets (generator variables on the generator collection, discriminator variables on the discriminator
  collection incl. the double backward through the gradient penalty)."""
  import json
  hw, growing, mc, batch, gs, max_steps = [int(v) for v in z[case + '/meta']]
  extra = json.loads(str(z[case + '/extra_flags'])) if (case + '/extra_flags') in z.files else {}
  cfg = O.Config(hw=hw, is_growing=bool(growing), alpha_grow=(gs / max_steps) if growing else 0.0,   # twingan.py:834-835
                 max_num_channels=mc, generator_norm_type=str(z[case + '/norm']), global_step=gs, **extra)
  arch = cfg.loss_architecture
  names = [str(n) for n in z[case + '/var_order']]
  trainable = {n: bool(t) for n, t in zip(names, z[case + '/var_trainable'])}
  provider = stable_hash_provider(2, conv_std=float(z[case + '/conv_std']) if (case + '/conv_std') in z.files else 0.08)
  template = O.init_params(cfg)
  assert set(template) == {n for n in names if trainable[n]}        # both discriminators this time
  params = {n: provider(n, list(p.shape)) for n, p in template.items()}
  for n in params:
    assert abs(float(params[n].sum()) - float(z['%s/var_sum/%s' % (case, n)])) < 1e-9, n
  state = {n: torch.as_tensor(z['%s/state_before/%s' % (case, n)]) for n in names if not trainable[n]}
  assert set(state) == set(O.init_norm_state(cfg))
  src, tgt = torch.as_tensor(z[case + '/in/sources']), torch.as_tensor(z[case + '/in/targets'])
  # the reference drew alpha ~ U[0,1) and the perturbation ~ U[-1,1) in this order per domain (image_generation.py:441-460)
  # (WGAN-GP: one alpha per domain, image_generation.py:421; gan / wgan / hinge draw nothing)
  log = [ast.literal_eval(str(r)) for r in z[case + '/random_log']]
  want_log = {'dragan': [(0.0, 1.0), (-1.0, 1.0)] * 2, 'wgan_gp': [(0.0, 1.0)] * 2}.get(arch, [])
  assert [(lo, hi) for _, lo, hi in log] == want_log
  u = lambda k: torch.as_tensor(z['%s/uniform01/%s' % (case, k)])
  rand = {}
  if arch in ('dragan', 'wgan_gp'):
    rand.update({'alpha_s': u('alpha_s'), 'alpha_t': u('alpha_t')})
  if arch == 'dragan':
    rand.update({'noise_s': 2 * u('noise_s') - 1, 'noise_t': 2 * u('noise_t') - 1})

  g_loss, d_loss, named, grads, ends, nets = O.step_gradients(cfg, params, state, src, tgt, rand)
  assert abs(float(g_loss) - float(z[case + '/generator_loss'])) < 1e-9 * abs(float(g_loss))
  assert abs(float(d_loss) - float(z[case + '/discriminator_loss'])) < 1e-9 * abs(float(d_loss))

  # every named loss, in the reference's collection order (domain s first, then t)
  def per_domain(names_, values):
    out, seen = {}, {}
    for n, v in zip(names_, values):
      n = str(n)
      dom = 's' if n not in seen else 't'
      seen[n] = True
      if n.startswith('l_cyc_'):
        out[n] = float(v)
      elif n.startswith('l_source_content'):
        out['l_content_s'] = float(v)
      elif n.startswith('l_target_content'):
        out['l_content_t'] = float(v)
      else:
        out['%s_%s' % (n, dom)] = float(v)
    return out
  ref_named = per_domain(z[case + '/gloss_names'], z[case + '/gloss_values'])
  ref_named.update(per_domain(z[case + '/dloss_names'], z[case + '/dloss_values']))
  assert set(ref_named) == set(named), (sorted(set(ref_named) ^ set(named)))
  for k, v in ref_named.items():
    assert abs(float(named[k]) - v) <= 1e-9 * max(abs(v), 1e-3), (k, float(named[k]), v)
  if hw >= 64:
    assert 'generator_fool_loss_cycle_s' in named    # twingan.py:466
    assert ('discriminator_real_loss_cycle_t' if arch in ('gan', 'dragan') else 'discriminator_loss_cycle_t') in named
  else:
    assert 'generator_fool_loss_cycle_s' not in named

  for ref_key, mine in (('s_prime_output', ends['s_prime']), ('t_cycle_output', ends['t_cycle']),
                        ('encoded_source_content_before_classification', ends['enc_s']),
                        ('encoded_t_prime_content_before_classification', ends['enc_t_prime']),
                        ('discriminator_real_s_prediction', ends['pred_real_s']),
                        ('discriminator_s_prime_prediction', ends['pred_s_prime']),
                        ('discriminator_t_cycle_prediction', ends['pred_t_cycle'])):
    assert _rel(mine, z['%s/ep/%s' % (case, ref_key)]) < 1e-6, ref_key      # float32 storage

  for n in params:
    if bool(z['%s/grad_is_none/%s' % (case, n)]):
      assert float(grads[n].abs().max()) == 0.0, n
    else:
      ref = z['%s/grad/%s' % (case, n)]
      if (ref.absmax if isinstance(ref, golden_store.Sample) else float(np.abs(ref).max())) < 1e-12:
        # mathematically zero on both sides (e.g. a residual shortcut's bias in front of a 1x1 conv + instance norm): only
        # rounding residue is left to compare
        assert float(grads[n].abs().max()) < 1e-12, n
      else:
        assert _rel(grads[n], ref) < 1e-5, (n, _rel(grads[n], ref))


def _meta():
  import json
  return json.load(open(os.path.join(HERE, 'golden', 'reference_flags_and_stages.json')))


def test_flag_defaults_follow_the_reference_or_its_documented_recipe():
  """tests/golden/reference_flags_and_stages.json holds the defaults of the reference's tf.flags.DEFINE_* calls (read with
  ast).  Flags must equal them, except where docs/training.md:10-37 (the TwinGAN recipe) overrides the default."""
  from twingan_b200 import twingan
  ref = _meta()['flag_defaults']
  f = twingan.Flags()
  same = dict(adam_beta1='adam_beta1', adam_beta2='adam_beta2', opt_epsilon='opt_epsilon', n_critic='n_critic',
              l_content_weight='l_content_weight', l_cyc_weight='l_cyc_weight', gan_weight='gan_weight',
              do_l_cyc_gan='do_l_cyc_gan', loss_architecture='loss_architecture',
              pggan_max_num_channels='pggan_max_num_channels', num_clones='num_clones')
  for mine, theirs in same.items():
    assert getattr(f, mine) == ref[theirs], (mine, getattr(f, mine), ref[theirs])
  # the recipe's overrides (docs/training.md): --learning_rate=0.0001 :25, --use_unet=True :29,
  # --gradient_penalty_lambda=0.25 :32, --do_pixel_norm=True :36
  assert (ref['learning_rate'], f.learning_rate) == (0.005, 1e-4)
  assert (ref['use_unet'], f.use_unet) == (False, True)
  assert (ref['gradient_penalty_lambda'], f.gradient_penalty_lambda) == (10, 0.25)
  assert (ref['do_pixel_norm'], f.do_pixel_norm) == (False, True)
  # the normaliser: reference default batch_norm, recipe batch_renorm (:34), this repo's default is the benchmark's
  # instance_norm ("per-domain AdaIN", BASELINE.json north_star); all three are supported and parity-tested
  assert ref['generator_norm_type'] == 'batch_norm' and f.generator_norm_type in ('instance_norm', 'batch_renorm', 'batch_norm')
  o = O.Config()
  assert (o.adam_beta1, o.adam_beta2, o.adam_eps) == (ref['adam_beta1'], ref['adam_beta2'], ref['opt_epsilon'])
  assert (o.l_content_weight, o.l_cyc_weight, o.gan_weight) == (ref['l_content_weight'], ref['l_cyc_weight'], ref['gan_weight'])


@pytest.mark.parametrize('tag', ['default', 'small'])
def test_stage_plan_matches_the_reference_runner_loop(tag):
  """The reference's own pggan_runner.main() was executed with a stub program that recorded the flags of every stage."""
  from twingan_b200 import pggan_runner as R
  m = _meta()
  fl = m['stages_%s_flags' % tag]
  ref = m['stages_' + tag]
  plan = R.stage_plan(fl['start_hw'], fl['max_hw'], fl['num_images_per_resolution'], fl['hw_to_batch_size'])
  assert len(plan) == len(ref)
  prev_dir = None
  for st, r in zip(plan, ref):
    assert os.path.basename(r['train_dir']) == st.name
    assert (r['train_image_size'], r['is_growing'], r['batch_size'], r['max_number_of_steps'], r['ignore_missing_vars']) == \
        (st.hw, st.is_growing, st.batch_size, st.max_number_of_steps, st.ignore_missing_vars)
    assert r['checkpoint_path'] == prev_dir          # warm start from the previous stage's directory (:146-147)
    prev_dir = r['train_dir']
  if tag == 'default':
    assert R.parse_hw_to_batch_size(fl['hw_to_batch_size']) == R.DEFAULT_HW_TO_BATCH_SIZE


def test_two_clones_through_the_reference_model_deploy(golden):
  """deployment/model_deploy.py (create_clones -> optimize_clones -> _sum_clones_gradients, imported as is) over two
  clones of the reference's _clone_fn on different batches: each clone's loss is divided by num_clones
  (model_deploy.py:265-267), gradients are summed per shared variable (:473-503).  That is what one NCCL all-reduce(sum)
  of per-rank gradients computed on loss / world reproduces (SURVEY 8e; twingan_b200/ddp.py)."""
  z = golden
  case = 'deploy2_in8'
  hw, mc, batch, n = [int(v) for v in z[case + '/meta']]
  assert n == 2 and [str(s) for s in z[case + '/clone_scopes']] == ['clone_0/', 'clone_1/']
  cfg = O.Config(hw=hw, max_num_channels=mc, generator_norm_type=str(z[case + '/norm']), num_clones=2)
  provider = stable_hash_provider(3, conv_std=0.08)
  template = O.init_params(cfg)
  assert set(template) == {str(s) for s in z[case + '/var_order']}
  params = {k: provider(k, list(p.shape)) for k, p in template.items()}
  total_g = total_d = 0.0
  summed = {k: torch.zeros_like(p) for k, p in params.items()}
  for c in range(2):
    u = lambda k: torch.as_tensor(z['%s/uniform01/%s_%d' % (case, k, c)])
    rand = {'alpha_s': u('alpha_s'), 'noise_s': 2 * u('noise_s') - 1, 'alpha_t': u('alpha_t'), 'noise_t': 2 * u('noise_t') - 1}
    gl, dl, _, grads, _, _ = O.step_gradients(cfg, params, {}, torch.as_tensor(z['%s/in/sources_%d' % (case, c)]),
                                              torch.as_tensor(z['%s/in/targets_%d' % (case, c)]), rand)
    total_g += float(gl)
    total_d += float(dl)
    for k in summed:
      summed[k] += grads[k]
  assert abs(total_g - float(z[case + '/generator_loss'])) < 1e-9 * abs(total_g)
  assert abs(total_d - float(z[case + '/discriminator_loss'])) < 1e-9 * abs(total_d)
  n_g, n_d = [int(v) for v in z[case + '/n_grads']]
  assert n_g + n_d == len(params)
  for k in params:
    assert _rel(summed[k], z['%s/grad/%s' % (case, k)]) < 1e-5, (k, _rel(summed[k], z['%s/grad/%s' % (case, k)]))


@pytest.mark.parametrize('case', CLONE_CASES)
def test_inference_tensor_matches_the_reference(golden, case):
  """`custom_generated_t_style_source` -- the tensor the reference's inference wrapper fetches
  (inference/image_translation_infer.py:46-99; built at twingan.py:300-365): eval-mode encoder with the source domain's
  normaliser parameters, eval-mode generator with the target domain's, UNet skips, moving statistics for batch norms."""
  z = golden
  hw, growing, mc, batch, gs, max_steps = [int(v) for v in z[case + '/meta']]
  cfg = O.Config(hw=hw, is_growing=bool(growing), alpha_grow=(gs / max_steps) if growing else 0.0,
                 max_num_channels=mc, generator_norm_type=str(z[case + '/norm']), global_step=gs)
  names = [str(n) for n in z[case + '/var_order']]
  trainable = {n: bool(t) for n, t in zip(names, z[case + '/var_trainable'])}
  provider = stable_hash_provider(2, conv_std=0.08)
  params = {n: provider(n, list(p.shape)) for n, p in O.init_params(cfg).items()}
  state = {n: torch.as_tensor(z['%s/state_before/%s' % (case, n)]) for n in names if not trainable[n]}
  got = O.inference(cfg, params, state, torch.as_tensor(z[case + '/in/sources']))
  assert _rel(got, z[case + '/infer/custom_generated_t_style_source']) < 1e-6      # float32 storage
