"""Golden vectors produced by THE REFERENCE'S OWN network code.

Runs the reference's nets/pggan.py (+ nets/pggan_utils.py, libs/batch_norm.py, libs/instance_norm.py and the leaky-ReLU
of util_misc.py:68-86) under tests/golden/tf18_shim.py -- a torch-backed stand-in for the few dozen TensorFlow-1.8 API
entry points those files use -- with the wiring of twingan.py:196-270,370-373 (scopes `encoder_content`, `generator`,
`discriminator_s`; per-domain `_s` / `_t` normaliser postfixes; UNet end points), and stores inputs, every variable the
reference created (under the name the reference gave it), outputs, end points, gradients and the normaliser state after
the pass in tests/golden/reference_pggan.npz, in the compact form of tests/golden/golden_store.py (seeded inputs as
their seeds, large result tensors as statistics plus a fixed sample of elements).

Needs a checkout of the reference (jerryli27/TwinGAN); the .npz files do not.  tests/test_cpu_reference_golden.py then holds
oracle/twingan_oracle.py to these vectors.  What this does and does not pin is stated at the top of tf18_shim.py.

  python tests/golden/make_reference_golden.py --reference <TwinGAN checkout> [--f4]
"""
from __future__ import annotations

import argparse
import json
import ast
import functools
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import tf18_shim as tfs  # noqa: E402
import golden_store  # noqa: E402
from golden_provider import stable_hash_provider  # noqa: E402

CASES = [
    # name, hw, is_growing, alpha, max channels, norm type, batch, global_step, store values?
    ('in16', 16, False, 0.0, 16, 'instance_norm', 3, 0, True),
    ('in16grow', 16, True, 0.3, 16, 'instance_norm', 3, 0, True),
    ('renorm8grow', 8, True, 0.6, 16, 'batch_renorm', 4, 15000, True),
    ('bn8', 8, False, 0.0, 16, 'batch_norm', 4, 0, True),
    ('in4', 4, False, 0.0, 16, 'instance_norm', 2, 0, True),
    # the training recipe's real sizes (docs/training.md:32): variable names + shapes and end-point keys + shapes only
    ('full256', 256, False, 0.0, 256, 'batch_renorm', 1, 0, False),
    ('full128grow', 128, True, 0.5, 256, 'instance_norm', 1, 0, False),
]


def load_reference(ref_root):
  tf = tfs.install()
  sys.path.insert(0, ref_root)
  # Python-2 implicit relative imports: `import pggan_utils` inside nets/, `from batch_norm import ...` inside libs/
  sys.path.insert(1, os.path.join(ref_root, 'nets'))
  sys.path.insert(2, os.path.join(ref_root, 'libs'))
  # util_misc.py is Python-2 only (print statement, line 300+); the path needs ONE function of it.  Execute that
  # function's own source text, nothing else.
  src = open(os.path.join(ref_root, 'util_misc.py')).read()
  lines = src.split('\n')
  start = next(i for i, l in enumerate(lines) if l.startswith('def fp16_friendly_leaky_relu('))
  end = next(i for i in range(start + 1, len(lines)) if lines[i].startswith('def '))
  fn_src = '\n'.join(lines[start:end])
  ast.parse(fn_src)
  util_misc = types.ModuleType('util_misc')
  util_misc.__dict__['tf'] = tf
  exec(compile(fn_src, os.path.join(ref_root, 'util_misc.py'), 'exec'), util_misc.__dict__)
  sys.modules['util_misc'] = util_misc
  # flags the path reads that are defined in files we do not import (twingan.py / image_generation.py / libs/sn.py)
  for k, v in dict(generator_norm_type='batch_renorm', spectral_norm=False, spectral_norm_in_non_discriminator=False,
                   use_style_embedding=False).items():
    tfs._define(k, v)
  import nets.pggan as pggan          # noqa: E402  (the reference)
  pggan_utils = pggan.pggan_utils
  return tf, pggan, pggan_utils


def _stream(name, seed, draws):
  """The draws of one case's seeded generator, in order: tests/golden/golden_store.py replays them instead of storing them."""
  return np.array(json.dumps({'seed': seed, 'draws': [['%s/%s' % (name, k), kind, list(shape)] for k, kind, shape in draws]}))


def run_case(tf, pggan, pggan_utils, case, out):
  name, hw, growing, alpha, mc, norm, batch, global_step, store_values = case
  tfs.reset(stable_hash_provider(1), global_step=global_step)
  tfs.FLAGS.pggan_max_num_channels = mc
  tfs.FLAGS.generator_norm_type = norm
  g = torch.Generator().manual_seed(100 + hw)
  sources = tfs.Tensor(torch.rand((batch, hw, hw, 3), generator=g, dtype=torch.float64).requires_grad_(True))
  targets = tfs.Tensor(torch.rand((batch, hw, hw, 3), generator=g, dtype=torch.float64).requires_grad_(True))

  def scope_fn(postfix):   # twingan.py:_get_generator_arg_scope_fn + _copy_kwargs(scope_fn_postfix=...)
    return functools.partial(pggan.conditional_progressive_gan_generator_arg_scope, norm_type=norm,
                             conditional_layer_var_scope_postfix=postfix)

  common = dict(is_training=True, is_growing=growing, alpha_grow=alpha, do_self_attention=False, self_attention_hw=64,
                do_pixel_norm=True, dtype=tf.float32, target_shape=targets.shape)
  with tf.variable_scope('encoder_content'):
    enc_s, ep_s = pggan.encoder_before_classification(sources, arg_scope_fn=scope_fn('_s'), **common)
  with tf.variable_scope('encoder_content', reuse=tf.AUTO_REUSE):
    enc_t, ep_t = pggan.encoder_before_classification(targets, arg_scope_fn=scope_fn('_t'), **common)
  with tf.variable_scope('generator'):
    s_prime, gep_s = pggan.generator(enc_t, arg_scope_fn=scope_fn('_s'), unet_end_points=ep_t, **common)
  with tf.variable_scope('generator', reuse=tf.AUTO_REUSE):
    t_prime, gep_t = pggan.generator(enc_s, arg_scope_fn=scope_fn('_t'), unet_end_points=ep_s, **common)
  with tf.variable_scope('discriminator_s', reuse=False):
    pred_real, dep = pggan.discriminator(sources, is_training=True, is_growing=growing, alpha_grow=alpha,
                                         do_self_attention=False, self_attention_hw=64, do_dgrop=False)
  with tf.variable_scope('discriminator_s', reuse=True):
    pred_fake, _ = pggan.discriminator(s_prime, is_training=True, is_growing=growing, alpha_grow=alpha,
                                       do_self_attention=False, self_attention_hw=64, do_dgrop=False)

  outs = [('enc_s', enc_s), ('enc_t', enc_t), ('s_prime', s_prime), ('t_prime', t_prime), ('pred_real', pred_real),
          ('pred_fake', pred_fake)]
  out[name + '/meta'] = np.array([hw, int(growing), mc, batch, global_step], dtype=np.int64)
  out[name + '/alpha'] = np.array(alpha)
  out[name + '/norm'] = np.array(norm)
  out[name + '/var_order'] = np.array(list(tfs.STORE.vars.keys()))
  out[name + '/var_shapes'] = np.array([str(list(v.t.shape)) for v in tfs.STORE.vars.values()])
  out[name + '/var_trainable'] = np.array([bool(v.trainable) for v in tfs.STORE.vars.values()])
  for tag, ep in (('ep_s', ep_s), ('ep_t', ep_t), ('gep_s', gep_s), ('gep_t', gep_t), ('dep', dep)):
    keys = sorted(k for k, v in ep.items() if isinstance(v, tfs.Tensor))
    out[name + '/%s_keys' % tag] = np.array(keys)
    out[name + '/%s_shapes' % tag] = np.array([str(list(ep[k].t.shape)) for k in keys])
  print('%-12s %3d variables, outputs %s' % (name, len(tfs.STORE.vars),
                                              ', '.join('%s%s' % (k, list(v.t.shape)) for k, v in outs)))
  if not store_values:
    return

  # a scalar functional of everything, for gradients (fixed random cotangents)
  L = 0.0
  draws = [('in/sources', 'rand', sources.t.shape), ('in/targets', 'rand', targets.t.shape)]
  for k, v in outs:
    draws.append(('cot/' + k, 'randn', v.t.shape))
    cot = torch.randn(v.t.shape, generator=g, dtype=torch.float64)
    out[name + '/cot/' + k] = cot.numpy()
    L = L + (v.t * cot).sum()
  train_vars = [(n, v) for n, v in tfs.STORE.vars.items() if v.trainable]
  grads = torch.autograd.grad(L, [v.t for _, v in train_vars] + [sources.t, targets.t], allow_unused=True)
  f32 = lambda t: t.detach().to(torch.float32).numpy()
  out[name + '/in/sources'] = sources.t.detach().numpy()
  out[name + '/in/targets'] = targets.t.detach().numpy()
  out[name + '/rng_stream'] = _stream(name, 100 + hw, draws)
  provider = stable_hash_provider(1)
  for n, v in tfs.STORE.vars.items():
    if v.trainable:
      # a forward pass never modifies a trainable variable: the values are regenerated by stable_hash_provider(1) in
      # the test (checked against this checksum) instead of being stored
      out[name + '/var_sum/' + n] = np.array(float(v.t.detach().sum()))
    else:
      # normaliser state: the value handed out and the value AFTER the reference's moving-average pushes
      out[name + '/state_after/' + n] = v.t.detach().numpy()
      out[name + '/state_before/' + n] = provider(n, list(v.t.shape), None, False).numpy()
  for k, v in outs:
    out[name + '/out/' + k] = v.t.detach().numpy()
  for tag, ep in (('ep_s', ep_s), ('gep_s', gep_s), ('dep', dep)):
    for k, v in ep.items():
      if isinstance(v, tfs.Tensor):
        out[name + '/%s/%s' % (tag, k)] = f32(v.t)
  for (n, _), gr in zip(train_vars, grads):
    out[name + '/grad_is_none/' + n] = np.array(gr is None)
    if gr is not None:
      out[name + '/grad/' + n] = f32(gr)
  out[name + '/grad_in/sources'] = f32(grads[-2])
  out[name + '/grad_in/targets'] = f32(grads[-1])
  out[name + '/update_ops'] = np.array(tfs.STORE.update_ops)


# ------------------------------------------------------------------------------------------------------------
# the whole clone function + losses (twingan.py:146-521, image_generation.py:317-476, 1001-1006)
# ------------------------------------------------------------------------------------------------------------
CLONE_CASES = [
    # name, hw, is_growing, global_step, max_number_of_steps, max channels, norm type, batch
    ('clone_in8', 8, False, 0, 1000, 16, 'instance_norm', 3),
    ('clone_in16grow', 16, True, 250, 1000, 16, 'instance_norm', 2),
    ('clone_renorm8', 8, False, 0, 1000, 16, 'batch_renorm', 4),
    ('clone_in64', 64, False, 0, 1000, 8, 'instance_norm', 2),      # hw >= 64 switches the cycle GAN term on (twingan.py:466)
]


def _method_sources(path, class_name, names):
  """Source text of the named methods of `class_name` in `path`, decorators included, as written in the reference."""
  src = open(path).read()
  tree = ast.parse(src)
  lines = src.split('\n')
  cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == class_name)
  out = []
  for name in names:
    fn = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == name)
    first = min([fn.lineno] + [d.lineno for d in fn.decorator_list])
    out.append('\n'.join(lines[first - 1:fn.end_lineno]))
  return out


def _module_constants(path, env):
  """Top-level NAME = <simple expression> assignments of a reference module (scope and collection names)."""
  tree = ast.parse(open(path).read())
  consts = {}
  for node in tree.body:
    if isinstance(node, ast.Assign) and len(node.targets) == 1 and isinstance(node.targets[0], ast.Name) \
        and node.targets[0].id.isupper():
      ok = all(isinstance(n, (ast.Constant, ast.Name, ast.Attribute, ast.BinOp, ast.Add, ast.Mod, ast.Tuple, ast.Load))
               for n in ast.walk(node.value))
      if ok:
        try:
          consts[node.targets[0].id] = eval(compile(ast.Expression(node.value), path, 'eval'), dict(env, **consts))
        except Exception:   # noqa: BLE001 -- e.g. FLAGS = tf.flags.FLAGS is provided separately
          pass
  return consts


def build_reference_ganmodel(ref_root, tf, pggan):
  """A class made of the reference's own method sources: image_generation.GanModel's loss helpers as the base,
  twingan.GanModel's clone function / loss wiring on top.  The only edit is the mechanical Python-2 -> 3 spelling
  `.iteritems()` -> `.items()`."""
  ig_path, tw_path = os.path.join(ref_root, 'image_generation.py'), os.path.join(ref_root, 'twingan.py')
  base_methods = _method_sources(ig_path, 'GanModel', ['add_gan_loss', '_add_dragan_loss', '_add_wgan_gp_loss',
                                                        'get_perturbed_batch', 'get_growing_image'])
  top_methods = _method_sources(tw_path, 'GanModel', ['_clone_fn', 'add_loss', 'get_growing_source_and_target',
                                                       '_add_pggan_kwargs', '_copy_kwargs', '_get_generator_arg_scope_fn'])
  um = open(os.path.join(ref_root, 'util_misc.py')).read().split('\n')
  start = next(i for i, l in enumerate(um) if l.startswith('def combine_dicts('))
  end = next(i for i in range(start + 1, len(um)) if um[i].startswith('def '))
  combine_src = '\n'.join(um[start:end]).replace('.iteritems()', '.items()')
  sys.modules['util_misc'].__dict__.update({})
  exec(compile(combine_src, os.path.join(ref_root, 'util_misc.py'), 'exec'), sys.modules['util_misc'].__dict__)

  ig_consts = _module_constants(ig_path, {})
  env = {'image_generation': types.SimpleNamespace(**ig_consts)}
  tw_consts = _module_constants(tw_path, env)
  text = ('class _ImageGenerationGanModel(object):\n' + '\n\n'.join(base_methods) + '\n\n'
          '  @staticmethod\n  def _get_data_batched(batch_queue, batch_names, data_batched):\n    return data_batched if data_batched is not None else batch_queue.pop(0)\n\n\n'
          'class GanModel(_ImageGenerationGanModel):\n' + '\n\n'.join(top_methods) + '\n')
  import copy
  ns = dict(ig_consts)
  ns.update(tw_consts)
  ns.update({'tf': tf, 'FLAGS': tfs.FLAGS, 'copy': copy, 'functools': functools, 'util_misc': sys.modules['util_misc'],
             'pggan': pggan, 'slim': sys.modules['tensorflow.contrib.slim'], 'np': np})
  exec(compile(text, '<reference twingan.GanModel / image_generation.GanModel methods>', 'exec'), ns)
  return ns['GanModel'], ns


# SURVEY 8f-4: optional flags on the same wiring -- loss architectures (image_generation.py:330-389, 414-439) and the
# equalized learning rate (nets/pggan_utils.py:236-254); written to reference_f4.npz by `--f4`
F4_CLONE_CASES = [
    ('f4_wgan_gp8', 8, False, 0, 1000, 16, 'instance_norm', 3,
     dict(loss_architecture='wgan_gp', gradient_penalty_lambda=10.0, wgan_drift_loss_weight=0.1)),
    ('f4_wgan8', 8, False, 0, 1000, 16, 'instance_norm', 2, dict(loss_architecture='wgan', wgan_drift_loss_weight=0.0)),
    ('f4_hinge16grow', 16, True, 250, 1000, 16, 'instance_norm', 2, dict(loss_architecture='hinge')),
    ('f4_gan8', 8, False, 0, 1000, 16, 'batch_renorm', 3, dict(loss_architecture='gan')),
    ('f4_eqlr_dragan8', 8, False, 0, 1000, 16, 'instance_norm', 3, dict(equalized_learning_rate=True, _conv_std=1.0)),
    ('f4_res16grow', 16, True, 250, 1000, 16, 'instance_norm', 2, dict(use_res_block=True)),
    ('f4_res_eqlr_renorm8', 8, False, 0, 1000, 32, 'batch_renorm', 3, dict(use_res_block=True, equalized_learning_rate=True, _conv_std=1.0)),
    ('f4_eqlr_hinge64', 64, False, 0, 1000, 8, 'instance_norm', 2, dict(equalized_learning_rate=True, loss_architecture='hinge', _conv_std=1.0)),
]


def run_clone_case(tf, pggan, GanModel, ns, case, out):
  name, hw, growing, global_step, max_steps, mc, norm, batch = case[:8]
  extra = dict(case[8]) if len(case) > 8 else {}
  conv_std = extra.pop('_conv_std', 0.08)     # equalized lr multiplies every conv input by sqrt(2 / fan_in): N(0, 1) weights
  # wider 3x3 weights than N(0, 0.02) so that the discriminator's input gradients (DRAGAN slopes) are not ~0
  tfs.reset(stable_hash_provider(2, conv_std=conv_std), global_step=global_step)
  # several passes of one step share a domain's normaliser state; TF leaves read/write order between passes undefined
  # (SURVEY 8a.4-7).  Take the order in which every read of the step precedes every moving-average write.
  tfs.STORE.defer_updates = True
  F = tfs.FLAGS
  for k, v in dict(pggan_max_num_channels=mc, generator_norm_type=norm, generator_network='pggan', use_unet=True,
                   use_style_embedding=False, do_encoder_distillation=False, is_growing=growing,
                   grow_start_number_of_steps=0, max_number_of_steps=max_steps, do_self_attention=False,
                   self_attention_hw=64, do_pixel_norm=True, use_gdrop=False, use_conditional_labels=False,
                   loss_architecture='dragan', gan_weight=1.0, gradient_penalty_lambda=0.25, l_cyc_weight=1.0,
                   train_image_size=hw, do_l_cyc_gan=True, l_content_weight=0.1, wgan_drift_loss_weight=0.0,
                   equalized_learning_rate=False, use_res_block=False).items():
    setattr(F, k, v)
  for k, v in extra.items():
    setattr(F, k, v)
  arch = F.loss_architecture
  g = torch.Generator().manual_seed(500 + hw)
  # requires_grad: tf.gradients(prediction, interpolates) differentiates w.r.t. a tensor derived from the images
  sources = tfs.Tensor(torch.rand((batch, hw, hw, 3), generator=g, dtype=torch.float64).requires_grad_(True))
  targets = tfs.Tensor(torch.rand((batch, hw, hw, 3), generator=g, dtype=torch.float64).requires_grad_(True))
  # DRAGAN randomness in the order the reference draws it: per domain alpha [B,1,1,1] then noise [B,H,W,3]
  # (WGAN-GP: per domain one alpha [B,1,1,1], image_generation.py:421; gan / wgan / hinge draw nothing)
  draws, draw_keys = [], []
  for d_ in ('s', 't'):
    if arch in ('dragan', 'wgan_gp'):
      draws.append(torch.rand((batch, 1, 1, 1), generator=g, dtype=torch.float64))
      draw_keys.append('alpha_' + d_)
    if arch == 'dragan':
      draws.append(torch.rand((batch, hw, hw, 3), generator=g, dtype=torch.float64))
      draw_keys.append('noise_' + d_)
  tfs.STORE.random_queue = [d.clone() for d in draws]
  # the export placeholders (twingan.py:300-305) are fed the real batch: those eval-mode passes do not reach a loss
  tf.placeholder = lambda dtype, shape=None, name=None: tfs.Tensor(
      (sources if 'source' in (name or '') else targets).t.detach().clone())
  networks = {'generator_network_fn': pggan.generator, 'discriminator_network_fn': pggan.discriminator,
              'encoder_network_fn': pggan.encoder_before_classification}
  end_points = GanModel._clone_fn(networks, None, None, data_batched={'a_source': sources, 'b_source': targets},
                                  is_training=True, global_step=global_step)
  assert not tfs.STORE.random_queue, 'the reference drew less randomness than provided'
  gcol, dcol = ns['GENERATOR_LOSS_COLLECTION'], ns['DISCRIMINATOR_LOSS_COLLECTION']
  glosses, dlosses = tfs.STORE.losses[gcol], tfs.STORE.losses[dcol]
  g_total = sum(t.t for _, t in glosses)      # model_deploy._gather_clone_loss: tf.add_n(collection) / num_clones, one clone
  d_total = sum(t.t for _, t in dlosses)
  gvars = [(n, v) for n, v in tfs.STORE.vars.items() if v.trainable and not n.startswith('discriminator')]
  dvars = [(n, v) for n, v in tfs.STORE.vars.items() if v.trainable and n.startswith('discriminator')]
  ggrads = torch.autograd.grad(g_total, [v.t for _, v in gvars], retain_graph=True, allow_unused=True)
  dgrads = torch.autograd.grad(d_total, [v.t for _, v in dvars], allow_unused=True)

  f32 = lambda t: t.detach().to(torch.float32).numpy()
  out[name + '/meta'] = np.array([hw, int(growing), mc, batch, global_step, max_steps], dtype=np.int64)
  out[name + '/norm'] = np.array(norm)
  out[name + '/in/sources'] = sources.t.detach().numpy()
  out[name + '/in/targets'] = targets.t.detach().numpy()
  out[name + '/random_log'] = np.array([str(r) for r in tfs.STORE.random_log])
  for key, d in zip(draw_keys, draws):
    out[name + '/uniform01/' + key] = d.numpy()
  out[name + '/rng_stream'] = _stream(name, 500 + hw, [('in/sources', 'rand', sources.t.shape),
                                                       ('in/targets', 'rand', targets.t.shape)] +
                                      [('uniform01/' + k, 'rand', d.shape) for k, d in zip(draw_keys, draws)])
  out[name + '/extra_flags'] = np.array(json.dumps(extra, sort_keys=True))
  out[name + '/var_order'] = np.array(list(tfs.STORE.vars.keys()))
  out[name + '/var_trainable'] = np.array([bool(v.trainable) for v in tfs.STORE.vars.values()])
  out[name + '/var_shapes'] = np.array([str(list(v.t.shape)) for v in tfs.STORE.vars.values()])
  provider = stable_hash_provider(2, conv_std=conv_std)
  out[name + '/conv_std'] = np.array(conv_std)
  for n, v in tfs.STORE.vars.items():
    if v.trainable:
      out[name + '/var_sum/' + n] = np.array(float(v.t.detach().sum()))
    else:
      out[name + '/state_before/' + n] = provider(n, list(v.t.shape), None, False).numpy()
  out[name + '/gloss_names'] = np.array([sc for sc, _ in glosses])
  out[name + '/gloss_values'] = np.array([float(t.t) for _, t in glosses])
  out[name + '/dloss_names'] = np.array([sc for sc, _ in dlosses])
  out[name + '/dloss_values'] = np.array([float(t.t) for _, t in dlosses])
  out[name + '/generator_loss'] = np.array(float(g_total))
  out[name + '/discriminator_loss'] = np.array(float(d_total))
  for k in ('s_prime_output', 't_cycle_output', 'encoded_source_content_before_classification',
            'encoded_t_prime_content_before_classification', 'discriminator_real_s_prediction',
            'discriminator_s_prime_prediction', 'discriminator_t_cycle_prediction'):
    out[name + '/ep/' + k] = f32(end_points[k].t)
  # the export / inference graph of the same function (twingan.py:300-365; inference/image_translation_infer.py:46-99 runs
  # exactly this tensor): G(E(sources_ph; '_s', eval); '_t', eval, UNet skips) on the raw placeholder batch
  out[name + '/infer/custom_generated_t_style_source'] = f32(end_points[ns['CUSTOM_GENERATED_TARGETS']].t)
  out[name + '/end_point_keys'] = np.array(sorted(k for k, v in end_points.items() if isinstance(v, tfs.Tensor)))
  for (n, _), gr in list(zip(gvars, ggrads)) + list(zip(dvars, dgrads)):
    out[name + '/grad_is_none/' + n] = np.array(gr is None)
    if gr is not None:
      out[name + '/grad/' + n] = f32(gr)
  print('%-15s G losses: %s | D losses: %s' % (name, ', '.join('%s=%.4f' % (sc, float(t.t)) for sc, t in glosses),
                                                 ', '.join('%s=%.4f' % (sc, float(t.t)) for sc, t in dlosses)))


# ------------------------------------------------------------------------------------------------------------
# data parallelism: deployment/model_deploy.py create_clones / optimize_clones over two clones (SURVEY 8a18, 8e)
# ------------------------------------------------------------------------------------------------------------
def run_deploy_case(tf, pggan, GanModel, ns, out, name='deploy2_in8', hw=8, mc=16, norm='instance_norm', batch=2):
  from deployment import model_deploy          # the reference's (slim-derived) deployment module, imported as is
  tfs.reset(stable_hash_provider(3, conv_std=0.08), global_step=0)
  tfs.STORE.defer_updates = True
  F = tfs.FLAGS
  for k, v in dict(pggan_max_num_channels=mc, generator_norm_type=norm, generator_network='pggan', use_unet=True,
                   use_style_embedding=False, do_encoder_distillation=False, is_growing=False,
                   grow_start_number_of_steps=0, max_number_of_steps=1000, do_self_attention=False,
                   self_attention_hw=64, do_pixel_norm=True, use_gdrop=False, use_conditional_labels=False,
                   loss_architecture='dragan', gan_weight=1.0, gradient_penalty_lambda=0.25, l_cyc_weight=1.0,
                   train_image_size=hw, do_l_cyc_gan=True, l_content_weight=0.1).items():
    setattr(F, k, v)
  g = torch.Generator().manual_seed(900)
  batches, draws = [], []
  for c in range(2):
    s_ = tfs.Tensor(torch.rand((batch, hw, hw, 3), generator=g, dtype=torch.float64).requires_grad_(True))
    t_ = tfs.Tensor(torch.rand((batch, hw, hw, 3), generator=g, dtype=torch.float64).requires_grad_(True))
    batches.append({'a_source': s_, 'b_source': t_})
    for _ in ('s', 't'):
      draws.append(torch.rand((batch, 1, 1, 1), generator=g, dtype=torch.float64))
      draws.append(torch.rand((batch, hw, hw, 3), generator=g, dtype=torch.float64))
  tfs.STORE.random_queue = [d.clone() for d in draws]
  current = {'i': 0}

  def placeholder(dtype, shape=None, name=None):
    b = batches[min(current['i'], 1)]
    return tfs.Tensor((b['a_source'] if 'source' in (name or '') else b['b_source']).t.detach().clone())
  tf.placeholder = placeholder
  networks = {'generator_network_fn': pggan.generator, 'discriminator_network_fn': pggan.discriminator,
              'encoder_network_fn': pggan.encoder_before_classification}
  queue = list(batches)

  def model_fn(networks_, batch_queue, batch_names, **kw):
    r = GanModel._clone_fn(networks_, batch_queue, batch_names, **kw)
    current['i'] += 1
    return r
  config = model_deploy.DeploymentConfig(num_clones=2)
  clones = model_deploy.create_clones(config, model_fn, args=[networks, queue, None],
                                      kwargs={'is_training': True, 'global_step': 0})
  assert len(clones) == 2 and not queue and not tfs.STORE.random_queue

  class _Optimizer(object):       # tf.train.Optimizer.compute_gradients: d loss / d var for var in var_list
    def compute_gradients(self, loss, var_list=None, **unused):
      gs = torch.autograd.grad(loss.t, [v.t for v in var_list], retain_graph=True, allow_unused=True)
      return [(None if g_ is None else tfs.Tensor(g_), v) for g_, v in zip(gs, var_list)]

  gvars = [v for n, v in tfs.STORE.vars.items() if v.trainable and not n.startswith('discriminator')]
  dvars = [v for n, v in tfs.STORE.vars.items() if v.trainable and n.startswith('discriminator')]
  # image_generation.py:599-610
  g_loss, g_gv = model_deploy.optimize_clones(clones, _Optimizer(), gradient_scale=1.0,
                                              loss_collection=ns['GENERATOR_LOSS_COLLECTION'], var_list=gvars)
  d_loss, d_gv = model_deploy.optimize_clones(clones, _Optimizer(), gradient_scale=1.0,
                                              loss_collection=ns['DISCRIMINATOR_LOSS_COLLECTION'], var_list=dvars)
  out[name + '/meta'] = np.array([hw, mc, batch, 2], dtype=np.int64)
  out[name + '/norm'] = np.array(norm)
  out[name + '/clone_scopes'] = np.array([c.scope for c in clones])
  for c in range(2):
    out[name + '/in/sources_%d' % c] = batches[c]['a_source'].t.detach().numpy()
    out[name + '/in/targets_%d' % c] = batches[c]['b_source'].t.detach().numpy()
    for j, key in enumerate(('alpha_s', 'noise_s', 'alpha_t', 'noise_t')):
      out[name + '/uniform01/%s_%d' % (key, c)] = draws[4 * c + j].numpy()
  out[name + '/rng_stream'] = _stream(name, 900, [
      d for c in range(2) for d in [('in/sources_%d' % c, 'rand', batches[c]['a_source'].t.shape),
                                    ('in/targets_%d' % c, 'rand', batches[c]['b_source'].t.shape)] +
      [('uniform01/%s_%d' % (key, c), 'rand', draws[4 * c + j].shape)
       for j, key in enumerate(('alpha_s', 'noise_s', 'alpha_t', 'noise_t'))]])
  out[name + '/var_order'] = np.array([n for n, v in tfs.STORE.vars.items() if v.trainable])
  out[name + '/var_shapes'] = np.array([str(list(v.t.shape)) for n, v in tfs.STORE.vars.items() if v.trainable])
  out[name + '/generator_loss'] = np.array(float(g_loss.t))
  out[name + '/discriminator_loss'] = np.array(float(d_loss.t))
  for gr, v in list(g_gv) + list(d_gv):
    out[name + '/grad/' + v.name] = gr.t.detach().to(torch.float32).numpy()
  out[name + '/n_grads'] = np.array([len(g_gv), len(d_gv)])
  print('%-15s 2 clones %s: generator_loss=%.6f discriminator_loss=%.6f, %d + %d summed gradients' % (
      name, [c.scope for c in clones], float(g_loss.t), float(d_loss.t), len(g_gv), len(d_gv)))


# ------------------------------------------------------------------------------------------------------------
# flag defaults and the stage loop of pggan_runner.py
# ------------------------------------------------------------------------------------------------------------
def reference_flag_defaults(ref_root):
  """{flag name: default} from the tf.flags.DEFINE_* calls of the files on the path (read with ast, nothing executed)."""
  out = {}
  for rel in ('model/model_inheritor.py', 'image_generation.py', 'twingan.py', 'nets/pggan.py', 'pggan_runner.py'):
    tree = ast.parse(open(os.path.join(ref_root, rel)).read())
    for node in ast.walk(tree):
      if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr.startswith('DEFINE_') \
          and len(node.args) >= 2 and isinstance(node.args[0], ast.Constant):
        try:
          out[node.args[0].value] = ast.literal_eval(node.args[1])
        except ValueError:
          pass
  return out


def reference_stage_loop(ref_root, tf, flag_values):
  """Execute pggan_runner.main() (its own source; `.iteritems()` -> `.items()`) with a stub program object and record the
  flags it sets for every stage (pggan_runner.py:82-160)."""
  src = open(os.path.join(ref_root, 'pggan_runner.py')).read()
  tree = ast.parse(src)
  lines = src.split('\n')
  text = []
  for name in ('set_flags', 'main'):
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == name)
    text.append('\n'.join(lines[fn.lineno - 1:fn.end_lineno]).replace('.iteritems()', '.items()'))
  stages = []

  class _Program(object):
    def main(self):
      F = tfs.FLAGS
      stages.append({k: getattr(F, k) for k in ('is_growing', 'train_image_size', 'max_number_of_steps', 'train_dir',
                                                  'batch_size', 'ignore_missing_vars')}
                    | {'checkpoint_path': F._v.get('checkpoint_path')})

  for k, v in flag_values.items():
    setattr(tfs.FLAGS, k, v)
  tfs.FLAGS._v.pop('checkpoint_path', None)
  import math
  import time
  tf.train.latest_checkpoint = lambda d: None            # a fresh run: nothing trained yet
  tf.logging.set_verbosity = lambda *a, **k: None
  tf.reset_default_graph = lambda: None
  ns = {'tf': tf, 'FLAGS': tfs.FLAGS, 'os': os, 'ast': ast, 'math': math, 'time': time,
        'select_program': lambda name: _Program()}
  exec(compile('\n\n'.join(text), os.path.join(ref_root, 'pggan_runner.py'), 'exec'), ns)
  ns['main'](None)
  return stages


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--reference', required=True, help='checkout of the reference project (jerryli27/TwinGAN)')
  ap.add_argument('--out', default=os.path.join(HERE, 'reference_pggan.npz'))
  ap.add_argument('--f4', action='store_true', help='only the SURVEY 8f-4 optional-flag cases -> reference_f4.npz')
  args = ap.parse_args()
  tf, pggan, pggan_utils = load_reference(args.reference)
  out = {}
  if args.f4:
    GanModel, ns = build_reference_ganmodel(args.reference, tf, pggan)
    for case in F4_CLONE_CASES:
      run_clone_case(tf, pggan, GanModel, ns, case, out)
    path = os.path.join(os.path.dirname(args.out), 'reference_f4.npz')
    golden_store.save(path, out)
    print('wrote %s (%.1f MB, %d arrays)' % (path, os.path.getsize(path) / 1e6, len(out)))
    return
  for case in CASES:
    run_case(tf, pggan, pggan_utils, case, out)
  GanModel, ns = build_reference_ganmodel(args.reference, tf, pggan)
  for case in CLONE_CASES:
    run_clone_case(tf, pggan, GanModel, ns, case, out)
  run_deploy_case(tf, pggan, GanModel, ns, out)
  golden_store.save(args.out, out)
  import json
  meta = {'flag_defaults': reference_flag_defaults(args.reference)}
  for tag, fl in (('default', dict(train_dir='/ckpt', is_training=True, do_export=False, program_name='twingan',
                                   num_images_per_resolution=300000, start_hw=4, max_hw=256,
                                   hw_to_batch_size=meta['flag_defaults']['hw_to_batch_size'])),
                  ('small', dict(train_dir='/ckpt', is_training=True, do_export=False, program_name='twingan',
                                 num_images_per_resolution=1000, start_hw=8, max_hw=32,
                                 hw_to_batch_size='{8: 8, 16: 4, 32: 3}'))):
    meta['stages_' + tag] = reference_stage_loop(args.reference, tf, fl)
    meta['stages_' + tag + '_flags'] = fl
  jpath = os.path.join(os.path.dirname(args.out), 'reference_flags_and_stages.json')
  json.dump(meta, open(jpath, 'w'), indent=1, sort_keys=True, default=str)
  print('wrote %s (%d flag defaults, %d + %d stages)' % (jpath, len(meta['flag_defaults']), len(meta['stages_default']),
                                                        len(meta['stages_small'])))
  print('wrote %s (%.1f MB, %d arrays)' % (args.out, os.path.getsize(args.out) / 1e6, len(out)))


if __name__ == '__main__':
  main()
