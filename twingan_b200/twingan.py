"""TwinGAN model + trainer step -- host-side mirror of twingan.py (GanModel._clone_fn :146-445,
add_loss :451-521), the GAN losses of image_generation.py (:317-476), its optimisation
(:587-662, model/model_inheritor.py:515-565) and the data-parallel gradient aggregation of
deployment/model_deploy.py (:242-364, :473-503).

One `train_step` = everything a reference `session.run(train_tensor)` computes (all 16 network passes
+ the two DRAGAN passes, the generator-set AND discriminator-set gradients) followed by BOTH Adam
applies ("mode B", SURVEY 8d).  Data parallelism: one process per GPU, per-rank loss / world
(model_deploy.py:265-267) and ONE NCCL all-reduce(sum) over the flat gradient buffer replacing
tf.add_n (:499).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional

import torch

from . import ddp, ops, pggan
from . import pggan_utils as pu
from .variables import VariableStore

ENCODER_CONTENT_VAR_SCOPE = 'encoder_content'
GENERATOR_VAR_SCOPE = 'generator'
DISCRIMINATOR_VAR_SCOPE_SOURCE = 'discriminator_s'
DISCRIMINATOR_VAR_SCOPE_TARGET = 'discriminator_t'


@dataclass
class Flags:
  """The reference's tf.flags that reach the hot path (defaults: docs/training.md:10-37 recipe)."""
  train_image_size: int = 256
  is_growing: bool = False
  alpha_grow: float = 0.0                        # twingan.py:834-835 (computed from global_step there)
  pggan_max_num_channels: int = 256
  generator_norm_type: str = pu.INSTANCE_NORM_TYPE
  do_pixel_norm: bool = True
  use_unet: bool = True
  loss_architecture: str = 'dragan'
  gradient_penalty_lambda: float = 0.25
  gan_weight: float = 1.0
  l_cyc_weight: float = 1.0
  do_l_cyc_gan: bool = True
  l_content_weight: float = 0.1
  learning_rate: float = 1e-4
  adam_beta1: float = 0.5
  adam_beta2: float = 0.99
  opt_epsilon: float = 1e-8
  global_step: int = 0
  num_clones: int = 1                            # world size
  n_critic: int = 2                              # image_generation.py:87-90 (only used by train_step_alternating)
  # optional reference flags, off in the recipe (SURVEY 8f-4)
  equalized_learning_rate: bool = False          # nets/pggan.py:39-41
  wgan_drift_loss_weight: float = 0.0            # image_generation.py:96-98
  use_res_block: bool = False                    # nets/pggan.py:43-45
  # Engine option (not a reference flag): run the network passes that share conv weights as one batch each -- E(s),E(t)
  # -> one 2B pass, the four G passes -> one 4B pass, E(t'),E(s') -> one 2B pass, D_x(real, cycle, prime) -> one 3B pass
  # per domain -- instead of 16 separate passes.  Same arithmetic per sample; batch statistics stay per original pass.
  batch_passes: bool = True


class GanModel:
  """TwinGAN on one GPU (one clone).  `group` (torch.distributed process group or None) gives DDP."""

  def __init__(self, flags: Flags, device='cuda', seed: int = 1234, process_group=None):
    self.flags = flags
    self.device = torch.device(device)
    self.pg = process_group
    self.variables = VariableStore(self.device)
    pggan.declare_variables(self.variables, flags.train_image_size, flags.is_growing, flags.pggan_max_num_channels,
                            flags.use_unet, flags.generator_norm_type, flags.use_res_block)
    self.variables.materialize()
    self.variables.init_random(seed, 1.0 if flags.equalized_learning_rate else 0.02)
    self.flat_grad = torch.zeros_like(self.variables.flat)
    v = self.variables
    self._grad_view = {n: self.flat_grad[o:o + math.prod(s)].view(s) for n, (o, s) in v.offsets.items()}
    self.last_losses: Dict[str, torch.Tensor] = {}
    # Step counters {adam_t, global_step} live on the device (twg_step_schedule / twg_step_advance): the bias-corrected
    # Adam step sizes of the two applies and the batch-renorm clipping are derived from them INSIDE the step, so a
    # captured step can be replayed while time advances and no host buffer is in flight.  The host keeps mirrors
    # (variables.adam_t, flags.global_step); _sync_counters uploads them when they were changed from outside.
    self._counters = torch.zeros(2, device=self.device, dtype=torch.int32)
    self._counters_mirror = (0, 0)
    self._lr_dev = torch.zeros(2, device=self.device, dtype=torch.float32)
    self._clip_dev = torch.tensor([0.9, 1.1, 0.1], device=self.device, dtype=torch.float32)
    self._graph = None
    self._g_cut, self._d_cut = [], []            # in-step tensors autograd is asked about (compute_gradients)
    self.n_critic_counter = 0                    # image_generation.py:622

  def _sync_counters(self):
    want = (int(self.variables.adam_t), int(self.flags.global_step))
    if want != self._counters_mirror:
      self._counters.copy_(torch.tensor(want, dtype=torch.int32))     # pageable source: complete when copy_ returns
      self._counters_mirror = want

  def _schedule(self):
    """lr_t of the step's two Adam applies and the renorm clipping, from the device counters."""
    from ._lib import lib
    f = self.flags
    lib().call('twg_step_schedule', self._counters.data_ptr(), float(f.learning_rate), float(f.adam_beta1),
               float(f.adam_beta2), self._lr_dev.data_ptr(), self._clip_dev.data_ptr(), ops._st())

  # -- scopes -----------------------------------------------------------------------------------
  def _gen_scope(self, var_scope, postfix, is_training, stats, tags=None):
    f = self.flags
    return pu.pggan_generator_arg_scope(self.variables, var_scope, f.generator_norm_type, postfix, is_training,
                                        f.global_step, stats, self._clip_dev if is_training else None, tags,
                                        f.equalized_learning_rate, f.use_res_block)

  def _encoder(self, x, postfix, is_training=True, stats=None, tags=None):
    """`postfix`: '_s' / '_t', or a tuple of them -- one per equal block of the batch (batched passes)."""
    f = self.flags
    return pggan.encoder_before_classification(
        x, is_training=is_training, is_growing=f.is_growing, alpha_grow=f.alpha_grow,
        max_num_channels=f.pggan_max_num_channels,
        arg_scope=self._gen_scope(ENCODER_CONTENT_VAR_SCOPE, postfix, is_training, stats, tags),
        do_pixel_norm=f.do_pixel_norm)

  def _generator(self, code, postfix, unet, target_shape, is_training=True, stats=None, tags=None):
    f = self.flags
    return pggan.generator(
        code, is_training=is_training, is_growing=f.is_growing, alpha_grow=f.alpha_grow, target_shape=target_shape,
        max_num_channels=f.pggan_max_num_channels,
        arg_scope=self._gen_scope(GENERATOR_VAR_SCOPE, postfix, is_training, stats, tags),
        do_pixel_norm=f.do_pixel_norm, unet_end_points=unet if f.use_unet else None)

  def _discriminator(self, x, var_scope, groups=1):
    f = self.flags
    return pggan.discriminator(x, is_training=True, is_growing=f.is_growing, alpha_grow=f.alpha_grow,
                               arg_scope=pu.pggan_discriminator_arg_scope(self.variables, var_scope, True,
                                                                          f.equalized_learning_rate, f.use_res_block),
                               max_num_channels=f.pggan_max_num_channels, minibatch_groups=groups)

  # -- graph (twingan.py:146-445) -------------------------------------------------------------------
  def clone_fn(self, sources, targets, dragan_rand):
    """Forward of all passes + losses.  Returns (generator_loss, discriminator_loss, named, end_points, stats)."""
    if self.flags.batch_passes:
      return self._clone_fn_batched(sources, targets, dragan_rand)
    return self._clone_fn_pass_by_pass(sources, targets, dragan_rand)

  # order of the reference's passes (twingan.py:198-284): E(s) E(t) G->s' G->s~ G->t' G->t~ E(t') E(s').  The batched
  # layout is E1 = [s | t], G = [s_cycle | t_cycle | t_prime | s_prime], E2 = [t_prime | s_prime], D_x = [real | cycle | prime]
  _E1_TAGS, _G_TAGS, _E2_TAGS = (1, 2), (4, 6, 5, 3), (7, 8)

  def _clone_fn_batched(self, sources, targets, dragan_rand):
    f = self.flags
    B = int(sources.shape[0])
    stats = []
    x = ops.cat_batch(sources, targets)
    if f.is_growing:   # twingan.py:827-839
      x = ops.growing_image(x, f.alpha_grow)
    # Autograd is asked for gradients w.r.t. tensors born inside the step (see compute_gradients): the image batch for the
    # generator-loss backward, the discriminators' inputs for the discriminator-loss backward.
    x.requires_grad_(True)
    self._g_cut, self._d_cut = [x], []
    with ops.trace_tag('E1'):
      enc, ep = self._encoder(x, ('_s', '_t'), stats=stats, tags=self._E1_TAGS)
    with ops.trace_tag('G'):
      # s_cycle = G(enc_s;_s), t_cycle = G(enc_t;_t), t_prime = G(enc_s;_t), s_prime = G(enc_t;_s): codes and UNet skips are
      # the encoder batch used twice (the skip is indexed n % 2B by the join kernel)
      gout, _ = self._generator(ops.repeat_batch(enc), ('_s', '_t', '_t', '_s'), ep, (4 * B,) + tuple(x.shape[1:]),
                                stats=stats, tags=self._G_TAGS)
    d_s_in, d_t_in, e2_in, l_cyc_s, l_cyc_t = ops.FanoutFn.apply(gout, x, f.l_cyc_weight)
    self._d_cut += [d_s_in, d_t_in]
    with ops.trace_tag('E2'):
      enc2, _ = self._encoder(e2_in, ('_t', '_s'), stats=stats, tags=self._E2_TAGS)
    with ops.trace_tag('Ds'):
      pred_s, _ = self._discriminator(d_s_in, DISCRIMINATOR_VAR_SCOPE_SOURCE, groups=3)
    with ops.trace_tag('Dt'):
      pred_t, _ = self._discriminator(d_t_in, DISCRIMINATOR_VAR_SCOPE_TARGET, groups=3)
    gl, dl = {}, {}
    gl['l_cyc_s'], gl['l_cyc_t'] = l_cyc_s, l_cyc_t
    cyc = f.train_image_size >= 64 and f.do_l_cyc_gan       # twingan.py:466
    for dom, pred, dscope in (('s', pred_s, DISCRIMINATOR_VAR_SCOPE_SOURCE), ('t', pred_t, DISCRIMINATOR_VAR_SCOPE_TARGET)):
      original = x.detach()[0:B] if dom == 's' else x.detach()[B:2 * B]
      if f.loss_architecture in ('gan', 'dragan'):
        fool_c, fool_p, fake_c, real_c, fake_p, real_p = ops.GanLossesFn.apply(pred, f.gan_weight)
        if cyc:
          gl['generator_fool_loss_cycle_' + dom] = fool_c
          dl['discriminator_fake_loss_cycle_' + dom] = fake_c
          dl['discriminator_real_loss_cycle_' + dom] = real_c
        gl['generator_fool_loss_prime_' + dom] = fool_p
        dl['discriminator_fake_loss_prime_' + dom] = fake_p
        dl['discriminator_real_loss_prime_' + dom] = real_p
        if f.loss_architecture == 'dragan':
          with ops.trace_tag('DR' + dom):
            dl['discriminator_gradient_penalty_prime_' + dom] = self._add_dragan_loss(
                original, dscope, dragan_rand['alpha_' + dom], dragan_rand['noise_' + dom])
      else:
        # wgan / wgan_gp / hinge (SURVEY 8f-4): the terms of add_gan_loss on the blocks [real | cycle | prime] of the batch
        real_pred = pred[0:B]
        for post, fake_pred in ((('cycle', pred[B:2 * B]),) if cyc else ()) + (('prime', pred[2 * B:3 * B]),):
          fake_img = gout[3 * B:4 * B] if dom == 's' else gout[2 * B:3 * B]     # s_prime / t_prime (only used for 'prime')
          with ops.trace_tag('DR' + dom):
            self._add_gan_loss_optional(gl, dl, dom, post, fake_pred, real_pred, fake_img, original, dscope, dragan_rand)
    if f.l_content_weight:
      # l_content_s = |enc_s - enc_t_prime|, l_content_t = |enc_t - enc_s_prime| (twingan.py:485-505): block g of enc vs enc2
      gl['l_content_s'], gl['l_content_t'] = ops.L1GroupsFn.apply(enc2, enc, f.l_content_weight)
    inv = 1.0 / f.num_clones
    g_loss = ops.sum_scalars(list(gl.values()), inv)
    d_loss = ops.sum_scalars(list(dl.values()), inv)
    named = dict(gl)
    named.update(dl)
    with torch.no_grad():
      ends = {'sources': x[0:B], 'targets': x[B:2 * B], 's_cycle': gout[0:B], 't_cycle': gout[B:2 * B],
              't_prime': gout[2 * B:3 * B], 's_prime': gout[3 * B:4 * B], 'enc_s': enc[0:B], 'enc_t': enc[B:2 * B],
              'enc_t_prime': enc2[0:B], 'enc_s_prime': enc2[B:2 * B],
              'pred_real_s': pred_s[0:B], 'pred_s_cycle': pred_s[B:2 * B], 'pred_s_prime': pred_s[2 * B:3 * B],
              'pred_real_t': pred_t[0:B], 'pred_t_cycle': pred_t[B:2 * B], 'pred_t_prime': pred_t[2 * B:3 * B]}
    stats.sort(key=lambda e: e[4])     # EMA pushes in the reference's program order (stable: layers stay in order)
    return g_loss, d_loss, named, ends, stats

  @staticmethod
  def trace_in_reference_order(trace, batch):
    """Test hook: ops.ACTIVE_SET_TRACE of a batched step -> the per-pass, program-order lists the parity harness consumes."""
    B = int(batch)
    by_tag = {}
    for tag, t in trace['lrelu']:
      by_tag.setdefault(tag, []).append(t)
    if None in by_tag or 'E1' not in by_tag:       # pass-by-pass step: already in program order
      return {'lrelu': [t for _, t in trace['lrelu']], 'l1': [t for _, t in trace['l1']]}
    order = [('E1', 0), ('E1', 1), ('G', 3), ('G', 0), ('G', 2), ('G', 1), ('E2', 0), ('E2', 1),
             ('Ds', 0), ('Ds', 2), ('Ds', 1), ('Dt', 0), ('Dt', 2), ('Dt', 1)]
    lrelu = []
    for tag, blk in order:
      lrelu.extend(t[blk * B:(blk + 1) * B] for t in by_tag[tag])
    lrelu.extend(by_tag.get('DRs', []))
    lrelu.extend(by_tag.get('DRt', []))
    l1s = [t for _, t in trace['l1']]            # [l_cyc (s|t), l_content (s|t)]
    l1 = [l1s[0][0:B]] + ([l1s[1][0:B]] if len(l1s) > 1 else []) + [l1s[0][B:2 * B]] + ([l1s[1][B:2 * B]] if len(l1s) > 1 else [])
    return {'lrelu': lrelu, 'l1': l1}

  def _clone_fn_pass_by_pass(self, sources, targets, dragan_rand):
    """The reference's own pass structure (16 separate network passes); kept as the A/B and parity twin of the batched
    step (tests/test_gpu_fullsize.py holds the two to each other at the full 256x256 size)."""
    f = self.flags
    stats = []
    if f.is_growing:   # twingan.py:827-839
      sources = ops.growing_image(sources, f.alpha_grow)
      targets = ops.growing_image(targets, f.alpha_grow)
    # in-step leaves autograd is asked about (compute_gradients): the encoder inputs for the generator-loss backward;
    # separate leaves for the discriminators' real passes, so the discriminator-loss backward stops at D's inputs
    sources = sources.detach().requires_grad_(True)
    targets = targets.detach().requires_grad_(True)
    real_s = sources.detach().requires_grad_(True)
    real_t = targets.detach().requires_grad_(True)
    self._g_cut, self._d_cut = [sources, targets], [real_s, real_t]
    enc_s, ep_s = self._encoder(sources, '_s', stats=stats)
    enc_t, ep_t = self._encoder(targets, '_t', stats=stats)
    s_prime, _ = self._generator(enc_t, '_s', ep_t, sources.shape, stats=stats)
    s_cycle, _ = self._generator(enc_s, '_s', ep_s, sources.shape, stats=stats)
    t_prime, _ = self._generator(enc_s, '_t', ep_s, targets.shape, stats=stats)
    t_cycle, _ = self._generator(enc_t, '_t', ep_t, targets.shape, stats=stats)
    enc_t_prime, _ = self._encoder(t_prime, '_t', stats=stats)
    enc_s_prime, _ = self._encoder(s_prime, '_s', stats=stats)
    self._d_cut += [s_prime, s_cycle, t_prime, t_cycle]
    ends = {'sources': sources, 'targets': targets, 's_prime': s_prime, 's_cycle': s_cycle, 't_prime': t_prime,
            't_cycle': t_cycle, 'enc_s': enc_s, 'enc_t': enc_t, 'enc_s_prime': enc_s_prime,
            'enc_t_prime': enc_t_prime}
    preds = {
        'real_s': self._discriminator(real_s, DISCRIMINATOR_VAR_SCOPE_SOURCE)[0],
        's_prime': self._discriminator(s_prime, DISCRIMINATOR_VAR_SCOPE_SOURCE)[0],
        's_cycle': self._discriminator(s_cycle, DISCRIMINATOR_VAR_SCOPE_SOURCE)[0],
        'real_t': self._discriminator(real_t, DISCRIMINATOR_VAR_SCOPE_TARGET)[0],
        't_prime': self._discriminator(t_prime, DISCRIMINATOR_VAR_SCOPE_TARGET)[0],
        't_cycle': self._discriminator(t_cycle, DISCRIMINATOR_VAR_SCOPE_TARGET)[0],
    }
    ends.update({'pred_' + k: v for k, v in preds.items()})
    g_losses, d_losses = self.add_loss(ends, preds, dragan_rand)
    inv = 1.0 / f.num_clones
    g_loss = ops.sum_scalars(list(g_losses.values()), inv)
    d_loss = ops.sum_scalars(list(d_losses.values()), inv)
    named = dict(g_losses)
    named.update(d_losses)
    return g_loss, d_loss, named, ends, stats

  # -- losses (twingan.py:451-521, image_generation.py:317-476) ------------------------------------
  def add_loss(self, ends, preds, dragan_rand):
    f = self.flags
    gl, dl = {}, {}
    for dom in ('s', 't'):
      opp = 't' if dom == 's' else 's'
      original = ends['sources'] if dom == 's' else ends['targets']
      dscope = DISCRIMINATOR_VAR_SCOPE_SOURCE if dom == 's' else DISCRIMINATOR_VAR_SCOPE_TARGET
      gl['l_cyc_' + dom] = ops.absolute_difference(original, ends[dom + '_cycle'], f.l_cyc_weight)
      real_pred = preds['real_' + dom]
      posts = (['cycle'] if (f.train_image_size >= 64 and f.do_l_cyc_gan) else []) + ['prime']
      for post in posts:
        fake_pred = preds['%s_%s' % (dom, post)]
        if f.loss_architecture not in ('gan', 'dragan'):
          self._add_gan_loss_optional(gl, dl, dom, post, fake_pred, real_pred, ends['%s_%s' % (dom, post)], original, dscope,
                                      dragan_rand)
          continue
        gl['generator_fool_loss_%s_%s' % (post, dom)] = ops.sigmoid_cross_entropy(1.0, fake_pred, f.gan_weight)
        dl['discriminator_fake_loss_%s_%s' % (post, dom)] = ops.sigmoid_cross_entropy(0.0, fake_pred, f.gan_weight)
        dl['discriminator_real_loss_%s_%s' % (post, dom)] = ops.sigmoid_cross_entropy(1.0, real_pred, f.gan_weight)
        if post == 'prime' and f.loss_architecture == 'dragan':
          dl['discriminator_gradient_penalty_prime_' + dom] = self._add_dragan_loss(
              original, dscope, dragan_rand['alpha_' + dom], dragan_rand['noise_' + dom])
      if f.l_content_weight:
        gl['l_content_' + dom] = ops.absolute_difference(ends['enc_' + dom], ends['enc_%s_prime' % opp],
                                                         f.l_content_weight)
    return gl, dl

  def _add_gan_loss_optional(self, gl, dl, dom, post, fake_pred, real_pred, fake_image, real_image, dscope, rand):
    """add_gan_loss for --loss_architecture wgan / wgan_gp / hinge (image_generation.py:330-389); `post` = 'cycle' is the
    only_real_fake_loss call of twingan.py:467-474."""
    f = self.flags
    arch, w = f.loss_architecture, f.gan_weight
    if arch not in ('wgan', 'wgan_gp', 'hinge'):
      raise NotImplementedError('unsupported loss architecture: %s' % arch)      # image_generation.py:401
    key = '%s_%s' % (post, dom)
    gl['generator_fool_loss_' + key] = ops.logit_mean(fake_pred, -1.0, 0.0, 0, w)          # -mean(D(G)), :332-336
    if arch == 'hinge':                                                                    # :381-389
      dl['discriminator_loss_' + key] = ops.sum_scalars([ops.logit_mean(fake_pred, 1.0, 1.0, 1, w),
                                                         ops.logit_mean(real_pred, -1.0, 1.0, 1, w)])
      return
    dl['discriminator_loss_' + key] = ops.sum_scalars([ops.logit_mean(fake_pred, 1.0, 0.0, 0, w),     # :348-355
                                                       ops.logit_mean(real_pred, -1.0, 0.0, 0, w)])
    if post == 'cycle':
      return
    if f.wgan_drift_loss_weight:                                                           # :359-367
      dl['discriminator_drift_loss_' + key] = ops.logit_mean(real_pred, 1.0, 0.0, 2, f.wgan_drift_loss_weight)
    if arch == 'wgan_gp':                                                                  # :372-379
      dl['discriminator_gradient_penalty_' + key] = self._add_wgan_gp_loss(real_image, fake_image, dscope, rand['alpha_' + dom])

  def _add_wgan_gp_loss(self, real_image, generated_image, dscope, alpha):
    """image_generation.py:414-439: penalty on D's input gradient at real + alpha (generated - real), alpha ~U[0,1]
    [B,1,1,1] an explicit input.  The term lives in the discriminator collection, so the interpolate is a leaf."""
    with torch.no_grad():
      real, fake = real_image.detach(), generated_image.detach()
      diff = ops.AxpbyFn.apply(fake, real, 1.0, -1.0)
      step = torch.empty_like(diff)
      from ._lib import lib
      B = int(real.shape[0])
      lib().call('twg_scale_rows', diff.data_ptr(), ops._check(alpha).data_ptr(), ops._one(diff.device).data_ptr(),
                 step.data_ptr(), B, diff.numel() // B, ops._st())
      xhat = ops.AxpbyFn.apply(real.contiguous(), step, 1.0, 1.0)
    xhat.requires_grad_(True)
    return self._gradient_penalty_at(xhat, dscope)

  def _gradient_penalty_at(self, xhat, dscope):
    self._d_cut.append(xhat)
    pred, _ = self._discriminator(xhat, dscope)
    seed = torch.ones_like(pred).requires_grad_(True)
    self._d_cut.append(seed)
    with ops.skip_param_grads('D'):   # tf.gradients(pred, [interpolates]) only walks to the input
      (grad,) = torch.autograd.grad(pred, xhat, grad_outputs=seed, create_graph=True)
    return ops.gradient_penalty(grad, self.flags.gradient_penalty_lambda)

  def _add_dragan_loss(self, real_image, dscope, alpha, noise):
    """image_generation.py:451-476; alpha ~U[0,1] [B,1,1,1] and noise ~U[-1,1] are explicit inputs."""
    xhat = ops.dragan_xhat(real_image.detach(), alpha, noise).requires_grad_(True)
    self._d_cut.append(xhat)
    pred, _ = self._discriminator(xhat, dscope)
    # the seed is an in-step leaf too: the top layer's double-backward node has no other differentiable ancestor than the
    # weights, and the engine only visits nodes that lead to a tensor it was asked about (compute_gradients)
    seed = torch.ones_like(pred).requires_grad_(True)
    self._d_cut.append(seed)
    with ops.skip_param_grads('D'):   # tf.gradients(pred, [interpolates]) only walks to the input
      (grad,) = torch.autograd.grad(pred, xhat, grad_outputs=seed, create_graph=True)
    return ops.gradient_penalty(grad, self.flags.gradient_penalty_lambda)

  # -- gradients + optimisation (image_generation.py:587-662) ---------------------------------------
  def compute_gradients(self, sources, targets, dragan_rand, after_generator_backward=None):
    """Both gradient sets of one step into the flat gradient buffer.  Every parameter gradient is accumulated straight
    into its slice of that buffer by the kernel that produces it ("sinks": wgrad atomics, normaliser / bias column
    sums), so autograd neither sums per-use gradients of a shared variable nor packs them afterwards.
    `after_generator_backward`: callback run between the two backward passes (gradient all-reduce overlap)."""
    v = self.variables
    ops.begin_step()
    self._sync_counters()
    self._schedule()
    v.snapshot_state()
    self.flat_grad.zero_()
    ops.register_grad_sinks({v[n].data_ptr(): self._grad_view[n] for n in v.offsets})
    ops.require_sinks(True)
    try:
      g_loss, d_loss, named, ends, stats = self.clone_fn(sources, targets, dragan_rand)
      # No parameter gradient travels through autograd (they all land in their sinks), so autograd is asked for the
      # gradients w.r.t. tensors created inside this step -- the image batch for the generator loss; the discriminators'
      # inputs, which also cut the walk off before it would enter G and E, for the discriminator loss -- instead of the
      # persistent variables.  Besides being all the engine needs to visit the right nodes (var_list semantics come from
      # skip_param_grads), this keeps the engine from synchronising with the streams the variables' gradient
      # accumulators were created on, which a CUDA-graph capture of the step does not survive.
      with ops.skip_param_grads('D'):
        torch.autograd.grad(g_loss, self._g_cut, retain_graph=True, allow_unused=True)
      if after_generator_backward is not None:
        after_generator_backward()       # the generator-set slice of the buffer is final from here on
      with ops.skip_param_grads('G'):
        torch.autograd.grad(d_loss, self._d_cut, allow_unused=True)
      ops.flush_padded_sinks()
    finally:
      ops.drop_padded_sinks()
      ops.require_sinks(False)
      ops.register_grad_sinks({})      # sinks are only valid while this model's step is being differentiated
      self._g_cut, self._d_cut = [], []
    self.last_losses = {'generator_loss': g_loss.detach(), 'discriminator_loss': d_loss.detach()}
    self.last_losses.update({k: t.detach() for k, t in named.items()})
    return g_loss.detach(), d_loss.detach(), ends, stats

  def allreduce_gradients(self, group: Optional[str] = None):
    """deployment/model_deploy.py:473-503 (tf.add_n over clones) -> NCCL all-reduce(sum) of the flat bucket ('G' / 'D' set
    or, with group=None, the whole buffer).  The 1/num_clones factor is already in the loss (model_deploy.py:265-267)."""
    if self.pg is not None:
      ddp.allreduce_flat_(self.flat_grad if group is None else self.variables.group_slice(self.flat_grad, group), self.pg)

  def apply_gradients(self):
    """Generator apply then discriminator apply, one shared Adam (beta powers advance per apply;
    SURVEY 8a.4-5/8; image_generation.py:640-646)."""
    self._apply_gradients_kernels()
    self._advance_host_mirrors()

  def _advance_host_mirrors(self):
    self.variables.adam_t += 2
    self.flags.global_step += 1
    self._counters_mirror = (self._counters_mirror[0] + 2, self._counters_mirror[1] + 1)

  def _apply_gradients_kernels(self):
    """Device side of the two applies: Adam on both groups with the step sizes twg_step_schedule derived from the device
    counters, one launch that rebuilds the split-bf16 planes of every conv weight, counters += (2, 1)."""
    from ._lib import lib
    f, v = self.flags, self.variables
    for i, group in enumerate(('G', 'D')):
      ops.adam_(v.group_slice(v.flat, group), v.group_slice(self.flat_grad, group), v.group_slice(v.adam_m, group),
                v.group_slice(v.adam_v, group), self._lr_dev[i:i + 1], f.adam_beta1, f.adam_beta2, f.opt_epsilon)
    if v.weight_table is not None:
      v.weight_table.refresh()
    lib().call('twg_step_advance', self._counters.data_ptr(), 2, 1, ops._st())

  def apply_stat_updates(self, stats):
    """EMA pushes in program order (libs/batch_norm.py:295-319, 359-393)."""
    for key, kind, C, batch_stats, *_ in stats:
      # batch_renorm is configured with decay 0.99 (nets/pggan_utils.py:165); plain batch_norm keeps
      # conditional_batch_norm's default 0.999 (libs/batch_norm.py:44)
      ops.norm_update_stats(self.variables.state_record(key), batch_stats, kind, C,
                            decay=0.99 if kind == ops.NORM_RENORM else 0.999)

  # -- gradient all-reduce overlapped with the discriminator backward ---------------------------------------------
  def _comm_stream(self):
    if getattr(self, '_comm', None) is None:
      self._comm = torch.cuda.Stream(device=self.device)
    return self._comm

  def _allreduce_async(self, group):
    """Launch the all-reduce of one gradient set on the side stream once the main stream has produced it."""
    comm = self._comm_stream()
    comm.wait_stream(torch.cuda.current_stream(self.device))
    with torch.cuda.stream(comm):
      self.allreduce_gradients(group)

  def train_step(self, sources, targets, dragan_rand):
    """Mode B (SURVEY 8d): one batch, both gradient sets, BOTH Adam applies -- the measured unit.  With a process group
    the generator-set all-reduce runs on a side stream while the discriminator backward computes."""
    overlap = self.pg is not None and self.device.type == 'cuda'
    g_loss, d_loss, ends, stats = self.compute_gradients(
        sources, targets, dragan_rand, (lambda: self._allreduce_async('G')) if overlap else None)
    if overlap:
      self._allreduce_async('D')
      torch.cuda.current_stream(self.device).wait_stream(self._comm_stream())
    else:
      self.allreduce_gradients()
    self.apply_gradients()
    self.apply_stat_updates(stats)
    return g_loss, d_loss

  def train_step_alternating(self, sources, targets, dragan_rand):
    """Mode A, the reference's own trajectory (image_generation.py:599-655): every run computes BOTH gradient sets but
    applies only one -- the generator set when n_critic_counter % n_critic == 0 (so the very first run is a generator
    turn), the discriminator set otherwise; the counter advances on every apply, global_step only on generator turns,
    and the single Adam object's beta powers advance on every apply.  The normalisers' moving-average pushes are
    created outside the tf.cond branches and attached as control dependencies, so they run on every turn.
    Returns (generator_loss, discriminator_loss, 'G' | 'D')."""
    f, v = self.flags, self.variables
    g_loss, d_loss, ends, stats = self.compute_gradients(sources, targets, dragan_rand)
    self.allreduce_gradients()
    turn = 'G' if self.n_critic_counter % f.n_critic == 0 else 'D'
    v.adam_t += 1
    t = v.adam_t
    lr_t = f.learning_rate * math.sqrt(1.0 - f.adam_beta2 ** t) / (1.0 - f.adam_beta1 ** t)
    ops.adam_(v.group_slice(v.flat, turn), v.group_slice(self.flat_grad, turn), v.group_slice(v.adam_m, turn),
              v.group_slice(v.adam_v, turn), lr_t, f.adam_beta1, f.adam_beta2, f.opt_epsilon)
    if v.weight_table is not None:
      v.weight_table.refresh()
    self.apply_stat_updates(stats)
    self.n_critic_counter += 1
    if turn == 'G':
      f.global_step += 1
    return g_loss, d_loss, turn

  # -- CUDA-graph replay of the whole step -------------------------------------------------------------
  def capture(self, sources, targets, dragan_rand, warmup: int = 2):
    """Capture the step as CUDA graphs over static input buffers: forward + generator-set backward, discriminator-set
    backward, and the two Adam applies + weight-plane rebuild + EMA pushes + counter advance.  `train_step_graphed` then
    copies a batch into the static buffers and replays them (the gradient all-reduces are eager NCCL calls on a side
    stream in between).  The warm-up steps run on the live buffers; parameters, optimiser slots, normaliser state and the
    step counters are restored afterwards, so capturing leaves the model exactly where it was."""
    assert self.device.type == 'cuda'
    from ._lib import lib
    v = self.variables
    self._sync_counters()
    saved = [t.clone() for t in (v.flat, v.adam_m, v.adam_v, v.state, v.state_snapshot, self._counters)]
    saved_host = (v.adam_t, self.flags.global_step, self._counters_mirror)
    self._static = {'s': sources.clone(), 't': targets.clone(), 'r': {k: t.clone() for k, t in dragan_rand.items()}}
    side = torch.cuda.Stream(device=self.device)      # warm-up AND capture run on this one stream
    side.wait_stream(torch.cuda.current_stream(self.device))
    with torch.cuda.stream(side):
      for _ in range(warmup):
        _, _, _, stats = self.compute_gradients(self._static['s'], self._static['t'], self._static['r'])
        self._apply_gradients_kernels()
        self.apply_stat_updates(stats)
    torch.cuda.current_stream(self.device).wait_stream(side)
    torch.cuda.synchronize(self.device)
    with torch.no_grad():
      for dst, src in zip((v.flat, v.adam_m, v.adam_v, v.state, v.state_snapshot, self._counters), saved):
        dst.copy_(src)
    v.adam_t, self.flags.global_step, self._counters_mirror = saved_host
    if v.weight_table is not None:
      v.weight_table.refresh()             # planes of the restored weights; graph 1 only looks them up
    torch.cuda.synchronize(self.device)
    L = lib()
    n0 = L.launch_count()
    st = self._static
    # graph 1a: forward of all passes + generator-set backward; graph 1b: discriminator-set backward.  autograd's tape
    # lives across the two captures (retain_graph), so the split point is the callback inside compute_gradients; both
    # graphs share one memory pool and are always replayed in this order.
    self._g1a = torch.cuda.CUDAGraph()
    self._g1b = torch.cuda.CUDAGraph()
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    cap_stream = side
    cap_stream.wait_stream(torch.cuda.current_stream(self.device))
    with torch.cuda.stream(cap_stream):
      self._g1a.capture_begin()

      def split():
        self._g1a.capture_end()
        self._g1b.capture_begin(pool=self._g1a.pool())

      gl, dl, _, stats = self.compute_gradients(st['s'], st['t'], st['r'], after_generator_backward=split)
      self._g1b.capture_end()
    torch.cuda.current_stream(self.device).wait_stream(cap_stream)
    st['gl'], st['dl'] = gl, dl
    self._g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(self._g2, pool=self._g1a.pool()):
      self._apply_gradients_kernels()
      self.apply_stat_updates(stats)
    self.launches_per_step = L.launch_count() - n0
    # the capture itself executed nothing, but _apply_gradients_kernels marked the planes fresh: they still are
    self._graph = True

  def train_step_graphed(self, sources, targets, dragan_rand):
    st = self._static
    st['s'].copy_(sources, non_blocking=True)
    st['t'].copy_(targets, non_blocking=True)
    for k, t in dragan_rand.items():
      st['r'][k].copy_(t, non_blocking=True)
    self._sync_counters()
    if self.variables.weight_table is not None and self.variables.weight_table.dirty:
      self.variables.weight_table.refresh()      # variables were changed from outside since the last apply
    self._g1a.replay()
    if self.pg is not None:
      self._allreduce_async('G')
    self._g1b.replay()
    if self.pg is not None:
      self._allreduce_async('D')
      torch.cuda.current_stream(self.device).wait_stream(self._comm_stream())
    self._g2.replay()
    self._advance_host_mirrors()
    return st['gl'], st['dl']

  # -- inference (inference/image_translation_infer.py:46-99; twingan.py:310-365) --------------------
  @torch.no_grad()
  def infer(self, sources):
    """custom_generated_t_style_source: G(E(x; '_s', eval); '_t', eval, UNet skips)."""
    code, ep = self._encoder(sources, '_s', is_training=False)
    out, _ = self._generator(code, '_t', ep, sources.shape, is_training=False)
    return out


class InferencePipeline(object):
  """Pipelined translation of streams of HOST image batches (the loop of inference/image_translation_infer.py:88-99).
  `run(host_batches)` yields (pinned host output, event) per batch -- wait on the event before reading.  The host->device
  copy of batch k+1 and the device->host copy of result k-1 run on side streams while batch k computes; the device
  staging slots and the pinned result slots are allocated once and reused across `run` calls.
  `use_graph`: the ~90 kernel launches of a batch are captured once per batch shape into a CUDA graph over a static input
  buffer and replayed.  The tensor-core convs of the graph read the weights through the persistent weight-plane table,
  which the replay cannot rebuild by itself: `_infer` refreshes the table first when the variables changed since it was
  last built (`load_dict`, `init_random`), so a replay after a reload translates with the new weights."""

  def __init__(self, model: GanModel, depth: int = 2, use_graph: bool = False):
    from .prefetch import HostReturner
    self.model, self.depth = model, depth
    self.feed = None
    self.back = HostReturner(model.device, depth)
    self.use_graph = bool(use_graph) and model.device.type == 'cuda'
    self._graphs = {}            # batch shape -> (graph, static input, static output)

  def _infer(self, x):
    if not self.use_graph:
      return self.model.infer(x)
    key = tuple(x.shape)
    ent = self._graphs.get(key)
    if ent is None:
      dev = self.model.device
      static_in = x.clone()
      side = torch.cuda.Stream(device=dev)
      side.wait_stream(torch.cuda.current_stream(dev))
      with torch.cuda.stream(side):
        for _ in range(2):                              # warm-up on the capture stream (lazy one-time set-up, allocator)
          self.model.infer(static_in)
        graph = torch.cuda.CUDAGraph()
        graph.capture_begin()
        static_out = self.model.infer(static_in)
        graph.capture_end()
      torch.cuda.current_stream(dev).wait_stream(side)
      ent = (graph, static_in, static_out)
      self._graphs[key] = ent
    graph, static_in, static_out = ent
    static_in.copy_(x, non_blocking=True)
    table = self.model.variables.weight_table
    if table is not None and table.dirty:
      table.refresh()            # variables changed since the capture (load_dict, init): the graph reads these planes
    graph.replay()
    return static_out.clone()                           # the static buffer is overwritten by the next replay

  def run(self, host_batches):
    from .prefetch import DevicePrefetcher
    if self.feed is None:
      self.feed = DevicePrefetcher(host_batches, self.model.device, self.depth)
    else:
      self.feed.restart(host_batches)
    for x in self.feed:
      y = self._infer(x)
      self.feed.release()
      yield self.back.put(y)
    self.back.synchronize()


def infer_batches(model: GanModel, host_batches, depth: int = 2):
  """One-shot form of InferencePipeline.run."""
  yield from InferencePipeline(model, depth).run(host_batches)


def make_dragan_rand(batch, hw, device, generator=None):
  """tf.random_uniform draws of image_generation.py:448,458 as explicit tensors."""
  r = {}
  for d in ('s', 't'):
    r['alpha_' + d] = torch.rand((batch, 1, 1, 1), device=device, generator=generator)
    r['noise_' + d] = torch.rand((batch, hw, hw, 3), device=device, generator=generator) * 2 - 1
  return r
