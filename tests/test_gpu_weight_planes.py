"""The split-bf16 weight operands every tensor-core conv of the step reads: the persistent WeightPlaneTable (one
k_split_weights_table launch per optimiser step) against twg_split_weights and a torch restatement, and the graphed
inference pipeline seeing a weight reload."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = 'cuda:0'


def _torch_planes(w, dgrad):
  """HWIO -> [tap][co][ci] (forward operand) or [flip(tap)][ci][co] (dgrad operand); hi = bf16_rn(w), lo = bf16_rn(w - hi)."""
  k, _, ci, co = w.shape
  t = w.reshape(k * k, ci, co)
  t = t.flip(0) if dgrad else t.permute(0, 2, 1)
  t = t.contiguous().reshape(-1)
  hi = t.to(torch.bfloat16)
  lo = (t - hi.float()).to(torch.bfloat16)
  return torch.stack([hi, lo])


def test_weight_plane_table_equals_split_weights_bit_for_bit(built_lib):
  from twingan_b200 import ops, twingan
  model = twingan.GanModel(twingan.Flags(train_image_size=256), device=DEV, seed=1234)
  v = model.variables
  table = v.weight_table
  table.dirty = True
  table.refresh()
  checked = 0
  for name, w in v.vars.items():
    for dgrad in (False, True):
      if (w.data_ptr(), dgrad) not in table.index:
        continue
      got = table.get(w.data_ptr(), dgrad)
      k, _, ci, co = w.shape
      direct = torch.empty_like(got)
      built_lib.call('twg_split_weights', w.data_ptr(), direct.data_ptr(), k, ci, co, int(dgrad), ops._st())
      want = _torch_planes(w.detach(), dgrad)
      assert torch.equal(got.view(torch.int16), direct.view(torch.int16)), (name, dgrad)
      assert torch.equal(got.view(torch.int16), want.view(torch.int16)), (name, dgrad)
      checked += 1
  # every 3x3 / 1x1 weight with tensor-core channel counts, in both layouts
  eligible = [n for n, w in v.vars.items() if n.endswith('/weights') and w.dim() == 4 and w.shape[0] in (1, 3)
              and all(ops._tc_channels_ok(int(c)) for c in w.shape[2:])]
  assert checked == 2 * len(eligible) and checked >= 40, (checked, len(eligible))


def test_graphed_inference_sees_reloaded_weights(built_lib):
  """InferencePipeline(use_graph=True): run, load other weights with load_dict, run again -- the replay must translate
  with the new weights (its tensor-core convs read the weight-plane table, which the reload marks stale)."""
  from twingan_b200 import ops, twingan
  ops.set_precision(1)
  model = twingan.GanModel(twingan.Flags(train_image_size=32, pggan_max_num_channels=32), device=DEV)
  g = torch.Generator().manual_seed(17)
  host = [torch.rand((3, 32, 32, 3), generator=g).pin_memory() for _ in range(2)]
  pipe = twingan.InferencePipeline(model, use_graph=True)

  def run():
    outs = []
    for out, ev in pipe.run(iter(host)):
      ev.synchronize()
      outs.append(out.clone())
    return outs

  first = run()
  params = model.variables.to_dict()
  gw = torch.Generator(device=DEV).manual_seed(23)
  new = {n: t * 1.5 + 0.02 * torch.randn(t.shape, device=DEV, generator=gw) if n.endswith('/weights') else t
         for n, t in params.items()}
  model.variables.load_dict(new)
  second = run()
  want = [model.infer(h.cuda()).cpu() for h in host]
  again = [model.infer(h.cuda()).cpu() for h in host]
  # run-to-run noise of the eager call (fp32 atomics order in split-K convs, amplified by the normalisers)
  noise = max(float((a - b).abs().max()) for a, b in zip(want, again))
  tol = 4.0 * noise + 1e-6 * max(float(b.abs().max()) for b in want)
  for i, (a, b) in enumerate(zip(second, want)):
    assert float((a - b).abs().max()) <= tol, (i, float((a - b).abs().max()), noise)
  # and the reload did change the translation
  assert max(float((a - b).abs().max()) for a, b in zip(first, second)) > 1e-2
