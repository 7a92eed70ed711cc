"""GPU: one training step of the BASELINE.json configs C3 (DIN), C4 (DSSM) and C5 (MMoE over a DCN backbone) at config
shape, built from their pipeline-config text through EasyRecEstimator, against a float64 restatement.

Each workload goes through one harness:
  1. architecture: the trainable parameter shapes equal the layer list the (strictly parsed) config declares;
  2. integer stage: the rows of K1 are bit-exact with the oracle's hashing (padded history positions -> -1);
  3. forward: the pooled lookup outputs within 1e-6 of the oracle's gather; logits and loss within 1e-4 of a
     float64 torch restatement evaluated on the device's pooled inputs and weights, with the ReLU decisions of the
     device run (a pre-activation within fp32 noise of zero would otherwise flip a mask, and the batch-norm chain
     turns one flip into an O(1/B) change of every gradient - see tools/fp32_order_sensitivity.py);
  4. backward: every dense gradient and the gradient of every looked-up output matrix no worse than an fp32 torch run
     of the same restatement by a bounded factor (the rule of test_gpu_dense.py; see no_worse), at p99.9 and at the
     maximum;
  5. update: a second estimator with the same seed starts from identical weights and takes one Trainer step; touched
     table rows and Adagrad accumulators against the oracle's row update fed with the float64 gradients, untouched
     rows bit-identical, dense parameters against Adagrad (acc0 0.1) on the float64 gradients plus l2 * w on kernels.

Only hash-bucket counts are scaled down (C4: item 2M / user 1M rows, C5: a 2M-row shared table); batch, widths,
towers, slots and sequence length are the configs'.
"""
import collections

import numpy as np
import pytest
import torch
from google.protobuf import text_format

from easyrec_b200 import backbone, layers as L, workloads
from easyrec_b200.config import proto_loader
from easyrec_b200.estimator import EasyRecEstimator
from oracle import oracle as O

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
SEED = 7
F64, F32 = torch.float64, torch.float32


# ---- the config as declared ------------------------------------------------------------------------------------------
def _strict(text):
  cfg = proto_loader.default_schema().EasyRecConfig()
  text_format.Merge(text, cfg, allow_unknown_field=False)
  return cfg


def _width(cfg, names):
  dims = {f.input_names[0]: f.embedding_dim for f in cfg.feature_config.features}
  return sum(dims[n] for n in names)


def _group(cfg, name):
  return [g for g in cfg.model_config.feature_groups if g.group_name == name][0].feature_names


def _dnn_shapes(n_in, units, use_bn=True, last_no_bn=False):
  out = []
  for k, u in enumerate(units):
    out += [(n_in, u), (u,)]
    if use_bn and not (last_no_bn and k + 1 == len(units)):
      out += [(u,), (u,)]
    n_in = u
  return out, n_in


def _mlp_shapes(n_in, mlp):
  """backbone MLP message: bias / batch norm per use_bias / use_bn, the last layer per use_final_*"""
  out, units = [], list(mlp.hidden_units)
  for k, u in enumerate(units):
    last = k + 1 == len(units)
    out.append((n_in, u))
    if mlp.use_final_bias if last else mlp.use_bias:
      out.append((u,))
    if mlp.use_final_bn if last else mlp.use_bn:
      out += [(u,), (u,)]
    n_in = u
  return out, n_in


def expected_shapes_c3(cfg):
  mt, out, total = cfg.model_config.multi_tower, [], 0
  for t in mt.towers:
    w = _width(cfg, _group(cfg, t.input))
    s, d = _dnn_shapes(w, t.dnn.hidden_units, t.dnn.use_bn)
    out += [(w,), (w,)] + s          # the tower's batch norm, then its DNN
    total += d
  for t in mt.din_towers:
    sg = [g for g in cfg.model_config.seq_att_groups if g.group_name == t.input][0]
    dh = _width(cfg, [m.hist_seq[0] for m in sg.seq_att_map])
    s, _ = _dnn_shapes(4 * dh, t.dnn.hidden_units, t.dnn.use_bn, last_no_bn=True)
    out += s
    total += 2 * dh                  # attended history + key
  s, d = _dnn_shapes(total, mt.final_dnn.hidden_units, mt.final_dnn.use_bn)
  return out + s + [(d, 1), (1,)]


def expected_shapes_c4(cfg):
  c, out = cfg.model_config.dssm, []
  for tower, group in ((c.user_tower, 'user'), (c.item_tower, 'item')):
    units = list(tower.dnn.hidden_units)
    s, d = _dnn_shapes(_width(cfg, _group(cfg, group)), units[:-1], tower.dnn.use_bn)
    out += s + [(d, units[-1]), (units[-1],)]
  return out + ([(1,), (1,)] if c.scale_simi else [])


def expected_shapes_c5(cfg):
  mc, out = cfg.model_config, []
  blocks = {b.name: b for b in mc.backbone.blocks}
  w = _width(cfg, _group(cfg, blocks['deep'].inputs[0].feature_group_name))
  s, d_deep = _mlp_shapes(w, blocks['deep'].keras_layer.mlp)
  out += s
  assert blocks['cross'].recurrent.keras_layer.class_name == 'Cross'
  out += [(w, w), (w,)] * blocks['cross'].recurrent.num_steps
  both = d_deep + w
  mm = blocks['mmoe'].keras_layer.mmoe
  for _ in range(mm.num_expert):
    s, d_exp = _mlp_shapes(both, mm.expert_mlp)
    out += s
  out += [(both, mm.num_expert), (mm.num_expert,)] * mm.num_task
  for t in mc.model_params.task_towers:
    s, d = _dnn_shapes(d_exp, t.dnn.hidden_units, t.dnn.use_bn)
    out += s + [(d, 1), (1,)]
  return out


def _assert_architecture(model, expected):
  got = collections.Counter(tuple(p.shape) for p in model.parameters() if p.requires_grad)
  want = collections.Counter(expected)
  assert got == want, 'trainable parameter shapes differ from the config: missing %s, unexpected %s' % (
      dict(want - got), dict(got - want))


# ---- device run ------------------------------------------------------------------------------------------------------
def _to_dev(x):
  if isinstance(x, dict):
    return {k: _to_dev(v) for k, v in x.items()}
  if isinstance(x, (tuple, list)):
    return tuple(_to_dev(v) for v in x)
  return x.to(DEV)


def _leaves(il):
  """{(dim, output key): the looked-up output matrix} of the last lookup - the autograd leaves whose .grad the row
  update reads - and per arena (arena, rows, merged call, output key of every merged output buffer)"""
  leaves, arenas = {}, []
  for m, rows, _, outs, _ in il._pending:
    dim = m.arena.dim
    subs = list(il.subcalls[dim])
    keys = []
    for k, (si, b) in enumerate(m.buf_of):
      keys.append([kk for (d, kk), (sk, j) in il.out_index.items() if d == dim and sk == subs[si] and j == b][0])
      leaves[(dim, keys[-1])] = outs[k]
    arenas.append((m.arena, rows, m, keys))
  return leaves, arenas


def _device_step(est, feats, labels):
  """forward with the ReLU decisions recorded, loss, backward - outside the Trainer, nothing is updated"""
  model = est.model
  model.train()
  masks = {}
  hooks = [m.register_forward_hook(lambda mod, i, o: masks.__setitem__(mod, (o > 0).detach()))
           for m in model.modules() if isinstance(m, L.DenseLayer) and m.relu]
  logits = model(feats)
  for h in hooks:
    h.remove()
  for m in model.modules():
    if isinstance(m, (L.DNN, backbone.MLP)):
      assert all(isinstance(a, torch.nn.Identity) for a in list(m.acts) + list(m.dropouts))
  leaves, arenas = _leaves(est.input_layer)
  loss, _ = model.loss(logits, labels)
  loss.backward()
  torch.cuda.synchronize()
  grads = {n: (p.grad if p.grad is not None else torch.zeros_like(p)).detach().clone()
           for n, p in model.named_parameters() if p.requires_grad}
  return dict(logits=logits.detach(), loss=float(loss.detach()), masks=masks, leaves=leaves, arenas=arenas, grads=grads)


# ---- restatements (plain torch, any dtype) ---------------------------------------------------------------------------
def _bn(z):
  mu = z.mean(0)
  return (z - mu) / torch.sqrt(((z - mu)**2).mean(0) + L.BN_EPS)


def _stack(x, mod, P, masks):
  """DNN / backbone MLP: dense -> batch norm (batch statistics) -> ReLU by the device's decision"""
  for lay in mod.layers:
    z = x @ P[lay.kernel] + P[lay.bias]
    if lay.use_bn:
      z = _bn(z) * P[lay.gamma] + P[lay.beta]
    x = z * masks[lay].to(z.dtype) if lay.relu else z
  return x


def _dense(x, lay, P):
  return x @ P[lay.kernel] + P[lay.bias]


def _ce(logits, labels):
  return torch.nn.functional.binary_cross_entropy_with_logits(logits, labels.to(logits.dtype))


def _sq(xs):
  return sum((x * x).sum() for x in xs)


def restate_c3(cfg, model, P, X, masks, batch):
  lens, labels = batch['lens'], batch['labels']
  B, T = lens.shape[0], batch['T']
  feas = []
  for g, bn, dnn in zip(model.tower_groups, model.tower_bn, model.tower_dnn):
    feas.append(_stack(_bn(X[(16, g)]) * P[bn.gamma] + P[bn.beta], dnn, P, masks))
  key = X[(16, 'din/key')]
  hist = X[(16, 'din/hist')].reshape(B, T, -1)
  q = key[:, None, :].expand_as(hist)
  # attention MLP over all B*T rows (its batch norm sees the padded ones too), last layer linear
  s = _stack(torch.cat([q, hist, q - hist, q * hist], -1).reshape(B * T, -1), model.din_dnn[0], P, masks).reshape(B, T)
  valid = torch.arange(T, device=DEV)[None, :] < lens[:, None]
  s = torch.where(valid, s, torch.full_like(s, -2.0**32 + 1))      # len 0: uniform over the (zero) history
  att = (torch.softmax(s, 1)[:, :, None] * hist).sum(1)
  feas.append(torch.cat([att, key], 1))
  logits = _dense(_stack(torch.cat(feas, 1), model.final_dnn, P, masks), model.output, P)[:, 0]
  reg = cfg.model_config.embedding_regularization * 0.5 * _sq([X[(16, 'user')], X[(16, 'item')], key, hist])
  return logits, _ce(logits, labels) + reg


def restate_c4(cfg, model, P, X, masks, batch):
  c = cfg.model_config.dssm
  xu, xi = X[(16, 'user')], X[(16, 'item')]
  u = _dense(_stack(xu, model.user_dnn, P, masks), model.user_out, P)
  i = _dense(_stack(xi, model.item_dnn, P, masks), model.item_out, P)
  u = u / torch.sqrt(torch.clamp((u * u).sum(1, keepdim=True), min=1e-12))
  i = i / torch.sqrt(torch.clamp((i * i).sum(1, keepdim=True), min=1e-12))
  sim = (u @ i.t()) / c.temperature * P[model.sim_w].abs() + P[model.sim_b]
  ids = batch['item_ids']
  dup = ids[None, :] == ids[:, None]
  dup.fill_diagonal_(False)                                       # in-batch duplicates of the positive, not itself
  masked = torch.where(dup, sim - 1e32, sim)
  p_diag = torch.softmax(masked, 1).diagonal()
  ce = -torch.log(p_diag + 1e-12).mean()
  reg_pos = torch.relu(-(u * i).sum(1)).mean()
  return sim, ce + reg_pos + cfg.model_config.embedding_regularization * 0.5 * _sq([xu, xi])


def restate_c5(cfg, model, P, X, masks, batch):
  mods = model.backbone.mods
  x0 = X[(32, 'all')]
  deep = _stack(x0, mods['deep'], P, masks)
  x = x0
  k = 0
  while 'cross_%d' % k in mods:                                   # DCN-v2 full rank: x0 * (x W + b) + x
    x = x0 * _dense(x, mods['cross_%d' % k].dense, P) + x
    k += 1
  both = torch.cat([deep, x], 1)
  mm = mods['mmoe']
  ex = torch.stack([_stack(both, e, P, masks) for e in mm.experts], 1)
  tasks = [(torch.softmax(_dense(both, g, P), 1)[:, :, None] * ex).sum(1) for g in mm.gates]
  logits = torch.stack([_dense(_stack(t, d, P, masks), o, P)[:, 0]
                        for t, d, o in zip(tasks, model.tower_dnn, model.tower_out)], 1)
  labels = batch['labels']
  loss = sum(t.weight * _ce(logits[:, j], labels[:, j]) for j, t in enumerate(cfg.model_config.model_params.task_towers))
  return logits, loss + cfg.model_config.embedding_regularization * 0.5 * _sq([x0])


def _reference(restate, cfg, model, run, batch, dt):
  class Params(dict):
    def __getitem__(self, p):
      return dict.__getitem__(self, id(p))
  P = Params()
  for p in model.parameters():
    P[id(p)] = p.detach().to(dt).clone().requires_grad_(p.requires_grad)
  X = {k: v.detach().to(dt).clone().requires_grad_(True) for k, v in run['leaves'].items()}
  logits, loss = restate(cfg, model, P, X, run['masks'], batch)
  loss.backward()
  grads = {n: (P[p].grad if P[p].grad is not None else torch.zeros_like(P[p])) for n, p in model.named_parameters()
           if p.requires_grad}
  return dict(logits=logits.detach(), loss=float(loss.detach()), grads=grads, leaf_grads={k: v.grad for k, v in X.items()})


def no_worse(mine, t32, t64, what, factor=64.0):
  """the device's error against float64 may exceed that of an fp32 torch evaluation by a bounded factor only, at the
  99.9th percentile and at the maximum (test_gpu_dense.py's rule).  That test allows 4x on one DNN with well-spread
  upstream gradients; here the gradients come through the whole model, every GEMM on the device is 3xTF32 (operands
  split into two TF32 halves, about 2^-21 per product against fp32's 2^-24), and reductions over the batch that cancel
  (batch-norm parameters, the 1280 x 1280 Cross kernels, the DSSM towers behind l2_normalize) magnify that difference.
  Measured on a B200: up to 31x the fp32 torch error (C4 item tower, C5 Cross kernels), at most 2e-4 of the gradient's
  mean magnitude.  Returns a description of the violation, or None."""
  em, et = (mine.double() - t64).abs().flatten(), (t32.double() - t64).abs().flatten()
  qm = float(torch.quantile(em[:4000000], 0.999)) if em.numel() > 1000 else float(em.max())
  qt = float(torch.quantile(et[:4000000], 0.999)) if et.numel() > 1000 else float(et.max())
  scale = float(t64.abs().mean())
  print('%-50s p99.9 %.3g / fp32 %.3g   max %.3g / fp32 %.3g   (scale %.3g)' % (
      what, qm, qt, float(em.max()), float(et.max()), scale))
  if qm > factor * qt + 2e-6 * scale:
    return '%s: p99.9 error %.3g vs torch fp32 %.3g (scale %.3g)' % (what, qm, qt, scale)
  if float(em.max()) > factor * float(et.max()) + 1e-5 * scale:
    return '%s: max error %.3g vs torch fp32 %.3g (scale %.3g)' % (what, float(em.max()), float(et.max()), scale)
  return None


# ---- the harness -----------------------------------------------------------------------------------------------------
def _segments(bufs, blocks, dim):
  """per-segment [n_seg, dim] rows of the output matrices, slot after slot (the oracle's gather / update layout)"""
  return torch.cat([bufs[b][:n, c:c + dim] for n, b, c in blocks], 0)


def _row_stats(got, want, what):
  d = np.abs(got - want)
  assert np.median(d) < 1e-6, '%s: median row error %.3g' % (what, np.median(d))
  assert (d > 1e-5).mean() < 0.02, '%s: %.3g of the elements off by > 1e-5' % (what, (d > 1e-5).mean())
  assert d.max() < 5e-3, '%s: max row error %.3g' % (what, d.max())


def run_parity(text, restate, expected_shapes, l2_section, feats, labels, batch, oracle_rows, est_kw=None):
  """oracle_rows(input layer) -> ({dim: rows}, {dim: weights}): the oracle's rows and weights of every lookup of each
  arena, slot after slot (the table offsets are the input layer's).  Returns (the stepped estimator, initial tables)."""
  torch.backends.cuda.matmul.allow_tf32 = False
  cfg = _strict(text)
  est = EasyRecEstimator(text, device=DEV, seed=SEED, **(est_kw or {}))
  model, il = est.model, est.input_layer
  _assert_architecture(model, expected_shapes(cfg))
  want_rows, want_w = oracle_rows(il)
  w0 = {n: p.detach().clone() for n, p in model.named_parameters()}
  tables0 = {d: (a.weight.detach().clone(), a.state0.detach().clone()) for d, a in il.arenas.items()}
  run = _device_step(est, feats, labels)

  # integer stage and pooled outputs
  plan = {}
  for arena, rows, m, keys in run['arenas']:
    d = arena.dim
    got = rows.cpu().numpy()
    assert np.array_equal(got, want_rows[d]), 'dim %d: %d of %d rows differ from the oracle' % (
        d, int((got != want_rows[d]).sum()), got.size)
    uniq = np.unique(got[got >= 0])
    rows_c = np.where(got >= 0, np.searchsorted(uniq, got), -1)
    idx = torch.from_numpy(uniq).to(DEV)
    want, _ = O.embedding_fwd(arena.weight[idx].cpu().numpy(), rows_c, np.arange(got.size + 1, dtype=np.int32), 0,
                              weights=want_w[d])
    blocks = [(int(r['n_seg']), int(r['out_buf']), int(r['out_col'])) for r in m.slots_np]
    got_pooled = _segments([run['leaves'][(d, k)].detach() for k in keys], blocks, d).cpu().numpy()
    err = np.abs(got_pooled - want).max()
    assert err <= 1e-6, 'dim %d: pooled outputs off the oracle gather by %.3g' % (d, err)
    plan[d] = (rows_c, idx, keys, blocks)

  # forward and backward against float64 (and the fp32 torch baseline of the backward rule)
  r64 = _reference(restate, cfg, model, run, batch, F64)
  r32 = _reference(restate, cfg, model, run, batch, F32)
  lerr = float((run['logits'].double() - r64['logits']).abs().max())
  assert lerr < 1e-4, 'logits off float64 by %.3g (fp32 torch: %.3g)' % (
      lerr, float((r32['logits'].double() - r64['logits']).abs().max()))
  assert abs(run['loss'] - r64['loss']) < 1e-4, 'loss %.7f vs float64 %.7f' % (run['loss'], r64['loss'])
  problems = []   # (gradient checks are reported together, after the update stage)
  for n, g in run['grads'].items():
    if float(r64['grads'][n].abs().max()) < 1e-14:
      # zero by construction - biases under batch norm, the beta of a batch norm feeding one, the bias of the DIN score
      # and of the DSSM similarity (softmax is shift invariant): rounding noise only, against the fp32 run's and the
      # layer's scale
      sib = [r64['grads'][n.rsplit('.', 1)[0] + x] for x in ('.kernel', '.gamma') if n.rsplit('.', 1)[0] + x in r64['grads']]
      noise = 10 * float(r32['grads'][n].abs().max()) + 1e-6 * max(float(t.abs().max()) for t in sib or r64['grads'].values())
      if float(g.abs().max()) > noise:
        problems.append('grad of %s: %.3g where float64 has 0 (allowed %.3g)' % (n, float(g.abs().max()), noise))
      continue
    problems.append(no_worse(g, r32['grads'][n], r64['grads'][n], 'grad of %s' % n))
  for k, leaf in run['leaves'].items():
    assert leaf.grad is not None, 'no gradient reached the looked-up output %s' % (k,)
    problems.append(no_worse(leaf.grad, r32['leaf_grads'][k], r64['leaf_grads'][k], 'grad of looked-up output %s' % (k,)))
  problems = [p for p in problems if p]

  # one Trainer step of a second, identically seeded estimator
  del run, est
  est2 = EasyRecEstimator(text, device=DEV, seed=SEED, **(est_kw or {}))
  for n, p in est2.model.named_parameters():
    assert torch.equal(p.detach(), w0[n]), 'initial %s differs between two estimators of one seed' % n
  for d, a in est2.input_layer.arenas.items():
    assert torch.equal(a.weight, tables0[d][0]) and torch.equal(a.state0, tables0[d][1]), 'initial table %d' % d
  lr = float(est2._opt['lr_fn'](0))
  loss, _ = est2.trainer.train_step(feats, labels)
  torch.cuda.synchronize()
  l2 = getattr(cfg.model_config, l2_section).l2_regularization
  kernels = sum(0.5 * l2 * float((w0[n].double()**2).sum()) for n in r64['grads'] if n.endswith('kernel'))
  assert abs(float(loss) - (r64['loss'] + kernels)) < 1e-4, 'step loss %.7f vs float64 %.7f' % (
      float(loss), r64['loss'] + kernels)
  for d, a in est2.input_layer.arenas.items():
    rows_c, idx, keys, blocks = plan[d]
    gseg = _segments([r64['leaf_grads'][(d, k)] for k in keys], blocks, d).float().cpu().numpy()
    t_c, s_c = tables0[d][0][idx].cpu().numpy(), tables0[d][1][idx].cpu().numpy()
    O.embedding_bwd(t_c, s_c, None, rows_c, None, gseg, O.OPT_ADAGRAD, lr, weights=want_w[d])
    _row_stats(a.weight[idx].cpu().numpy(), t_c, 'dim %d touched rows' % d)
    _row_stats(a.state0[idx].cpu().numpy(), s_c, 'dim %d adagrad accumulators' % d)
    keep = torch.ones(a.n_rows, dtype=torch.bool, device=DEV)
    keep[idx] = False
    assert torch.equal(a.weight[keep], tables0[d][0][keep]), 'dim %d: an untouched row moved' % d
    assert torch.equal(a.state0[keep], tables0[d][1][keep]), 'dim %d: an untouched accumulator moved' % d
  for n, p in est2.model.named_parameters():
    if not p.requires_grad:
      assert torch.equal(p.detach(), w0[n]), '%s is not trained but moved' % n
      continue
    w = w0[n].double()
    g = r64['grads'][n] + (l2 * w if n.endswith('kernel') else 0.0)
    want = w - lr * g / torch.sqrt(0.1 + g * g)
    err = float((p.detach().double() - want).abs().max())
    assert err < 2e-4, '%s after one step: off Adagrad on the float64 gradient by %.3g' % (n, err)
  assert not problems, 'gradients worse than an fp32 torch evaluation:\n' + '\n'.join(problems)
  return est2, tables0


def _hashed(ids, tables, name, nb):          # IdFeature with hash_bucket_size: Fingerprint64(decimal text) % nb
  return O.bucketize(np.ascontiguousarray(ids), 0, nb, tables[name][0])[0]


def _ident(ids, tables, name, nb):           # num_buckets, or a STRING field the reader already hashed
  return O.bucketize(np.ascontiguousarray(ids), 2, nb, tables[name][0])[0]


def _one_row(B, tables, name):               # RawFeature with an embedding: every sample reads row 0, weighted
  return O.bucketize(np.zeros(B, np.int64), 4, 1, tables[name][0])[0]


def test_c3_din_training_step_matches_float64():
  """C3 at config shape: batch 4096, two 50-step histories, 1M-row item tables, attention MLP [128, 64, 32, 1].
  Some histories are empty and some full; one row of the history table is named only at padded positions."""
  check_c3(4096, 50, 1_000_000)


def check_c3(B, T, V):
  f, labels = workloads.c3_batch(B, T, 11, V)
  lens = f['seq_fea']['hist_items'][1].numpy().copy()
  lens[:8], lens[8:16] = 0, T
  valid = np.arange(T)[None, :] < lens[:, None]
  hist_items = f['seq_fea']['hist_items'][0].numpy().copy()
  hist_cates = f['seq_fea']['hist_cates'][0].numpy()
  ghost = int(np.setdiff1d(np.arange(V), hist_items[valid])[0])
  hist_items[~valid] = ghost
  f['seq_fea'] = {'hist_items': (torch.from_numpy(hist_items), torch.from_numpy(lens)),
                  'hist_cates': (torch.from_numpy(hist_cates), torch.from_numpy(lens.copy()))}
  ids = f['sparse_fea'].numpy().reshape(4, B)
  price = f['dense_fea'].numpy()[:, 0]      # min 0, max 1: the normalised value is the value

  def oracle_rows(il):
    tb = il.arenas[16].tables
    single = [_hashed(ids[0], tb, 'user_id_embedding', 1000000), _ident(ids[1], tb, 'age_embedding', 100),
              _hashed(ids[2], tb, 'item_id_embedding', V), _hashed(ids[3], tb, 'cate_id_embedding', 10000),
              _one_row(B, tb, 'price_embedding'),
              _hashed(ids[2], tb, 'din/item_id_embedding', V), _hashed(ids[3], tb, 'din/cate_id_embedding', 10000)]
    seq = [_ident(hist_items.reshape(-1), tb, 'din/hist_items_embedding', V),
           _ident(hist_cates.reshape(-1), tb, 'din/hist_cates_embedding', 10000)]
    for r in seq:
      r[~valid.reshape(-1)] = -1             # positions t >= len look nothing up
    w = np.ones(7 * B + 2 * B * T, np.float32)
    w[4 * B:5 * B] = price
    return {16: np.concatenate(single + seq)}, {16: w}

  feats = _to_dev(f)
  batch = {'lens': feats['seq_fea']['hist_items'][1].long(), 'T': T, 'labels': labels.to(DEV)}
  est, tables0 = run_parity(workloads.c3_config_text(B, V, T), restate_c3, expected_shapes_c3, 'multi_tower', feats,
                            labels.to(DEV), batch, oracle_rows, est_kw=dict(default_seq_len=T))
  a = est.input_layer.arenas[16]
  row = a.tables['din/hist_items_embedding'][0] + ghost
  assert torch.equal(a.weight[row], tables0[16][0][row]) and torch.equal(a.state0[row], tables0[16][1][row]), \
      'a history row named only at padded positions was updated'


def test_c4_dssm_training_step_matches_float64():
  """C4 at config shape: batch 4096, towers [256, 128, 64] + Dense(32), cosine / temperature 0.05 / |sim_w|, in-batch
  softmax with duplicate items masked (item table 2M rows, user table 1M rows)."""
  check_c4(4096, 2_000_000, 1_000_000)


def check_c4(B, item_vocab, user_vocab):
  f, labels = workloads.c4_batch(B, 13)
  item = f['item_ids'].numpy()
  assert B - np.unique(item).size > B // 40, 'the batch must repeat item ids to test the duplicate mask'
  ids = f['sparse_fea'].numpy().reshape(8, B)
  price = f['dense_fea'].numpy()[:, 0]

  def oracle_rows(il):
    tb = il.arenas[16].tables
    rows = [_hashed(ids[0], tb, 'user_id_embedding', user_vocab), _ident(ids[1], tb, 'age_embedding', 100),
            _ident(ids[2], tb, 'gender_embedding', 3), _hashed(ids[3], tb, 'city_embedding', 10000),
            _ident(ids[4], tb, 'level_embedding', 10), _hashed(ids[5], tb, 'item_id_embedding', item_vocab),
            _hashed(ids[6], tb, 'cate_id_embedding', 10000), _hashed(ids[7], tb, 'brand_embedding', 1_000_000),
            _one_row(B, tb, 'price_embedding')]
    w = np.ones(9 * B, np.float32)
    w[8 * B:] = price
    return {16: np.concatenate(rows)}, {16: w}

  feats = _to_dev(f)
  text = workloads.c4_config_text(B, item_vocab=item_vocab, user_vocab=user_vocab, embedding_parallel=False)
  run_parity(text, restate_c4, expected_shapes_c4, 'dssm', feats, labels.to(DEV), {'item_ids': feats['item_ids']},
             oracle_rows)


def test_c5_mmoe_over_dcn_training_step_matches_float64():
  """C5 at config shape: batch 16384, 40 id slots x dim 32 over one shared table (2M rows), MLP [256, 128] beside three
  full-rank Cross layers, MMoE with 4 experts [128, 64] and 3 gates, three task towers dnn [64] + Dense(1)."""
  check_c5(16384, 2_000_000, 40)


def check_c5(B, V, n_feat):
  f, labels = workloads.c5_batch(B, 17, n_feat=n_feat)
  ids = f['sparse_fea'].numpy()

  def oracle_rows(il):
    return {32: _hashed(ids, il.arenas[32].tables, 'shared', V)}, {32: np.ones(ids.size, np.float32)}

  feats = _to_dev(f)
  text = workloads.c5_config_text(B, vocab=V, n_feat=n_feat, embedding_parallel=False)
  run_parity(text, restate_c5, expected_shapes_c5, 'model_params', feats, labels.to(DEV), {'labels': labels.to(DEV)},
             oracle_rows)
