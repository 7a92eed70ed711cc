"""CPU (kernel doubles, tests/host_doubles.py): the host-side behaviour added after the first review.

  * two hist_seq features of one DIN group own separate columns of the sequence matrix (forward and backward);
  * `adam_optimizer` = tf.train.AdamOptimizer: rows without a gradient decay as well (builders/optimizer_builder.py:61-66,
    behaviour stated at compat/adam_s.py:74-81), against the oracle restatement step by step;
  * multi-task towers read the label their `label_name` names (model/multi_task_model.py:114-122);
  * a resumed run (save -> restore) continues exactly like an uninterrupted one: dense optimizer slots, the
    learning-rate clock and Adam's beta powers are part of the checkpoint;
  * embedding_learning_rate_multiplier multiplies the table gradients (model/easy_rec_estimator.py:308-317);
  * the optimizer step scalars of the device block (what a captured CUDA graph reads) equal the struct's.
"""
import numpy as np
import pytest
import torch

from easyrec_b200 import _lib, builder, kernels as K, trainer as T
from easyrec_b200.config import config_util
from easyrec_b200.input import readers
from oracle import oracle as O
import host_doubles
from test_input_layer_host import oracle_kernels  # noqa: F401  (fixture)
from test_model_host import dense_kernels, interaction_doubles  # noqa: F401  (fixtures)

DIN2 = b'''
train_config { optimizer_config { adagrad_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.05 } } } } }
data_config { batch_size: 4 input_type: CSVInput separator: "," label_fields: "clk"
  input_fields { input_name: "clk" input_type: FLOAT } input_fields { input_name: "item_id" input_type: INT64 }
  input_fields { input_name: "cate_id" input_type: INT64 }
  input_fields { input_name: "hist" input_type: STRING } input_fields { input_name: "hist_c" input_type: STRING } }
feature_config {
  features { input_names: "item_id" feature_type: IdFeature embedding_dim: 8 num_buckets: 40 }
  features { input_names: "cate_id" feature_type: IdFeature embedding_dim: 8 num_buckets: 12 }
  features { input_names: "hist" feature_type: SequenceFeature embedding_dim: 8 num_buckets: 40 max_seq_len: 3 separator: "|" }
  features { input_names: "hist_c" feature_type: SequenceFeature embedding_dim: 8 num_buckets: 12 max_seq_len: 3 separator: "|" } }
model_config { model_class: "MultiTowerDIN"
  feature_groups { group_name: "item" feature_names: ["item_id", "cate_id"] wide_deep: DEEP }
  seq_att_groups { group_name: "din" seq_att_map { key: "item_id" hist_seq: "hist" } seq_att_map { key: "cate_id" hist_seq: "hist_c" } }
  multi_tower { towers { input: "item" dnn { hidden_units: [8] } }
                din_towers { input: "din" dnn { hidden_units: [8, 1] } } final_dnn { hidden_units: [8] } } }
'''


def test_two_hist_seq_features_of_one_group_keep_their_own_columns(tmp_path, interaction_doubles):  # noqa: F811
  """din_on_taobao.config's shape (tag_brand_list + tag_category_list in group 'din'): each history feature is looked
  up in its own table and lands in its own half of hist_seq_emb; the backward routes each half to its own table."""
  cfg = config_util.get_configs_from_pipeline_file(DIN2)
  il, model, opt = builder.build_model(cfg, 4, 'cpu', cpu_generator=torch.Generator().manual_seed(2))
  rows = ['1,5,1,7|8|9,2|3|4', '0,6,2,10,5', '1,7,3,,', '0,8,4,11|12,6|7']
  open(tmp_path / 's.csv', 'w').write('\n'.join(rows) + '\n')
  (feats, labels), = list(readers.make_input(cfg, il, str(tmp_path / 's.csv')))
  il.lookup(feats)
  so = il.seq_outputs['din']
  emb = so['hist_seq_emb'].detach().numpy()
  assert emb.shape == (4, 3, 16)
  a = il.arenas[8]
  tab = a.weight.numpy()

  def table(name):
    off, local, _ = a.tables[name]
    return tab[off:off + local]
  t_hist, t_cate = table('din/hist_embedding'), table('din/hist_c_embedding')
  want = np.zeros((4, 3, 16), np.float32)
  for b, (h, c) in enumerate([([7, 8, 9], [2, 3, 4]), ([10], [5]), ([], []), ([11, 12], [6, 7])]):
    for t, i in enumerate(h):
      want[b, t, :8] = t_hist[i]
    for t, i in enumerate(c):
      want[b, t, 8:] = t_cate[i]
  np.testing.assert_array_equal(emb, want)
  assert not np.array_equal(emb[0, :, :8], emb[0, :, 8:])          # the two halves are different tables
  key = so['key'].detach().numpy()
  np.testing.assert_array_equal(key[:, :8], table('din/item_id_embedding')[[5, 6, 7, 8]])
  np.testing.assert_array_equal(key[:, 8:], table('din/cate_id_embedding')[[1, 2, 3, 4]])
  # ---- backward: a gradient on the second half only moves rows of the second history table ----
  before = tab.copy()
  g = torch.zeros_like(so['hist_seq_emb'])
  g[:, :, 8:] = 1.0
  so['hist_seq_emb'].backward(g)
  il.set_optimizer_step(0.05, 0)
  il.backward_update()
  moved = np.flatnonzero((a.weight.numpy() != before).any(1))
  off_c, _, _ = a.tables['din/hist_c_embedding']
  assert sorted(moved.tolist()) == sorted(off_c + i for i in (2, 3, 4, 5, 6, 7))
  # ... and the whole model trains
  tr = T.Trainer(model, il, 'adagrad', lr_fn=opt['lr_fn'])
  losses = [float(tr.train_step(feats, labels)[0]) for _ in range(12)]
  assert all(np.isfinite(losses)) and losses[-1] < losses[0]


ADAM = b'''
train_config { optimizer_config { adam_optimizer { learning_rate { exponential_decay_learning_rate {
  initial_learning_rate: 0.01 decay_steps: 2 decay_factor: 0.5 min_learning_rate: 0.0001 } } }
  embedding_learning_rate_multiplier: 2.0 } }
data_config { batch_size: 8 input_type: CSVInput separator: "," label_fields: "label"
  input_fields { input_name: "label" input_type: FLOAT } input_fields { input_name: "c" input_type: INT64 }
  input_fields { input_name: "d" input_type: INT64 } }
feature_config {
  features { input_names: "c" feature_type: IdFeature embedding_dim: 4 num_buckets: 30 }
  features { input_names: "d" feature_type: IdFeature embedding_dim: 4 num_buckets: 10 } }
model_config { model_class: "DeepFM"
  feature_groups { group_name: "deep" feature_names: ["c", "d"] wide_deep: DEEP }
  feature_groups { group_name: "wide" feature_names: ["c", "d"] wide_deep: WIDE }
  deepfm { dnn { hidden_units: [8] } final_dnn { hidden_units: [4] } } }
'''


def test_adam_optimizer_decays_untouched_rows_like_tf_adam(dense_kernels):  # noqa: F811
  """Five steps of a DeepFM with `adam_optimizer`: after each step the deep arena equals the oracle's
  tf.train.AdamOptimizer sparse apply on the gradient the step produced - rows looked up in an EARLIER step keep
  moving (m, v decay, w -= lr_t*m/(sqrt(v)+eps)) although the current batch does not contain them."""
  from easyrec_b200.estimator import EasyRecEstimator
  est = EasyRecEstimator(ADAM, device='cpu', seed=1)
  il, tr = est.input_layer, est.trainer
  a = il.arenas[4]
  assert a.opt_kind == _lib.OPT_ADAM_ROWS and a.touched is not None and il.emb_grad_mult == 2.0
  rng = np.random.default_rng(0)
  w, m, v = (x.numpy().copy() for x in (a.weight, a.state0, a.state1))
  seen = set()
  for step in range(5):
    ids_c = rng.integers(0, 30, 8) if step < 2 else rng.integers(0, 5, 8)   # later batches miss most early rows
    ids_d = rng.integers(0, 10, 8)
    feats = {'sparse_fea': torch.from_numpy(np.concatenate([ids_c, ids_d]).astype(np.int64))}
    labels = torch.from_numpy((rng.uniform(size=8) < 0.5).astype(np.float32))
    # the gradient of this step's lookups, captured from the leaves K7 would read
    captured = {}
    real_bwd = K.embedding_bwd

    def spy(table, s0, s1, dim, rows, slots_dev, n_slots, n_seg, grad_bufs, opt, ws, **kw):
      if dim == 4:
        captured['rows'] = rows.numpy().copy()
        captured['g'] = grad_bufs[0].numpy().copy()
        captured['opt'] = (opt.lr, opt.beta1_power, opt.beta2_power, opt.grad_scale)
      return real_bwd(table, s0, s1, dim, rows, slots_dev, n_slots, n_seg, grad_bufs, opt, ws, **kw)
    K.embedding_bwd = spy
    try:
      tr.train_step(feats, labels)
    finally:
      K.embedding_bwd = real_bwd
    lr, b1p, b2p, gs = captured['opt']
    t = step + 1
    assert lr == pytest.approx(est._opt['lr_fn'](step)) and gs == 2.0
    assert b1p == pytest.approx(0.9**t, rel=1e-6) and b2p == pytest.approx(0.999**t, rel=1e-6)
    g = captured['g'][:, :8].reshape(8, 2, 4).transpose(1, 0, 2).reshape(16, 4)   # per-lookup rows, feature-major
    O.embedding_bwd_adam_dense(w, m, v, captured['rows'], None, g, lr, beta1_power=b1p, beta2_power=b2p, grad_scale=gs)
    np.testing.assert_array_equal(a.weight.numpy(), w)
    np.testing.assert_array_equal(a.state0.numpy(), m)
    np.testing.assert_array_equal(a.state1.numpy(), v)
    if step >= 2:   # rows of the first batches that this batch does not touch still moved
      cold = sorted(seen - set(captured['rows'].tolist()))
      assert cold and (np.abs(m[cold]).sum() > 0)
    seen |= set(captured['rows'].tolist())
    assert not a.touched.any()                      # the mask is left clean for the next step
  # the struct and the device block carry the same scalars
  o = il.opt_holder['opt']
  dev = il.hyper.dev.numpy()
  assert (o.lr, o.beta1_power, o.beta2_power, o.grad_scale) == tuple(float(x) for x in dev)
  assert o.hyper_dev == il.hyper.dev.data_ptr()


def test_oracle_adam_dense_equals_dense_adam_with_zero_gradient_on_cold_rows():
  """compat/adam_s.py:74-81: "the sparse behavior is equivalent to the dense behavior".  The oracle's sparse apply on
  some rows == TensorFlow's dense ApplyAdam formula (adam_update_numpy of TF's adam_test.py) on a gradient that is
  zero on every other row."""
  rng = np.random.default_rng(3)
  V, D = 20, 4
  w = rng.normal(size=(V, D)).astype(np.float32)
  m = (rng.normal(size=(V, D)) * 0.1).astype(np.float32)
  v = (rng.uniform(size=(V, D)) * 0.01).astype(np.float32)
  m[15:] = 0
  v[15:] = 0
  rows = np.array([3, 7, 3, 11], np.int64)
  g = rng.normal(size=(4, D)).astype(np.float32)
  full = np.zeros((V, D), np.float32)
  for r, gr in zip(rows, g):
    full[r] = full[r] + gr
  f = np.float32
  b1, b2, eps, lr, t = f(0.9), f(0.999), f(1e-8), f(0.01), 4
  b1p, b2p = f(0.9)**t, f(0.999)**t
  lr_t = O.adam_lr_t(lr, b1p, b2p)
  m_t = (full * (f(1) - b1) + m * b1).astype(np.float32)
  v_t = ((full * full) * (f(1) - b2) + v * b2).astype(np.float32)
  w_t = w - (lr_t * m_t) / (np.sqrt(v_t) + eps)
  w2, m2, v2 = w.copy(), m.copy(), v.copy()
  O.embedding_bwd_adam_dense(w2, m2, v2, rows, None, g, float(lr), beta1_power=float(b1p), beta2_power=float(b2p))
  np.testing.assert_allclose(m2, m_t, rtol=0, atol=1e-9)
  np.testing.assert_allclose(v2, v_t, rtol=0, atol=1e-9)
  np.testing.assert_allclose(w2, w_t, rtol=0, atol=1e-7)
  np.testing.assert_array_equal(w2[15:], w[15:])         # never-touched rows (m = v = 0) do not move at all


MTL = b'''
train_config { optimizer_config { adagrad_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.1 } } } } }
data_config { batch_size: 16 input_type: CSVInput separator: "," label_fields: ["buy", "aux", "clk"]
  input_fields { input_name: "buy" input_type: FLOAT } input_fields { input_name: "aux" input_type: FLOAT }
  input_fields { input_name: "clk" input_type: FLOAT } input_fields { input_name: "c" input_type: INT64 } }
feature_config { features { input_names: "c" feature_type: IdFeature embedding_dim: 4 num_buckets: 16 } }
model_config { model_class: "MMoE"
  feature_groups { group_name: "all" feature_names: ["c"] wide_deep: DEEP }
  mmoe { experts { expert_name: "e0" dnn { hidden_units: [8] } } experts { expert_name: "e1" dnn { hidden_units: [8] } }
         task_towers { tower_name: "ctr" label_name: "clk" dnn { hidden_units: [4] } }
         task_towers { tower_name: "cvr" label_name: "buy" dnn { hidden_units: [4] } } } }
'''


def test_task_towers_train_on_the_label_their_label_name_names(interaction_doubles):  # noqa: F811
  """tower order (ctr, cvr) differs from label_fields order (buy, aux, clk): the towers must read columns 2 and 0."""
  cfg = config_util.get_configs_from_pipeline_file(MTL)
  il, model, opt = builder.build_model(cfg, 16, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  assert model.label_cols == [2, 0]
  ids = torch.arange(16, dtype=torch.int64)
  labels = torch.zeros(16, 3)
  labels[:, 2] = (ids % 2 == 0).float()      # clk: even ids
  labels[:, 0] = (ids < 4).float()           # buy: small ids
  labels[:, 1] = 1.0 - labels[:, 2]          # aux: the opposite of clk (a tower bound by position would learn this one)
  logits = torch.from_numpy(np.random.default_rng(1).normal(size=(16, 2)).astype(np.float32))
  model._emb_outputs = ()
  loss, probs = model.loss(logits, labels)
  want = (O.sigmoid_ce(logits[:, 0].numpy(), labels[:, 2].numpy())[0] +      # ctr tower <- clk
          O.sigmoid_ce(logits[:, 1].numpy(), labels[:, 0].numpy())[0])       # cvr tower <- buy
  by_position = (O.sigmoid_ce(logits[:, 0].numpy(), labels[:, 0].numpy())[0] +
                 O.sigmoid_ce(logits[:, 1].numpy(), labels[:, 1].numpy())[0])
  assert float(loss) == pytest.approx(want, rel=1e-6) and abs(want - by_position) > 1e-3
  bad = config_util.get_configs_from_pipeline_file(MTL.replace(b'label_name: "buy"', b'label_name: "nope"'))
  with pytest.raises(ValueError, match='label_name'):
    builder.build_model(bad, 16, 'cpu', cpu_generator=torch.Generator().manual_seed(0))


def test_resumed_run_equals_the_uninterrupted_one(tmp_path, dense_kernels):  # noqa: F811
  """train(2N) == train(N) + save + restore + train(N): tables, dense parameters, dense optimizer slots, the decayed
  learning rate and Adam's beta powers all continue where they stopped."""
  from easyrec_b200.estimator import EasyRecEstimator
  text = ADAM.replace(b'train_config {', b'model_dir: "%s" train_config {' % str(tmp_path / 'm').encode())
  rng = np.random.default_rng(5)
  batches = []
  for _ in range(6):
    ids = np.concatenate([rng.integers(0, 30, 8), rng.integers(0, 10, 8)]).astype(np.int64)
    batches.append(({'sparse_fea': torch.from_numpy(ids)}, torch.from_numpy((rng.uniform(size=8) < 0.5).astype(np.float32))))
  full = EasyRecEstimator(text, device='cpu', seed=7)
  full.train(lambda: iter(batches), steps=6)
  half = EasyRecEstimator(text, device='cpu', seed=7)
  half.train(lambda: iter(batches[:3]), steps=3)
  path = half.save()
  resumed = EasyRecEstimator(text, device='cpu', seed=123)      # other initial weights: everything comes from the file
  resumed.restore(path)
  assert resumed.trainer.step == 3 and resumed.global_step == 3
  resumed.train(lambda: iter(batches[3:]), steps=3)
  for d in full.input_layer.arenas:
    np.testing.assert_array_equal(resumed.input_layer.arenas[d].storage.numpy(), full.input_layer.arenas[d].storage.numpy())
  np.testing.assert_array_equal(resumed.trainer.dense_opt.flat_p.numpy(), full.trainer.dense_opt.flat_p.numpy())
  np.testing.assert_array_equal(resumed.trainer.dense_opt.s0.numpy(), full.trainer.dense_opt.s0.numpy())
  np.testing.assert_array_equal(resumed.trainer.dense_opt.s1.numpy(), full.trainer.dense_opt.s1.numpy())
  assert resumed.input_layer.opt_holder['opt'].beta1_power == full.input_layer.opt_holder['opt'].beta1_power


def test_beta_powers_are_fp32_products_like_the_tf_accumulators():
  """compat/adam_s.py:233-245 (_finish): beta1_power <- beta1_power * beta1 in fp32, once per step."""
  h = K.StepHyper('cpu', 0.9, 0.999)
  b1p, b2p = np.float32(0.9), np.float32(0.999)
  for step in range(50):
    h.set(0.001, step)
    assert h.b1p == b1p and h.b2p == b2p
    b1p, b2p = np.float32(b1p * np.float32(0.9)), np.float32(b2p * np.float32(0.999))
  h2 = K.StepHyper('cpu', 0.9, 0.999)
  h2.set(0.001, 37)                          # a restored run starts in the middle: same accumulators
  h.set(0.001, 37)
  assert (h2.b1p, h2.b2p) == (h.b1p, h.b2p)


def test_dnn_use_bn_false_builds_plain_dense_relu_towers(dense_kernels):  # noqa: F811
  """protos/dnn.proto `use_bn: false` (layers/dnn.py:62-70): dense + bias -> relu, no batch norm - per DNN message."""
  text = workloads_c2(dnn_extra='use_bn: false')
  cfg = config_util.get_configs_from_pipeline_file(text)
  import os
  os.environ['ER_PLAN_ONLY'] = '1'
  try:
    il, model, _ = builder.build_model(cfg, 32, 'cpu', cpu_generator=torch.Generator().manual_seed(1))
  finally:
    del os.environ['ER_PLAN_ONLY']
  assert [l.use_bn for l in model.dnn.layers] == [False, False] and all(l.use_bn for l in model.final_dnn.layers)
  assert not hasattr(model.dnn.layers[0], 'gamma') or model.dnn.layers[0].gamma is None
  x = torch.randn(32, model.dnn.layers[0].kernel.shape[0])
  want = x
  for l in model.dnn.layers:
    want = torch.relu(want @ l.kernel + l.bias)
  torch.testing.assert_close(model.dnn(x), want, rtol=1e-5, atol=1e-6)


def workloads_c2(dnn_extra=''):
  from easyrec_b200 import workloads
  text = workloads.c2_config_text(1000, 32, dnn=(16, 8), final=(8, 4)).decode()
  return text.replace('dnn { hidden_units: [16, 8]', 'dnn { %s hidden_units: [16, 8]' % dnn_extra, 1).encode()


def test_backbone_embedding_layer_block_is_one_offset_table_of_the_blocks_width(interaction_doubles):  # noqa: F811
  """§8 a23 (layers/input_layer.py:209-243 + layers/keras/embedding.py:26-81): ids bucketized per feature, offset by the
  vocabularies before them, ONE Embedding(sum vocab, block dim) with Keras' uniform(-0.05, 0.05) init, concat."""
  import test_gpu_models as G
  cfg = config_util.get_configs_from_pipeline_file(G.BACKBONE_EMBLAYER_CFG.encode())
  B = 256
  il, model, opt = builder.build_model(cfg, B, 'cpu', cpu_generator=torch.Generator().manual_seed(1), default_seq_len=20)
  a = il.arenas[12]                                   # the block's width, not the features' own embedding_dim 16
  names = ['emb/user_id_embedding', 'emb/age_embedding', 'emb/item_id_embedding', 'emb/cate_embedding']
  vocab = [1000, 10, 5000, 200]
  assert list(a.tables) == names
  off = 0
  for n, v in zip(names, vocab):                      # offset += vocab, in feature-group order
    assert a.tables[n] == (off, v, v)
    off += v
  W = a.weight.numpy()
  assert np.abs(W).max() <= 0.05 and 0.02 < W.std() < 0.035   # uniform(-0.05, 0.05): std 0.0289
  rng = np.random.default_rng(0)
  ids = np.stack([rng.integers(0, 10**6, B), rng.integers(0, 10, B), rng.integers(0, 10**6, B), rng.integers(0, 500, B)])
  feats = {'sparse_fea': torch.from_numpy(ids.reshape(-1).astype(np.int64)),
           'dense_fea': torch.from_numpy(rng.uniform(0, 100, (B, 1)).astype(np.float32))}
  g = il.lookup(feats)
  out = g['ids'][0].detach().numpy()
  assert out.shape == (B, 48)
  off = 0
  for j, v in enumerate(vocab):
    rows = O.bucketize(ids[j], 2 if j == 1 else 0, v, 0)[0]   # string_to_hash_bucket_fast(as_string(id), vocab) / as is
    np.testing.assert_array_equal(out[:, 12 * j:12 * (j + 1)], W[off + rows])
    off += v
  # the Keras table carries no embedding regulariser; the input_layer group does
  assert model.groups == ['dense']
  tr = T.Trainer(model, il, 'adagrad', lr_fn=opt['lr_fn'])
  lab = torch.from_numpy((rng.uniform(size=B) < 0.3).astype(np.float32))
  losses = [float(tr.train_step(feats, lab)[0]) for _ in range(12)]
  assert losses[-1] < losses[0] - 0.01


def test_dnn_dropout_ratio_masks_in_training_only_and_redraws_every_step(dense_kernels):  # noqa: F811
  """protos/dnn.proto dropout_ratio (layers/dnn.py:77-82): tf.nn.dropout after every layer's activation while training."""
  text = workloads_c2(dnn_extra='dropout_ratio: [0.5, 0.25]')
  cfg = config_util.get_configs_from_pipeline_file(text)
  import os
  os.environ['ER_PLAN_ONLY'] = '1'
  try:
    il, model, _ = builder.build_model(cfg, 32, 'cpu', cpu_generator=torch.Generator().manual_seed(1))
  finally:
    del os.environ['ER_PLAN_ONLY']
  from easyrec_b200 import layers as L
  assert [type(d).__name__ for d in model.dnn.dropouts] == ['Dropout', 'Dropout'] and model.dnn.dropouts[0].rate == 0.5
  assert all(isinstance(d, torch.nn.Identity) for d in model.final_dnn.dropouts)
  x = torch.randn(32, model.dnn.layers[0].kernel.shape[0])
  model.train()
  y1 = model.dnn(x)
  (y1.sum()).backward()
  y2 = model.dnn(x)
  assert not torch.equal(y1, y2)                                   # the counter advanced with the backward pass
  assert int(model.dnn.dropouts[1].counter[0]) == 1
  zeros = float((y1 == 0).float().mean())
  assert zeros > 0.25                                              # relu zeros + the 25 % of the last layer
  model.eval()
  assert torch.equal(model.dnn(x), model.dnn(x))                   # inference: identity


def test_lookahead_iteration_names_the_next_batch_and_never_draws_one_it_will_not_train():
  from easyrec_b200.estimator import _with_next
  drawn = []

  def src(n):
    for i in range(n):
      drawn.append(i)
      yield ('f%d' % i, 'l%d' % i)
  # no lookahead: plain iteration
  assert [(f, n) for f, _, n in _with_next(src(3), 0, lambda: True)] == [('f0', None), ('f1', None), ('f2', None)]
  # lookahead with a step limit of 3 over a longer input: the 4th batch is never drawn
  drawn.clear()
  state = {'done': 0}
  out = []
  for f, l, nxt in _with_next(src(10), 1, lambda: state['done'] + 1 < 3):
    out.append((f, None if nxt is None else nxt[0]))
    state['done'] += 1
    if state['done'] >= 3:
      break
  assert out == [('f0', 'f1'), ('f1', 'f2'), ('f2', None)] and drawn == [0, 1, 2]
  # lookahead, input shorter than the limit: the last batch has no successor
  drawn.clear()
  state = {'done': 0}
  out = []
  for f, l, nxt in _with_next(src(2), 1, lambda: state['done'] + 1 < 100):
    out.append((f, None if nxt is None else nxt[0]))
    state['done'] += 1
  assert out == [('f0', 'f1'), ('f1', None)]


def test_keras_mlp_block_dropout_ratio_follows_the_activation_of_the_listed_layers(dense_kernels):  # noqa: F811
  """layers/keras/blocks.py:56-67,113-117: Dropout(rate) after a layer when 0 < rate < 1; layers past the list get none."""
  from easyrec_b200 import backbone as BB
  from easyrec_b200.config import config_util as cu
  import test_gpu_models as G
  text = G.BACKBONE_DCN_CFG.replace('mlp { hidden_units: [64, 32] }', 'mlp { hidden_units: [64, 32] dropout_ratio: [0.5] }')
  cfg = cu.get_configs_from_pipeline_file(text.encode())
  import os
  os.environ['ER_PLAN_ONLY'] = '1'
  try:
    il, model, _ = builder.build_model(cfg, 64, 'cpu', cpu_generator=torch.Generator().manual_seed(1), default_seq_len=20)
  finally:
    del os.environ['ER_PLAN_ONLY']
  mlp = [m for m in model.modules() if isinstance(m, BB.MLP) and len(m.layers) == 2 and m.layers[0].n_out == 64][0]
  assert type(mlp.dropouts[0]).__name__ == 'Dropout' and mlp.dropouts[0].rate == 0.5
  assert isinstance(mlp.dropouts[1], torch.nn.Identity)
  x = torch.randn(64, mlp.layers[0].kernel.shape[0])
  model.train()
  a, b = mlp(x), mlp(x)
  assert torch.equal(a, b)          # no backward in between: the same step, the same mask
  a.sum().backward()
  assert not torch.equal(mlp(x), a)
  model.eval()
  assert torch.equal(mlp(x), mlp(x))


def test_two_optimizer_configs_train_tables_with_the_first_and_everything_else_with_the_second(dense_kernels):  # noqa: F811
  """model/easy_rec_estimator.py:216-232 + EasyRecModel.get_grouped_vars (easy_rec_model.py:446-467): optimizer_config[0]
  for the embedding tables, [1] for the other variables - kinds, schedules and Adam state apart."""
  from easyrec_b200 import workloads
  from easyrec_b200.estimator import EasyRecEstimator
  text = workloads.c2_config_text(1000, 32, dnn=(16, 8), final=(8, 4)).decode()
  one = 'optimizer_config { adagrad_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.01 } } } }'
  assert one in text
  two = ('optimizer_config { adagrad_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.05 } } } } '
         'optimizer_config { adam_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.001 } } } }')
  est = EasyRecEstimator(text.replace(one, two).encode(), device='cpu', seed=3)
  il, tr = est.input_layer, est.trainer
  assert il.arenas[16].opt_kind == _lib.OPT_ADAGRAD and il.arenas[16].state1 is None
  assert tr.dense_opt.kind == _lib.OPT_ADAM_ROWS and tr.dense_opt.s1 is not None
  assert tr.dense_opt.hyper is not il.hyper
  ids, dense, labels = workloads.criteo_batch(32, 5)
  feats = {'sparse_fea': torch.from_numpy(ids), 'dense_fea': torch.from_numpy(dense)}
  w0 = il.arenas[16].weight.clone()
  p0 = tr.dense_opt.flat_p.clone()
  tr.train_step(feats, torch.from_numpy(labels))
  assert abs(il.hyper.lr - 0.05) < 1e-9 and abs(tr.dense_opt.hyper.lr - 0.001) < 1e-9
  # first Adam step moves every dense weight with a gradient by ~lr (|m/sqrt(v)| = 1 after bias correction)
  dp = (tr.dense_opt.flat_p - p0).abs()
  assert 0.0009 < float(dp[dp > 0].median()) < 0.0011
  # the touched rows took an Adagrad step of the embedding rate: |dw| = 0.05 |g| / sqrt(0.1 + g^2) < 0.05
  dw = (il.arenas[16].weight - w0).abs()
  assert 0 < float(dw.max()) < 0.05
  # three entries are refused
  cfg = config_util.get_configs_from_pipeline_file(text.replace(one, two + ' ' + one).encode())
  with pytest.raises(NotImplementedError, match='optimizer_config entries'):
    builder.check_scope(cfg)


def test_sample_weight_field_weighs_the_loss_by_nonzero_weight_mean(tmp_path, dense_kernels):  # noqa: F811
  """data_config.sample_weight (input/input.py:140-141) -> tf.losses.sigmoid_cross_entropy(weights=...)
  (model/rank_model.py:213-269): sum(w * ce) / count_nonzero(w); a zero-weight sample moves no table row."""
  from easyrec_b200.estimator import EasyRecEstimator
  cfg_text = b'''
train_config { optimizer_config { adagrad_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.05 } } } } }
data_config { batch_size: 8 input_type: CSVInput separator: "," label_fields: "label" sample_weight: "w"
  input_fields { input_name: "label" input_type: FLOAT } input_fields { input_name: "w" input_type: FLOAT }
  input_fields { input_name: "uid" input_type: INT64 } input_fields { input_name: "x" input_type: FLOAT } }
feature_config {
  features { input_names: "uid" feature_type: IdFeature embedding_dim: 4 num_buckets: 50 }
  features { input_names: "x" feature_type: RawFeature embedding_dim: 4 min_val: 0.0 max_val: 4.0 } }
model_config { model_class: "DeepFM"
  feature_groups { group_name: "deep" feature_names: ["uid", "x"] wide_deep: DEEP }
  feature_groups { group_name: "wide" feature_names: ["uid", "x"] wide_deep: WIDE }
  deepfm { dnn { hidden_units: [8] use_bn: false } final_dnn { hidden_units: [4] use_bn: false } } }
'''
  # (no batch norm: nothing couples the samples, so a zero-weight sample has a zero gradient)
  rows = [(1, 2.0, 3, 1.0), (0, 0.0, 7, 2.0), (1, 0.5, 9, 3.0), (0, 1.0, 11, 0.5), (1, 0.0, 13, 1.5), (0, 3.0, 15, 2.5),
          (1, 1.0, 17, 3.5), (0, 1.0, 19, 0.0)]
  path = tmp_path / 'sw.csv'
  path.write_text(''.join('%d,%g,%d,%g\n' % r for r in rows))
  est = EasyRecEstimator(cfg_text, device='cpu', seed=3)
  for engine in ('native', 'python'):
    (feats, labels), = list(readers.CSVInput(est._pipeline_config, est.input_layer, str(path), engine=engine))
    assert feats['sample_weight'].tolist() == [r[1] for r in rows]
  il = est.input_layer
  w0 = il.arenas[4].weight.clone()
  est.model.train()
  logits = est.model(feats).detach()
  want_loss, _, _ = O.sigmoid_ce(logits.numpy(), labels.numpy(), weights=feats['sample_weight'].numpy())
  il._pending = []
  loss, _ = est.trainer.train_step(feats, labels)
  reg = float(est.trainer.dense_opt.reg_loss[0])     # deepfm.l2_regularization defaults to 1e-4 (protos/deepfm.proto)
  assert abs(float(loss) - reg - want_loss) < 1e-6
  moved = ((il.arenas[4].weight - w0).abs().sum(1) > 0).nonzero().reshape(-1).tolist()
  off = il.arenas[4].tables['uid_embedding'][0]
  zero_w = [off + r[2] for r in rows if r[1] == 0.0]
  live = [off + r[2] for r in rows if r[1] != 0.0]
  assert all(r not in moved for r in zero_w) and all(r in moved for r in live)


CLIP_CFG = b'''
train_config { %s
  optimizer_config { momentum_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.5 } }
                                          momentum_optimizer_value: 0.0 } } }
data_config { batch_size: 16 input_type: DummyInput label_fields: "label" }
feature_config {
  features { input_names: "a" feature_type: IdFeature embedding_dim: 4 num_buckets: 6 embedding_name: "shared" }
  features { input_names: "b" feature_type: IdFeature embedding_dim: 4 num_buckets: 6 embedding_name: "shared" }
  features { input_names: "c" feature_type: IdFeature embedding_dim: 4 hash_bucket_size: 11 }
  features { input_names: "x" feature_type: RawFeature embedding_dim: 4 min_val: 0.0 max_val: 2.0 } }
model_config { model_class: "DeepFM"
  feature_groups { group_name: "deep" feature_names: ["a", "b", "c", "x"] wide_deep: DEEP }
  feature_groups { group_name: "wide" feature_names: ["a", "b", "c", "x"] wide_deep: WIDE }
  deepfm { dnn { hidden_units: [8] } final_dnn { hidden_units: [4] } l2_regularization: 1e-2 }
  embedding_regularization: 1e-3 }
'''


def test_global_norm_clipping_scales_every_gradient_by_clip_over_the_tf_global_norm(dense_kernels):  # noqa: F811
  """train_config.gradient_clipping_by_norm (compat/optimizers.py:365-376, 453-481): norm over the dense gradients
  (regularisers included) and the tables' IndexedSlices, which TF deduplicates per COLUMN even when columns share a
  table; every gradient is scaled by clip / max(norm, clip) before the update."""
  from easyrec_b200.estimator import EasyRecEstimator
  rng = np.random.default_rng(0)
  B = 16
  ids = np.stack([rng.integers(0, 6, B), rng.integers(0, 6, B), rng.integers(0, 1000, B)]).astype(np.int64)   # a, b collide
  feats = {'sparse_fea': torch.from_numpy(ids.reshape(-1)), 'dense_fea': torch.from_numpy(rng.uniform(0, 2, (B, 1)).astype(np.float32))}
  labels = torch.from_numpy((rng.uniform(size=B) < 0.4).astype(np.float32))
  plain = EasyRecEstimator(CLIP_CFG % b'', device='cpu', seed=11)
  clip = EasyRecEstimator(CLIP_CFG % b'gradient_clipping_by_norm: 0.05', device='cpu', seed=11)
  assert clip.trainer.clip_norm == pytest.approx(0.05) and plain.trainer.clip_norm == 0.0
  # -- the norm: an independent restatement from the per-lookup gradients of one backward pass
  tr, il = clip.trainer, clip.input_layer
  tr._set_hyper()
  clip.model.train()
  tr._segment_compute(feats, labels)
  want_sq = 0.0
  for m, rows, w, outs, seg_ids in il._pending:
    a, D = m.arena, m.arena.dim
    r = rows.numpy()
    for sl in m.slots_np:                      # one IndexedSlices per column: unique rows of THAT column
      g = outs[int(sl['out_buf'])].grad.numpy().reshape(-1, int(sl['out_stride']))[:, int(sl['out_col']):int(sl['out_col']) + D]
      lo = int(sl['seg_begin'])
      rr = r[lo:lo + int(sl['n_seg'])]
      ww = np.ones(rr.size, np.float32) if w is None else w.numpy()[lo:lo + rr.size]
      for u in np.unique(rr[rr >= 0]):
        want_sq += float(((g[rr == u] * ww[rr == u, None]).sum(0).astype(np.float64) ** 2).sum())
  opt = tr.dense_opt
  l2 = torch.from_numpy(opt._l2_vec_np)
  want_sq += float(((opt.flat_g + l2 * opt.flat_p).double() ** 2).sum())
  got_sparse = float(il.sparse_grad_sqnorm())
  got = float(torch.sqrt(torch.tensor(got_sparse) + ((opt.flat_g + l2 * opt.flat_p) ** 2).sum()))
  assert got == pytest.approx(np.sqrt(want_sq), rel=1e-5)
  il._pending = []
  # -- the step: with plain SGD every update is linear in its gradient, so clipped = scale * unclipped everywhere
  clip2 = EasyRecEstimator(CLIP_CFG % b'gradient_clipping_by_norm: 0.05', device='cpu', seed=11)
  before_p = plain.trainer.dense_opt.flat_p.clone()
  before_t = {d: a.weight.clone() for d, a in plain.input_layer.arenas.items()}
  plain.trainer.train_step(feats, labels)
  clip2.trainer.train_step(feats, labels)
  norm = float(clip2.trainer.last_grad_norm)
  assert norm == pytest.approx(np.sqrt(want_sq), rel=1e-5) and norm > 0.05
  scale = 0.05 / norm
  dp_plain = plain.trainer.dense_opt.flat_p - before_p
  dp_clip = clip2.trainer.dense_opt.flat_p - before_p
  torch.testing.assert_close(dp_clip, dp_plain * scale, rtol=1e-4, atol=2e-7)   # (differences of O(1) fp32 parameters)
  assert float(dp_plain.abs().max()) > 1e-3
  for d, a in clip2.input_layer.arenas.items():
    dt_plain = plain.input_layer.arenas[d].weight - before_t[d]
    torch.testing.assert_close(a.weight - before_t[d], dt_plain * scale, rtol=1e-4, atol=2e-8)
    assert float(dt_plain.abs().max()) > 1e-4
  # a clip above the norm leaves the step untouched
  loose = EasyRecEstimator(CLIP_CFG % b'gradient_clipping_by_norm: 1000.0', device='cpu', seed=11)
  loose.trainer.train_step(feats, labels)
  torch.testing.assert_close(loose.trainer.dense_opt.flat_p, plain.trainer.dense_opt.flat_p, rtol=1e-6, atol=2e-7)


@pytest.mark.parametrize('loss_type', ['L2_LOSS', 'SIGMOID_L2_LOSS'])
def test_l2_loss_types_train_the_rank_head_as_a_regressor(loss_type, dense_kernels):  # noqa: F811
  """model_config.loss_type L2_LOSS / SIGMOID_L2_LOSS (builders/loss_builder.py:52-55, model/rank_model.py:123-128):
  mean squared error between the label and y = logits / sigmoid(logits); predictions are `y`."""
  from easyrec_b200 import workloads
  from easyrec_b200.estimator import EasyRecEstimator
  text = workloads.c2_config_text(1000, 32, dnn=(16, 8), final=(8, 4)).decode()
  text = text.replace('model_config { model_class: "DeepFM"', 'model_config { model_class: "DeepFM" loss_type: %s' % loss_type)
  est = EasyRecEstimator(text.encode(), device='cpu', seed=3)
  assert est.model.loss_type == loss_type
  ids, dense, _ = workloads.criteo_batch(32, 5)
  labels = torch.from_numpy(np.random.default_rng(1).uniform(0, 1, 32).astype(np.float32))
  feats = {'sparse_fea': torch.from_numpy(ids), 'dense_fea': torch.from_numpy(dense)}
  est.model.train()
  logits = est.model(feats)
  y = torch.sigmoid(logits) if loss_type == 'SIGMOID_L2_LOSS' else logits
  loss, pred = est.model.loss(logits, labels)
  want = ((y - labels) ** 2).mean() + est.model.regularization_loss()
  assert abs(float(loss) - float(want)) < 1e-6 and torch.allclose(pred, y.detach())
  est.input_layer._pending = []
  losses = [float(est.trainer.train_step(feats, labels)[0]) for _ in range(30)]
  assert losses[-1] < losses[0]


def test_multi_tower_model_class_trains_from_its_config(interaction_doubles):  # noqa: F811
  """model_class MultiTower (model/multi_tower.py:17-62): batch-normed group -> DNN per tower, concat, final DNN."""
  import test_gpu_models as G
  text = G.HEAD + G.FEATS + '''
model_config { model_class: "MultiTower"
  feature_groups { group_name: "user" feature_names: ["user_id", "age"] wide_deep: DEEP }
  feature_groups { group_name: "item" feature_names: ["item_id", "cate", "price"] wide_deep: DEEP }
  multi_tower { towers { input: "user" dnn { hidden_units: [32, 16] } } towers { input: "item" dnn { hidden_units: [32, 16] } }
                final_dnn { hidden_units: [32, 16] } l2_regularization: 1e-5 }
  embedding_regularization: 1e-5 }
'''
  cfg = config_util.get_configs_from_pipeline_file(text.encode())
  B = 256
  il, model, opt = builder.build_model(cfg, B, 'cpu', cpu_generator=torch.Generator().manual_seed(1), default_seq_len=20)
  assert type(model).__name__ == 'MultiTower' and len(model.din_dnn) == 0 and len(model.tower_dnn) == 2
  rng = np.random.default_rng(0)
  ids = np.stack([rng.integers(0, 10**6, B), rng.integers(0, 10, B), rng.integers(0, 10**6, B), rng.integers(0, 500, B)])
  feats = {'sparse_fea': torch.from_numpy(ids.reshape(-1).astype(np.int64)),
           'dense_fea': torch.from_numpy(rng.uniform(0, 100, (B, 1)).astype(np.float32))}
  lab = torch.from_numpy((rng.uniform(size=B) < 0.3).astype(np.float32))
  tr = T.Trainer(model, il, 'adagrad', lr_fn=opt['lr_fn'])
  losses = [float(tr.train_step(feats, lab)[0]) for _ in range(15)]
  assert losses[-1] < losses[0] - 0.01


def test_in_group_sequence_features_append_target_attention_to_the_group(interaction_doubles):  # noqa: F811
  """feature_groups[...].sequence_features (layers/input_layer.py:96-111, layers/sequence_feature_layer.py:123-249):
  the key reuses the group's own embedding of that feature, the history lives in the group's scope (or the shared
  embedding_name), [attended history | key] is appended to the group's concat, the regulariser sees what was looked up."""
  import test_gpu_models as G
  feats_cfg = G.FEATS.replace('features { input_names: "item_id" feature_type: IdFeature embedding_dim: 16 hash_bucket_size: 5000 }',
                              'features { input_names: "item_id" feature_type: IdFeature embedding_dim: 16 hash_bucket_size: 5000 embedding_name: "item" }')
  feats_cfg = feats_cfg.replace('hash_bucket_size: 5000 max_seq_len: 20', 'hash_bucket_size: 5000 max_seq_len: 20 embedding_name: "item"')
  text = G.HEAD + feats_cfg + '''
model_config { model_class: "MultiTower"
  feature_groups { group_name: "user" feature_names: ["user_id", "age"] wide_deep: DEEP }
  feature_groups { group_name: "item" feature_names: ["item_id", "cate", "price"] wide_deep: DEEP
                   sequence_features { group_name: "seq" seq_att_map { key: "item_id" hist_seq: "hist_items" }
                                       seq_dnn { hidden_units: [8, 1] } } }
  multi_tower { towers { input: "user" dnn { hidden_units: [32, 16] } } towers { input: "item" dnn { hidden_units: [32, 16] } }
                final_dnn { hidden_units: [32, 16] } l2_regularization: 1e-5 }
  embedding_regularization: 1e-5 }
'''
  cfg = config_util.get_configs_from_pipeline_file(text.encode())
  B = 256
  il, model, opt = builder.build_model(cfg, B, 'cpu', cpu_generator=torch.Generator().manual_seed(1), default_seq_len=20)
  assert [e[1] for e in il.group_layout['item']] == ['emb', 'emb', 'emb', 'att'] and il.group_layout['item'][-1][2] == 32
  assert 'item' in il.arenas[16].tables and 'item_id_embedding' not in il.arenas[16].tables   # key and history share it
  assert sorted(dict(model.named_parameters())) != [] and any(n.startswith('input_attention.') for n, _ in model.named_parameters())
  rng = np.random.default_rng(0)
  ids = np.stack([rng.integers(0, 10**6, B), rng.integers(0, 10, B), rng.integers(0, 10**6, B), rng.integers(0, 500, B)])
  T_ = 20
  hist = rng.integers(0, 10**6, (B, T_)).astype(np.int64)
  lens = rng.integers(0, T_ + 1, B).astype(np.int32)
  feats = {'sparse_fea': torch.from_numpy(ids.reshape(-1).astype(np.int64)),
           'dense_fea': torch.from_numpy(rng.uniform(0, 100, (B, 1)).astype(np.float32)),
           'seq_fea': {'hist_items': (torch.from_numpy(hist), torch.from_numpy(lens))}}
  model.train()
  g = il.lookup(feats)
  concat, per = g['item']
  assert concat.shape == (B, 16 * 3 + 32) and len(per) == 4
  W = il.arenas[16].weight.detach().numpy()
  off = il.arenas[16].tables['item'][0]
  key = W[off + O.bucketize(ids[2], 0, 5000, 0)[0]]
  np.testing.assert_array_equal(concat[:, :16].detach().numpy(), key)                # the group's own item_id column
  np.testing.assert_array_equal(concat[:, 64:80].detach().numpy(), key)              # ... is the attention's key
  hrows = O.bucketize(hist.reshape(-1), 0, 5000, 0)[0].reshape(B, T_)
  he = W[off + hrows] * (np.arange(T_)[None, :] < lens[:, None])[:, :, None]
  dnn = il.attention_modules['item/seq']
  layers = [dict(W=l.kernel.detach().numpy(), b=l.bias.detach().numpy(),
                 **(dict(gamma=l.gamma.detach().numpy(), beta=l.beta.detach().numpy()) if l.use_bn else {})) for l in dnn.layers]
  want = O.din_attention(key, he.astype(np.float32), lens, layers)
  np.testing.assert_allclose(concat[:, 48:64].detach().numpy(), want, rtol=1e-4, atol=1e-6)
  assert len(concat._er_reg) == 4     # three looked-up columns + the history
  il._pending = []
  tr = T.Trainer(model, il, 'adagrad', lr_fn=opt['lr_fn'])
  lab = torch.from_numpy((rng.uniform(size=B) < 0.3).astype(np.float32))
  p0 = dnn.layers[0].kernel.detach().clone()
  losses = [float(tr.train_step(feats, lab)[0]) for _ in range(12)]
  assert losses[-1] < losses[0] - 0.01 and not torch.equal(dnn.layers[0].kernel.detach(), p0)   # the attention MLP trains


def test_dbmtl_and_simple_multi_task_train_from_their_configs(interaction_doubles):  # noqa: F811
  """model_class DBMTL (model/dbmtl.py:44-121: bottom DNN, MMoE experts, tower DNNs, relation DNNs over the towers a
  task depends on) and SimpleMultiTask (model/simple_multi_task.py:38-55), composed from the same layers as MMoE."""
  import test_gpu_models as G
  head = G.HEAD.replace('label_fields: "clk"', 'label_fields: ["clk", "buy"]')
  group = 'feature_groups { group_name: "all" feature_names: ["user_id", "age", "item_id", "cate", "price"] wide_deep: DEEP }'
  dbmtl = head + G.FEATS + '''
model_config { model_class: "DBMTL" %s
  dbmtl { bottom_dnn { hidden_units: [64] } expert_dnn { hidden_units: [32] } num_expert: 3
          task_towers { tower_name: "ctr" label_name: "clk" loss_type: CLASSIFICATION dnn { hidden_units: [16] }
                        relation_dnn { hidden_units: [8] } weight: 1.0 }
          task_towers { tower_name: "cvr" label_name: "buy" loss_type: CLASSIFICATION dnn { hidden_units: [16] }
                        relation_tower_names: ["ctr"] relation_dnn { hidden_units: [8] } weight: 0.5 }
          l2_regularization: 1e-5 }
  embedding_regularization: 1e-5 }
''' % group
  smt = head + G.FEATS + '''
model_config { model_class: "SimpleMultiTask" %s
  simple_multi_task { task_towers { tower_name: "ctr" label_name: "clk" dnn { hidden_units: [32, 16] } weight: 1.0 }
                      task_towers { tower_name: "cvr" label_name: "buy" dnn { hidden_units: [32, 16] } weight: 1.0 }
                      l2_regularization: 1e-5 }
  embedding_regularization: 1e-5 }
''' % group
  B = 256
  rng = np.random.default_rng(0)
  ids = np.stack([rng.integers(0, 10**6, B), rng.integers(0, 10, B), rng.integers(0, 10**6, B), rng.integers(0, 500, B)])
  feats = {'sparse_fea': torch.from_numpy(ids.reshape(-1).astype(np.int64)),
           'dense_fea': torch.from_numpy(rng.uniform(0, 100, (B, 1)).astype(np.float32))}
  lab = torch.from_numpy((rng.uniform(size=(B, 2)) < 0.3).astype(np.float32))
  for text, name in ((dbmtl, 'DBMTL'), (smt, 'SimpleMultiTask')):
    cfg = config_util.get_configs_from_pipeline_file(text.encode())
    il, model, opt = builder.build_model(cfg, B, 'cpu', cpu_generator=torch.Generator().manual_seed(1), default_seq_len=20)
    assert type(model).__name__ == name and model.label_cols == [0, 1]
    if name == 'DBMTL':
      assert model.relations == [[], [0]] and model.relation_dnn[1].layers[0].kernel.shape[0] == 16 + 8
    tr = T.Trainer(model, il, 'adagrad', lr_fn=opt['lr_fn'])
    losses = [float(tr.train_step(feats, lab)[0]) for _ in range(15)]
    assert losses[-1] < losses[0] - 0.01, (name, losses)


def test_wide_and_deep_and_fm_model_classes_match_their_formulas(interaction_doubles):  # noqa: F811
  """model/wide_and_deep.py:44-80 (with and without final_dnn) and model/fm.py:43-62 on the shared wide / deep groups."""
  import test_gpu_models as G
  feats_cfg = G.FEATS.replace('features { input_names: "price" feature_type: RawFeature embedding_dim: 16 min_val: 0 max_val: 100 }\n', '')
  groups = ('feature_groups { group_name: "deep" feature_names: ["user_id", "age", "item_id", "cate"] wide_deep: DEEP }\n'
            '  feature_groups { group_name: "wide" feature_names: ["user_id", "item_id", "cate"] wide_deep: WIDE }')
  B = 256
  rng = np.random.default_rng(0)
  ids = np.stack([rng.integers(0, 10**6, B), rng.integers(0, 10, B), rng.integers(0, 10**6, B), rng.integers(0, 500, B)])
  feats = {'sparse_fea': torch.from_numpy(ids.reshape(-1).astype(np.int64))}
  lab = torch.from_numpy((rng.uniform(size=B) < 0.3).astype(np.float32))
  cases = (('WideAndDeep', 'wide_and_deep { wide_output_dim: 4 dnn { hidden_units: [32, 16] } final_dnn { hidden_units: [8] } l2_regularization: 1e-5 }'),
           ('WideAndDeep', 'wide_and_deep { wide_output_dim: 4 dnn { hidden_units: [32, 16] } l2_regularization: 1e-5 }'),
           ('FM', 'fm { l2_regularization: 1e-5 }'))
  for name, body in cases:
    text = G.HEAD + feats_cfg + 'model_config { model_class: "%s"\n  %s\n  %s\n  embedding_regularization: 1e-5 }' % (name, groups, body)
    cfg = config_util.get_configs_from_pipeline_file(text.encode())
    il, model, opt = builder.build_model(cfg, B, 'cpu', cpu_generator=torch.Generator().manual_seed(1), default_seq_len=20)
    model.train()
    logits = model(feats).detach()
    g = il.lookup(feats)
    wide, deep = g['wide'][0].detach(), g['deep'][0].detach()
    il._pending = []
    if name == 'FM':
      assert wide.shape == (B, 3)                                       # wide_output_dim = num_class = 1
      v = deep.reshape(B, 4, 16)
      second = 0.5 * ((v.sum(1) ** 2) - (v ** 2).sum(1)).sum(1)
      torch.testing.assert_close(logits, wide.sum(1) + second + model.fm_bias.detach()[0], rtol=1e-5, atol=1e-6)
    elif 'final_dnn' in body:
      assert wide.shape == (B, 12)                                      # 3 features x wide_output_dim 4
      wide_fea = wide.reshape(B, 3, 4).sum(1)
      want = model.output(model.final_dnn(torch.cat([wide_fea, model.dnn(deep)], 1)))[:, 0].detach()
      torch.testing.assert_close(logits, want, rtol=1e-5, atol=1e-6)
    else:
      assert wide.shape == (B, 3)                                       # no final_dnn: the wide sum is the logit's other half
      want = (model.output(model.dnn(deep))[:, 0] + wide.sum(1)).detach()
      torch.testing.assert_close(logits, want, rtol=1e-5, atol=1e-6)
    tr = T.Trainer(model, il, 'adagrad', lr_fn=opt['lr_fn'])
    losses = [float(tr.train_step(feats, lab)[0]) for _ in range(15)]
    assert losses[-1] < losses[0] - 0.005, (name, losses)


def test_a_task_tower_with_an_l2_loss_type_is_trained_as_a_regressor(interaction_doubles):  # noqa: F811
  """TaskTower.loss_type (protos/tower.proto, model/multi_task_model.py:201-280): per tower CLASSIFICATION or an L2 loss."""
  import test_gpu_models as G
  text = G.MMOE_CFG.replace('loss_type: CLASSIFICATION weight: 0.5', 'loss_type: L2_LOSS weight: 0.5')
  assert text != G.MMOE_CFG
  cfg = config_util.get_configs_from_pipeline_file(text.encode())
  B = G.B
  il, model, opt = builder.build_model(cfg, B, 'cpu', cpu_generator=torch.Generator().manual_seed(1), default_seq_len=20)
  assert sorted(model.task_loss_types) == ['CLASSIFICATION', 'L2_LOSS']
  t_l2 = model.task_loss_types.index('L2_LOSS')
  rng = np.random.default_rng(0)
  ids = np.stack([rng.integers(0, 10**6, B), rng.integers(0, 10, B), rng.integers(0, 10**6, B), rng.integers(0, 500, B)])
  feats = {'sparse_fea': torch.from_numpy(ids.reshape(-1).astype(np.int64)),
           'dense_fea': torch.from_numpy(rng.uniform(0, 100, (B, 1)).astype(np.float32))}
  labels = torch.from_numpy(rng.uniform(0, 1, (B, 2)).astype(np.float32))
  model.train()
  logits = model(feats)
  loss, preds = model.loss(logits, labels)
  cols = model.label_cols
  want = 0.0
  for t, w in enumerate(model.task_weights):
    x, z = logits[:, t], labels[:, cols[t]]
    if t == t_l2:
      want = want + w * ((x - z) ** 2).mean()
    else:
      want = want + w * torch.nn.functional.binary_cross_entropy_with_logits(x, z)
  want = want + model.embedding_reg_loss(model._emb_outputs)
  assert abs(float(loss) - float(want)) < 1e-5
  torch.testing.assert_close(preds[:, t_l2], logits[:, t_l2].detach())     # a regressor predicts y = its output


def test_ple_model_class_trains_and_its_gates_mix_own_and_shared_experts(interaction_doubles):  # noqa: F811
  """model_class PLE (model/ple.py:36-128): two extraction networks, the last one without a shared gate."""
  import test_gpu_models as G
  head = G.HEAD.replace('label_fields: "clk"', 'label_fields: ["clk", "buy"]')
  text = head + G.FEATS + '''
model_config { model_class: "PLE"
  feature_groups { group_name: "all" feature_names: ["user_id", "age", "item_id", "cate", "price"] wide_deep: DEEP }
  ple { extraction_networks { network_name: "l1" expert_num_per_task: 2 share_num: 2
                              task_expert_net { hidden_units: [32] } share_expert_net { hidden_units: [32] } }
        extraction_networks { network_name: "l2" expert_num_per_task: 1 share_num: 1
                              task_expert_net { hidden_units: [16] } share_expert_net { hidden_units: [16] } }
        task_towers { tower_name: "ctr" label_name: "clk" dnn { hidden_units: [8] } weight: 1.0 }
        task_towers { tower_name: "cvr" label_name: "buy" dnn { hidden_units: [8] } weight: 1.0 }
        l2_regularization: 1e-5 }
  embedding_regularization: 1e-5 }
'''
  cfg = config_util.get_configs_from_pipeline_file(text.encode())
  B = 256
  il, model, opt = builder.build_model(cfg, B, 'cpu', cpu_generator=torch.Generator().manual_seed(1), default_seq_len=20)
  assert type(model).__name__ == 'PLE' and len(model.nets) == 2
  n1, n2 = model.nets
  assert n1.task_gate[0].kernel.shape[1] == 4 and n1.share_gate.kernel.shape[1] == 6      # 2 own + 2 shared; all 4 + 2 shared
  assert n2.share_gate is None and n2.task_gate[1].kernel.shape == (32, 2)
  rng = np.random.default_rng(0)
  ids = np.stack([rng.integers(0, 10**6, B), rng.integers(0, 10, B), rng.integers(0, 10**6, B), rng.integers(0, 500, B)])
  feats = {'sparse_fea': torch.from_numpy(ids.reshape(-1).astype(np.int64)),
           'dense_fea': torch.from_numpy(rng.uniform(0, 100, (B, 1)).astype(np.float32))}
  lab = torch.from_numpy((rng.uniform(size=(B, 2)) < 0.3).astype(np.float32))
  tr = T.Trainer(model, il, 'adagrad', lr_fn=opt['lr_fn'])
  losses = [float(tr.train_step(feats, lab)[0]) for _ in range(15)]
  assert losses[-1] < losses[0] - 0.01, losses


def test_backbone_embedding_layer_block_pools_padded_tag_features(interaction_doubles, tmp_path):  # noqa: F811
  """§8 a23, multi-valued inputs (layers/input_layer.py:232-235 + layers/keras/embedding.py:9-23, 60-78): the ragged tags
  are densified with '' up to the longest list of the batch, the PADDING is hashed and looked up too, and the positions are
  pooled by the block's combiner - 'weight' without weights = mean over ALL positions, with kv weights sum(w e)/sum(w)."""
  from easyrec_b200.input import readers
  text = b"""
train_config { optimizer_config { adagrad_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.05 } } } } }
data_config { batch_size: 4 input_type: CSVInput separator: "," label_fields: "label"
  input_fields { input_name: "label" input_type: FLOAT } input_fields { input_name: "u" input_type: INT64 }
  input_fields { input_name: "tags" input_type: STRING } input_fields { input_name: "kv" input_type: STRING } }
feature_config {
  features { input_names: "u" feature_type: IdFeature embedding_dim: 8 hash_bucket_size: 50 }
  features { input_names: "tags" feature_type: TagFeature embedding_dim: 8 hash_bucket_size: 31 separator: "|" }
  features { input_names: "kv" feature_type: TagFeature embedding_dim: 8 hash_bucket_size: 17 separator: "|" kv_separator: ":" } }
model_config { model_class: "RankModel"
  feature_groups { group_name: "ids" feature_names: ["u", "tags", "kv"] wide_deep: DEEP }
  backbone {
    blocks { name: "emb" inputs { feature_group_name: "ids" } embedding_layer { embedding_dim: 6 } }
    blocks { name: "mlp" inputs { block_name: "emb" } keras_layer { class_name: "MLP" mlp { hidden_units: [8] } } }
    concat_blocks: ["mlp"] } }
"""
  cfg = config_util.get_configs_from_pipeline_file(text)
  il, model, opt = builder.build_model(cfg, 4, 'cpu', cpu_generator=torch.Generator().manual_seed(1))
  pad_t, pad_k = O.fingerprint64('') % 31, O.fingerprint64('') % 17
  assert il.pad_tags == {'tags': (pad_t, True), 'kv': (pad_k, True)}
  a = il.arenas[6]
  assert list(a.tables) == ['emb/u_embedding', 'emb/tags_embedding', 'emb/kv_embedding']    # offsets in group order
  open(tmp_path / 't.csv', 'w').write('1,7,a|b|c,x:2|y:0.5\n0,8,,z:1\n1,9,d,\n0,7,e|f,x:1|z:3\n')
  for engine in ('native', 'python'):
    (feats, labels), = list(readers.CSVInput(cfg, il, str(tmp_path / 't.csv'), engine=engine))
    ids, lens, w = feats['tag_fea']['tags']
    h = lambda s, nb: O.fingerprint64(s) % nb   # noqa: E731
    assert lens.tolist() == [3, 3, 3, 3] and w is None                       # padded to the batch's longest list
    assert ids.tolist() == [h('a', 31), h('b', 31), h('c', 31), pad_t, pad_t, pad_t, h('d', 31), pad_t, pad_t,
                            h('e', 31), h('f', 31), pad_t]
    ids_k, lens_k, w_k = feats['tag_fea']['kv']
    assert lens_k.tolist() == [2, 2, 2, 2] and w_k.tolist() == [2.0, 0.5, 1.0, 0.0, 0.0, 0.0, 1.0, 3.0]
    out = il.lookup(feats)['ids'][0].detach().numpy()
    W = a.weight.detach().numpy()
    o_t, o_k = a.tables['emb/tags_embedding'][0], a.tables['emb/kv_embedding'][0]
    want_tags = W[o_t + ids.numpy().reshape(4, 3)].mean(1)                    # 'weight' without weights: mean incl. padding
    np.testing.assert_allclose(out[:, 6:12], want_tags, rtol=1e-5, atol=1e-7)
    wk = w_k.numpy().reshape(4, 2)
    rows_k = W[o_k + ids_k.numpy().reshape(4, 2)]
    with np.errstate(invalid='ignore', divide='ignore'):
      want_kv = (rows_k * wk[:, :, None]).sum(1) / wk.sum(1, keepdims=True)
    want_kv[2] = 0.0   # a sample without tags: the reference divides 0 by 0 there (NaN); this path gives the zero vector
    np.testing.assert_allclose(out[:, 12:18], want_kv, rtol=1e-5, atol=1e-7)
    il._pending = []
  tr = T.Trainer(model, il, 'adagrad', lr_fn=opt['lr_fn'])
  feats, labels = list(readers.CSVInput(cfg, il, str(tmp_path / 't.csv')))[0]
  losses = [float(tr.train_step(feats, labels)[0]) for _ in range(20)]
  assert losses[-1] < losses[0] - 0.01
  # the padding row itself is trained (it is looked up like a tag)
  assert float((a.weight[a.tables['emb/tags_embedding'][0] + pad_t]).abs().sum()) > 0
  bad = config_util.get_configs_from_pipeline_file(text.replace(b'embedding_layer { embedding_dim: 6 }',
                                                                b'embedding_layer { embedding_dim: 6 combiner: "max" }'))
  with pytest.raises(NotImplementedError, match='combiner'):
    builder.build_model(bad, 4, 'cpu', cpu_generator=torch.Generator().manual_seed(1))


def test_global_norm_clipping_over_tag_slots(dense_kernels, tmp_path):  # noqa: F811
  """gradient_clipping_by_norm with multi-valued (CSR) slots: the IndexedSlices of a tag column hold one row per distinct
  tag of the column, summed over its lookups with their weights and the combiner's per-sample scale."""
  from easyrec_b200.estimator import EasyRecEstimator
  from easyrec_b200.input import readers
  text = b"""
train_config { %s
  optimizer_config { momentum_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.5 } }
                                          momentum_optimizer_value: 0.0 } } }
data_config { batch_size: 6 input_type: CSVInput separator: "," label_fields: "label"
  input_fields { input_name: "label" input_type: FLOAT } input_fields { input_name: "a" input_type: INT64 }
  input_fields { input_name: "t" input_type: STRING } input_fields { input_name: "s" input_type: STRING } }
feature_config {
  features { input_names: "a" feature_type: IdFeature embedding_dim: 4 num_buckets: 7 embedding_name: "e" }
  features { input_names: "t" feature_type: TagFeature embedding_dim: 4 num_buckets: 7 embedding_name: "e" separator: "|"
             kv_separator: ":" combiner: "mean" }
  features { input_names: "s" feature_type: TagFeature embedding_dim: 4 hash_bucket_size: 9 separator: "|" combiner: "sum" } }
model_config { model_class: "MultiTower"
  feature_groups { group_name: "g" feature_names: ["a", "t", "s"] wide_deep: DEEP }
  multi_tower { towers { input: "g" dnn { hidden_units: [8] } } final_dnn { hidden_units: [4] } l2_regularization: 1e-2 } }
"""
  open(tmp_path / 'c.csv', 'w').write('1,1,1:0.5|2:2|1:1,x|y\n0,2,,x\n1,1,3:1,\n0,6,2:1|2:3,y|y|z\n1,0,5:2,w\n0,3,1:1|4:1,x|w\n')
  plain = EasyRecEstimator(text % b'', device='cpu', seed=4)
  clip = EasyRecEstimator(text % b'gradient_clipping_by_norm: 0.02', device='cpu', seed=4)
  probe = EasyRecEstimator(text % b'', device='cpu', seed=4)
  (feats, labels), = list(readers.CSVInput(plain._pipeline_config, plain.input_layer, str(tmp_path / 'c.csv')))
  # -- the norm, restated lookup by lookup
  tr, il = probe.trainer, probe.input_layer
  tr._set_hyper()
  probe.model.train()
  tr._segment_compute(feats, labels)
  want_sq = 0.0
  for m, rows, w, outs, seg_ids in il._pending:
    D = m.arena.dim
    r = rows.numpy()
    seg = np.arange(r.size) if seg_ids is None else seg_ids.numpy()[:r.size]
    scale = np.ones(m.n_seg, np.float32) if m.seg_scale is None else m.seg_scale.numpy()
    ww = np.ones(r.size, np.float32) if w is None else w.numpy()
    for j, sl in enumerate(m.slots_np):
      lo, n = int(sl['seg_begin']), int(sl['n_seg'])
      g = outs[int(sl['out_buf'])].grad.numpy().reshape(-1, int(sl['out_stride']))[:, int(sl['out_col']):int(sl['out_col']) + D]
      mine = (r >= 0) & (seg >= lo) & (seg < lo + n)
      for u in np.unique(r[mine]):
        ls = np.flatnonzero(mine & (r == u))
        want_sq += float(((g[seg[ls] - lo] * (ww[ls] * scale[seg[ls]])[:, None]).sum(0).astype(np.float64) ** 2).sum())
  assert any(s is not None for _, _, _, _, s in il._pending)       # the call really holds CSR slots
  got_sparse = float(il.sparse_grad_sqnorm())
  assert got_sparse == pytest.approx(want_sq, rel=1e-5) and want_sq > 0
  il._pending = []
  # -- the step: SGD, clipped = scale * unclipped on the table and the towers
  p0 = plain.trainer.dense_opt.flat_p.clone()
  t0 = {d: a.weight.clone() for d, a in plain.input_layer.arenas.items()}
  plain.trainer.train_step(feats, labels)
  clip.trainer.train_step(feats, labels)
  norm = float(clip.trainer.last_grad_norm)
  assert norm > 0.02
  sc = 0.02 / norm
  torch.testing.assert_close(clip.trainer.dense_opt.flat_p - p0, (plain.trainer.dense_opt.flat_p - p0) * sc, rtol=1e-4, atol=2e-7)
  for d, a in clip.input_layer.arenas.items():
    torch.testing.assert_close(a.weight - t0[d], (plain.input_layer.arenas[d].weight - t0[d]) * sc, rtol=1e-4, atol=2e-8)


def test_c5_workload_config_builds_and_trains_with_kernel_doubles(interaction_doubles):  # noqa: F811
  """bench.py --workload mmoe_c5 (BASELINE.json configs[4]): the pipeline config text and the batch generator of
  easyrec_b200.workloads at a small size - MultiTaskModel over the Cross + MLP backbone, MMoE with 4 experts (the gate
  layers are the vector-sized GEMMs of er_gemm_small), three towers bound to their labels."""
  from easyrec_b200 import layers as L, workloads
  from easyrec_b200.estimator import EasyRecEstimator
  est = EasyRecEstimator(workloads.c5_config_text(64, 5000, n_feat=6, embedding_parallel=False), device='cpu', seed=2)
  assert est.model.tower_names == ['t0', 't1', 't2'] and est.model.label_cols == [0, 1, 2]
  # each task tower is the config's `dnn { hidden_units: [64] }` on the 64-wide MMoE output, then Dense(1)
  for dnn, out in zip(est.model.tower_dnn, est.model.tower_out):
    assert isinstance(dnn, L.DNN) and [tuple(l.kernel.shape) for l in dnn.layers] == [(64, 64)]
    assert tuple(out.kernel.shape) == (64, 1)
  assert list(est.input_layer.arenas[32].tables) == ['shared'] and est.input_layer.arenas[32].n_rows == 5000
  feats, labels = workloads.c5_batch(64, 1, n_feat=6)
  assert feats['sparse_fea'].numel() == 6 * 64 and labels.shape == (64, 3)
  losses = [float(est.trainer.train_step(feats, labels)[0]) for _ in range(15)]
  assert np.isfinite(losses).all() and losses[-1] < losses[0]
  ev = est.evaluate(lambda: [(feats, labels)])
  assert sorted(k for k in ev if k.startswith('auc')) == ['auc_t0', 'auc_t1', 'auc_t2']
