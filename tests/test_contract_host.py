"""CPU (kernel doubles): the reference's Python contract on the fused path.

  * `EasyRecModel.create_class(model_class)` + the reference constructor arguments + build_predict_graph /
    build_loss_graph / build_metric_graph / get_outputs (model/easy_rec_model.py:51-183, utils/load_class.py:203-222):
    one model is driven ONLY through those names and trains;
  * `InputLayer.__call__(features, group_name, is_combine, is_dict)` (layers/input_layer.py:245-278);
  * model_class "DLRM" (model/dlrm.py:38-73): the reference's own EmbeddingParallel sample config builds, and the
    interaction equals the einsum / upper-triangle restatement of the reference body."""
import os
import sys

import numpy as np
import pytest
import torch

from easyrec_b200 import builder, trainer as T
from easyrec_b200.config import config_util
from easyrec_b200.input import readers
from easyrec_b200.model.easy_rec_model import EasyRecModel
from test_input_layer_host import oracle_kernels  # noqa: F401  (fixture)
from test_model_host import dense_kernels, interaction_doubles  # noqa: F401  (fixtures)

CFG = b'''
train_config { optimizer_config { adagrad_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.1 } } } } }
eval_config { metrics_set { auc {} } }
data_config { batch_size: 32 input_type: CSVInput separator: "," label_fields: "label"
  input_fields { input_name: "label" input_type: FLOAT } input_fields { input_name: "u" input_type: INT64 }
  input_fields { input_name: "i" input_type: INT64 } input_fields { input_name: "x" input_type: FLOAT }
  input_fields { input_name: "y" input_type: FLOAT } }
feature_config {
  features { input_names: "u" feature_type: IdFeature embedding_dim: 8 num_buckets: 20 }
  features { input_names: "i" feature_type: IdFeature embedding_dim: 8 num_buckets: 30 }
  features { input_names: "x" feature_type: RawFeature }
  features { input_names: "y" feature_type: RawFeature } }
model_config { model_class: "DLRM"
  feature_groups { group_name: "sparse" feature_names: ["u", "i"] wide_deep: DEEP }
  feature_groups { group_name: "dense" feature_names: ["x", "y"] wide_deep: DEEP }
  dlrm { bot_dnn { hidden_units: [16, 8] } top_dnn { hidden_units: [16, 8] } arch_interaction_itself: %s
         arch_with_dense_feature: %s l2_regularization: 1e-5 }
  embedding_regularization: 1e-5 }
'''


def _batch(B=32, seed=0):
  rng = np.random.default_rng(seed)
  u, i = rng.integers(0, 20, B), rng.integers(0, 30, B)
  feats = {'sparse_fea': torch.from_numpy(np.concatenate([u, i]).astype(np.int64)),
           'dense_fea': torch.from_numpy(rng.uniform(0, 1, (B, 2)).astype(np.float32))}
  labels = torch.from_numpy(((u + i) % 2 == 0).astype(np.float32))
  return feats, labels


def test_a_model_driven_only_through_the_reference_contract(interaction_doubles):  # noqa: F811
  cfg = config_util.get_configs_from_pipeline_file(CFG % (b'false', b'false'))
  il, _, opt = builder.build_model(cfg, 32, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  feats, labels = _batch()
  cls = EasyRecModel.create_class(cfg.model_config.model_class)
  assert cls.__name__ == 'DLRM' and issubclass(cls, EasyRecModel)
  model = cls(cfg.model_config, config_util.get_feature_configs(cfg), feats, labels, is_training=True, input_layer=il,
              generator=torch.Generator().manual_seed(1))
  pred = model.build_predict_graph()
  assert sorted(pred) == ['logits', 'probs'] and tuple(pred['probs'].shape) == (32,)
  assert torch.allclose(pred['probs'], torch.sigmoid(pred['logits']))
  losses = model.build_loss_graph()
  assert 'cross_entropy_loss' in losses and 'regularization_loss' in losses
  total = sum(losses.values())
  metrics = model.build_metric_graph(cfg.eval_config)
  assert 0.0 <= metrics['auc'] <= 1.0 and model.get_outputs() == ['probs', 'logits']
  # the same object trains under the Trainer (it is the registered torch module underneath)
  tr = T.Trainer(model, il, 'adagrad', lr_fn=opt['lr_fn'])
  first = float(tr.train_step(feats, labels)[0])
  # (the trainer's loss adds the dense-kernel l2 term, evaluated inside the fused dense optimizer launch)
  assert first - float(tr.dense_opt.reg_loss[0]) == pytest.approx(float(total), rel=1e-5)
  for _ in range(30):
    last = float(tr.train_step(feats, labels)[0])
  assert last < first - 0.05
  model.set_inputs(feats, labels, is_training=False)
  model.build_predict_graph()
  assert model.build_metric_graph(cfg.eval_config)['auc'] > 0.8
  with pytest.raises(KeyError):
    EasyRecModel.create_class('NoSuchModel')


def test_input_layer_call_form(oracle_kernels):  # noqa: F811
  cfg = config_util.get_configs_from_pipeline_file(CFG % (b'false', b'false'))
  il, _, _ = builder.build_model(cfg, 32, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  feats, _ = _batch()
  concat, flist = il(feats, 'sparse')
  assert tuple(concat.shape)[0] == 32 and [tuple(f.shape) for f in flist] == [(32, 8), (32, 8)]
  assert torch.equal(concat[:, :16], torch.cat(flist, dim=1))
  concat2, flist2, by_name = il(feats, 'sparse', is_dict=True)
  assert concat2 is concat and sorted(by_name) == ['i', 'u'] and by_name['u'] is flist2[0]   # one lookup per batch
  dense, dlist = il(feats, 'dense')
  assert tuple(dense.shape) == (32, 2) and len(dlist) == 2
  seq, plain, plist = il(feats, 'sparse', is_combine=False)
  assert seq == [] and plain is concat and len(plist) == 2
  with pytest.raises(AssertionError, match='invalid group_name'):
    il(feats, 'nope')
  assert il.has_group('dense') and not il.has_group('nope')


@pytest.mark.parametrize('itself,with_dense', [(False, False), (True, True)])
def test_dlrm_interaction_matches_the_reference_body(itself, with_dense, interaction_doubles):  # noqa: F811
  """model/dlrm.py:46-66 restated in numpy: einsum('bne,bme->bnm'), rows i take columns i+offset.., concat with the
  sparse features (and the dense output)."""
  cfg = config_util.get_configs_from_pipeline_file(CFG % (str(itself).lower().encode(), str(with_dense).lower().encode()))
  il, model, _ = builder.build_model(cfg, 32, 'cpu', cpu_generator=torch.Generator().manual_seed(3))
  feats, _ = _batch(seed=2)
  captured = {}

  def hook(m, inp, out):
    captured['x'] = inp[0].detach().clone()
  model.top_dnn.register_forward_hook(hook)
  model.eval()
  model(feats)
  g = il.lookup(feats)
  sparse = [t.detach().numpy() for t in g['sparse'][1]]
  dense_fea = model.bot_dnn(g['dense'][0].contiguous()).detach().numpy()
  all_feas = np.stack([dense_fea] + sparse, axis=1)
  inter = np.einsum('bne,bme->bnm', all_feas, all_feas)
  off = 0 if itself else 1
  upper = np.concatenate([inter[:, i, i + off:] for i in range(all_feas.shape[1])], axis=1)
  want = np.concatenate([upper] + sparse + ([dense_fea] if with_dense else []), axis=1)
  np.testing.assert_allclose(captured['x'].numpy(), want, rtol=1e-5, atol=1e-6)


def test_reference_dlrm_ep_config_builds(monkeypatch):
  """the reference's own EmbeddingParallel test config (model_class DLRM over the packed Parquet criteo form)"""
  sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
  import reference_configs
  cfg = config_util.get_configs_from_pipeline_file(
      reference_configs.load()['samples/model_config/dlrm_on_criteo_parquet_ep.config'])
  monkeypatch.setenv('ER_PLAN_ONLY', '1')   # (a 10M-row table: the plan is what is checked)
  il, model, opt = builder.build_model(cfg, 64, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  assert type(model).__name__ == 'DLRM' and builder.embedding_parallel(cfg)
  assert len(model.sparse_dims) == 26 and model.n_fea == 27
