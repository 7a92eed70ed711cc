"""CPU: pipeline-config loading (runtime proto2 schema, text_format) and config -> model plan.

The subset schema is cross-checked field by field against a record of the reference's protos, and the reference's
sample configs, stored under tests/golden (reference_configs.py), are parsed and built."""
import os
import sys

import pytest
import torch

from easyrec_b200 import builder
from easyrec_b200.config import config_util

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
import reference_configs  # noqa: E402

REF_CONFIGS = reference_configs.load()

MINI = b'''
model_dir: "/tmp/m"
train_config { num_steps: 7 optimizer_config { adam_optimizer { learning_rate { exponential_decay_learning_rate {
  initial_learning_rate: 0.001 decay_steps: 1000 decay_factor: 0.5 min_learning_rate: 0.00001 } } } } }
data_config { batch_size: 32 input_type: CSVInput separator: "\\t" label_fields: "label"
  input_fields { input_name: "label" input_type: FLOAT } input_fields { input_name: "F1" input_type: FLOAT }
  input_fields { input_name: "C1" input_type: INT64 } }
feature_config {
  features { input_names: "F1" feature_type: RawFeature embedding_dim: 16 min_val: 0.0 max_val: 10.0 }
  features { input_names: "C1" feature_type: IdFeature embedding_dim: 16 hash_bucket_size: 1000 unknown_future_field: 3 }
}
model_config { model_class: "DeepFM"
  feature_groups { group_name: "deep" feature_names: "F1" feature_names: "C1" wide_deep: DEEP }
  feature_groups { group_name: "wide" feature_names: "F1" feature_names: "C1" wide_deep: WIDE }
  deepfm { dnn { hidden_units: [32, 16] } final_dnn { hidden_units: [16] } l2_regularization: 1e-5 }
  embedding_regularization: 1e-5 }
'''


def test_subset_schema_parses_config_and_skips_unknown_fields():
  cfg = config_util.get_configs_from_pipeline_file(MINI)
  assert cfg.model_config.model_class == 'DeepFM'
  assert cfg.data_config.separator == '\t'
  assert [f.input_names[0] for f in config_util.get_feature_configs(cfg)] == ['F1', 'C1']
  assert cfg.model_config.deepfm.wide_output_dim == 1  # proto default
  assert list(cfg.model_config.deepfm.dnn.hidden_units) == [32, 16]
  cfg = config_util.edit_config(cfg, {'train_config.num_steps': 11, 'data_config.batch_size': 64,
                                      'model_config.deepfm.dnn.hidden_units[0]': 48})
  assert cfg.train_config.num_steps == 11 and cfg.data_config.batch_size == 64
  assert cfg.model_config.deepfm.dnn.hidden_units[0] == 48


def test_config_to_table_plan_and_schedule():
  cfg = config_util.get_configs_from_pipeline_file(MINI)
  il, model, opt = builder.build_model(cfg, 32, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  assert set(il.arenas) == {16, 1}
  assert il.arenas[16].n_rows == 1 + 1000  # raw projection row + hashed table
  assert [e[0] for e in il.group_layout['deep']] == ['F1', 'C1']  # config order
  assert opt['kind'] == 'adam_optimizer'
  lr = opt['lr_fn']
  assert abs(lr(0) - 0.001) < 1e-9 and abs(lr(999) - 0.001) < 1e-9   # staircase (proto floats are fp32)
  assert abs(lr(1000) - 0.0005) < 1e-9 and lr(10**7) == pytest.approx(0.00001)
  assert model.l2_of('dnn.layers.0.kernel', None) == pytest.approx(1e-5)
  assert model.l2_of('dnn.layers.0.bias', None) == 0.0


def test_subset_schema_is_consistent_with_reference_protos():
  sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tools'))
  import check_subset_schema
  assert check_subset_schema.check(reference_configs.record()['schema']) == []


def test_every_reference_sample_config_parses():
  """every config parses under the subset schema (unknown fields skipped), and every field it keeps is one the
  reference's complete schema parsed out of the same config (strictly, when the record was written)."""
  full = reference_configs.recorded_field_paths()
  assert len(REF_CONFIGS) > 200 and set(full) == set(REF_CONFIGS)
  for p, text in REF_CONFIGS.items():
    kept = reference_configs.field_paths(config_util.get_configs_from_pipeline_file(text))
    assert kept <= full[p], (p, sorted(kept - full[p]))


@pytest.mark.parametrize('rel', ['examples/configs/deepfm_on_criteo.config', 'samples/model_config/din_on_taobao.config',
                                 'samples/model_config/dcn_on_taobao.config', 'samples/model_config/dssm_on_taobao.config',
                                 'samples/model_config/mmoe_on_taobao.config',
                                 'samples/model_config/dcn_backbone_on_taobao.config',
                                 'samples/model_config/dlrm_backbone_on_taobao.config',
                                 'samples/model_config/mmoe_backbone_on_taobao.config',
                                 'samples/model_config/simple_multi_task_backbone_on_taobao.config',
                                 'samples/model_config/dssm_on_taobao_backbone.config',
                                 'samples/model_config/dssm_senet_on_taobao_backbone.config',
                                 'examples/configs/deepfm_backbone_on_criteo.config',
                                 'examples/configs/dlrm_backbone_on_criteo.config',
                                 'examples/configs/dlrm_senet_on_criteo.config',
                                 'examples/configs/wide_and_deep_backbone_on_movielens.config'])
def test_baseline_model_families_build_from_unmodified_reference_configs(rel, monkeypatch):
  monkeypatch.setenv('ER_PLAN_ONLY', '1')   # the plan is what is checked: the 10M-row criteo tables are not randomised
  cfg = config_util.get_configs_from_pipeline_file(REF_CONFIGS[rel])
  il, model, opt = builder.build_model(cfg, 16, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  assert sum(p.numel() for p in model.parameters()) > 1000
  assert all(a.n_rows > 0 for a in il.arenas.values())


def test_parquet_and_csv_inputs_pack_the_same_batches(tmp_path):
  """ParquetInput (scalar and list columns) and CSVInput yield the reference's packed batch form."""
  import numpy as np
  import pyarrow as pa
  import pyarrow.parquet as pq
  from easyrec_b200.input import readers
  cfg = config_util.get_configs_from_pipeline_file(MINI)
  il, model, _ = builder.build_model(cfg, 4, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  rng = np.random.default_rng(0)
  n = 9
  lab = (rng.uniform(size=n) < 0.5).astype(np.float32)
  f1 = rng.uniform(0, 10, n).astype(np.float32)
  c1 = rng.integers(0, 2**40, n).astype(np.int64)
  pq.write_table(pa.table({'label': lab, 'F1': f1, 'C1': pa.array([[int(v)] for v in c1], pa.list_(pa.int64()))}),
                 str(tmp_path / 'a.parquet'), row_group_size=5)
  with open(tmp_path / 'a.csv', 'w') as f:
    for i in range(n):
      f.write('%g\t%r\t%d\n' % (lab[i], float(f1[i]), c1[i]))
  pb = list(readers.ParquetInput(cfg, il, str(tmp_path / 'a.parquet')))
  cb = list(readers.CSVInput(cfg, il, str(tmp_path / 'a.csv')))
  assert len(pb) == len(cb) == 2   # 9 rows -> two full batches of 4, ragged tail skipped
  for (pf, pl), (cf, cl) in zip(pb, cb):
    assert torch.equal(pf['sparse_fea'], cf['sparse_fea']) and pf['sparse_fea'].dtype == torch.int64
    assert torch.allclose(pf['dense_fea'], cf['dense_fea'])
    assert torch.equal(pl, cl)
  assert torch.equal(pb[0][0]['sparse_fea'], torch.from_numpy(c1[:4]))


BACKBONE_WIRING = MINI.replace(b'model_class: "DeepFM"', b'model_class: "RankModel"').replace(
    b'deepfm { dnn { hidden_units: [32, 16] } final_dnn { hidden_units: [16] } l2_regularization: 1e-5 }',
    b'''backbone {
      blocks { name: "feats" inputs { feature_group_name: "deep" } input_layer { only_output_feature_list: true } }
      blocks { name: "halves" inputs { feature_group_name: "deep" }
               repeat { num_repeat: 2 input_fn: "lambda x, i: x[:, i * 16:(i + 1) * 16]" output_concat_axis: 1
                        keras_layer { class_name: "MLP" mlp { hidden_units: [8] } } } }
      blocks { name: "scaled" inputs { block_name: "halves" input_slice: "[:, :8]" } lambda { expression: "lambda x: x * 2.0" } }
      blocks { name: "fm" inputs { block_name: "feats" } keras_layer { class_name: "FM" fm { use_variant: true } } }
      blocks { name: "cross" inputs { feature_group_name: "deep" input_fn: "lambda x: [x, x]" }
               recurrent { num_steps: 2 fixed_input_index: 0 keras_layer { class_name: "Cross" } } }
      blocks { name: "cube" inputs { feature_group_name: "deep" } input_layer { only_output_3d_tensor: true } }
      blocks { name: "cube_sum" inputs { block_name: "cube" } lambda { expression: "lambda x: tf.reduce_sum(x, axis=1)" } }
      blocks { name: "pair" inputs { feature_group_name: "deep" } input_layer { output_2d_tensor_and_feature_list: true } }
      blocks { name: "pair_first" inputs { block_name: "pair" input_slice: "[1]" } lambda { expression: "lambda x: x[0]" } }
      concat_blocks: ["halves", "scaled", "fm", "cross", "cube_sum", "pair_first"]
      top_mlp { hidden_units: [12] }
    }
    model_params { l2_regularization: 1e-5 }''')


def test_backbone_wiring_shapes_and_parameters_without_a_gpu():
  """block inputs / input_fn / input_slice / lambda / repeat / recurrent / concat_blocks / top_mlp are resolved by a
  shape-only dry run (meta tensors): widths and parameter shapes must follow layers/backbone.py semantics."""
  cfg = config_util.get_configs_from_pipeline_file(BACKBONE_WIRING)
  il, model, opt = builder.build_model(cfg, 32, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  bb = model.backbone
  # halves: 2 x MLP(16 -> 8) concatenated = 16; scaled: 8; fm (use_variant): 16; cross: 32; cube_sum ([B,2,16] summed
  # over the features): 16; pair_first (first tensor of the pair's feature list): 16 -> concat 104 -> top_mlp 12
  assert bb.out_dim == 12 and model.output is not None
  shapes = {n: tuple(p.shape) for n, p in model.named_parameters()}
  assert shapes['backbone.mods.halves_0.layers.0.kernel'] == (16, 8)
  assert shapes['backbone.mods.halves_1.layers.0.kernel'] == (16, 8)
  assert shapes['backbone.mods.cross_0.dense.kernel'] == (32, 32) and 'backbone.mods.cross_1.dense.kernel' in shapes
  assert shapes['backbone.mods.backbone_top_mlp.layers.0.kernel'] == (104, 12)
  assert model.l2_of('backbone.mods.cross_0.dense.kernel', None) == pytest.approx(1e-5)


def test_cross_layer_variants_have_the_keras_parameter_shapes():
  """layers/keras/interaction.py:213-245: full-rank W [d, d] + bias, or U [d, p] (no bias) and V [p, d] + bias."""
  from easyrec_b200 import backbone as BB
  full = BB.Cross(12, {'diag_scale': 0.1})
  assert tuple(full.dense.kernel.shape) == (12, 12) and full.dense_u is None
  low = BB.Cross(12, {'projection_dim': 3.0})     # st_params numbers arrive as floats
  assert tuple(low.dense_u.kernel.shape) == (12, 3) and tuple(low.dense.kernel.shape) == (3, 12)
  assert not low.dense_u.bias.requires_grad and low.dense.bias.requires_grad
  with pytest.raises(ValueError):
    BB.Cross(12, {'diag_scale': -1.0})


def test_reference_criteo_config_reads_kaggle_format_lines(tmp_path):
  """examples/configs/deepfm_on_criteo.config as it is (STRING categorical fields with hash_bucket_size, FLOAT
  integer counts, empty cells) over lines in the Criteo Kaggle layout (examples/data/criteo/process_criteo_kaggle.py):
  the categorical tokens are hashed on the host - Fingerprint64(bytes) % hash_bucket_size - and an empty cell is
  the dropped id -1; the table plan takes those buckets unchanged."""
  import numpy as np
  from easyrec_b200 import _lib
  from easyrec_b200.input import readers
  from oracle import oracle as O
  cfg = config_util.get_configs_from_pipeline_file(REF_CONFIGS['examples/configs/deepfm_on_criteo.config'])
  cfg = config_util.edit_config(cfg, {'data_config.batch_size': 8})
  il, model, _ = builder.build_model(cfg, 8, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  rng = np.random.default_rng(3)
  rows = []
  for i in range(8):
    ints = ['' if rng.uniform() < 0.3 else str(rng.integers(0, 5000)) for _ in range(13)]
    cats = ['' if rng.uniform() < 0.2 else '%08x' % rng.integers(0, 2**32) for _ in range(26)]
    rows.append([str(i % 2)] + ints + cats)
  open(tmp_path / 'criteo_train_data', 'w').write(''.join('\t'.join(r) + '\n' for r in rows))
  (feats, labels), = list(readers.make_input(cfg, il, str(tmp_path / 'criteo_train_data')))
  assert labels.tolist() == [float(i % 2) for i in range(8)]
  names = il.sparse_names
  assert len(names) == 26 and all(il.features[n].bucket_mode == _lib.BUCKET_IDENTITY for n in names)
  ids = feats['sparse_fea'].reshape(26, 8).numpy()
  fields = [f.input_name for f in cfg.data_config.input_fields]
  hbs = {(fc.feature_name if fc.HasField('feature_name') else fc.input_names[0]): (fc.input_names[0], fc.hash_bucket_size)
         for fc in config_util.get_feature_configs(cfg)}
  for k, n in enumerate(names):
    col = fields.index(hbs[n][0])
    want = [O.fingerprint64(r[col]) % hbs[n][1] if r[col] != '' else -1 for r in rows]
    assert ids[k].tolist() == want, n
  assert (ids == -1).any()
  dense = feats['dense_fea'].numpy()
  for k, n in enumerate(il.raw_names):
    col = fields.index(hbs[n][0])
    assert dense[:, il.raw_cols[n][0]].tolist() == [float(r[col] or 0) for r in rows]


def test_optimizers_without_a_fused_row_rule_are_refused():
  base = b'train_config { optimizer_config { %s { learning_rate { constant_learning_rate { learning_rate: 0.1 } } %s } } }'
  ok = config_util.get_configs_from_pipeline_file(base % (b'momentum_optimizer', b'momentum_optimizer_value: 0.0'))
  assert builder.optimizer_settings(ok)['kind'] == 'momentum_optimizer' and builder.optimizer_settings(ok)['momentum'] == 0.0
  # momentum > 0 (the proto default is 0.9) keeps an accumulator per row / parameter: built (ER_OPT_MOMENTUM)
  mom = builder.optimizer_settings(config_util.get_configs_from_pipeline_file(base % (b'momentum_optimizer', b'')))
  assert mom['momentum'] == pytest.approx(0.9) and mom['beta1'] == pytest.approx(0.9)
  with pytest.raises(ValueError, match='unsupported optimizer'):
    builder.optimizer_settings(config_util.get_configs_from_pipeline_file(
        b'train_config { optimizer_config { ftrl_optimizer { } } }'))


@pytest.mark.parametrize('rel,why', [
    ('samples/model_config/multi_tower_backbone_on_taobao.config', 'losses'),           # F1-reweighted + pairwise
    ('samples/model_config/deepfm_multi_cls_on_avazu_ctr.config', None),
    ('samples/model_config/wide_and_deep_two_opti.config', None),
    ('samples/model_config/taobao_fg_ev.config', 'ev_params')])
def test_configs_that_need_unimplemented_training_semantics_are_refused(rel, why):
  cfg = config_util.get_configs_from_pipeline_file(REF_CONFIGS[rel])
  with pytest.raises((NotImplementedError, KeyError, ValueError)) as e:
    builder.build_model(cfg, 16, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  if why:
    assert why in str(e.value)


def test_the_reference_regression_sample_builds_with_its_l2_loss():
  cfg = config_util.get_configs_from_pipeline_file(REF_CONFIGS['samples/model_config/deepfm_combo_on_avazu_reg.config'])
  os.environ['ER_PLAN_ONLY'] = '1'
  try:
    _, model, _ = builder.build_model(cfg, 16, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  finally:
    del os.environ['ER_PLAN_ONLY']
  assert model.loss_type == 'L2_LOSS'


def test_scope_check_names_every_offending_field():
  cfg = config_util.get_configs_from_pipeline_file(MINI.replace(
      b'embedding_regularization: 1e-5', b'embedding_regularization: 1e-5 num_class: 3 loss_type: SOFTMAX_CROSS_ENTROPY '
      b'variational_dropout { } losses { loss_type: PAIR_WISE_LOSS }'))
  with pytest.raises(NotImplementedError) as e:
    builder.check_scope(cfg)
  for word in ('num_class 3', 'SOFTMAX_CROSS_ENTROPY', 'variational_dropout', 'PAIR_WISE_LOSS'):
    assert word in str(e.value)
  builder.check_scope(config_util.get_configs_from_pipeline_file(MINI))   # the plain config passes


def test_feature_options_that_change_the_looked_up_rows_are_refused():
  for extra, word in ((b'vocab_list: ["a", "b"]', 'vocab'), (b'kv_separator: ":"', 'kv_separator'),   # on an IdFeature
                      (b'normalizer_fn: "tf.math.log1p"', 'normalizer_fn')):
    cfg = config_util.get_configs_from_pipeline_file(
        MINI.replace(b'hash_bucket_size: 1000 unknown_future_field: 3', b'hash_bucket_size: 1000 ' + extra))
    with pytest.raises(NotImplementedError, match=word):
      builder.build_model(cfg, 8, 'cpu', cpu_generator=torch.Generator().manual_seed(0))


def test_data_options_that_change_the_batches_or_the_loss_are_refused_and_headers_are_skipped(tmp_path):
  from easyrec_b200.input import readers
  # sample weights are built for the sigmoid-CE losses (tests/test_round2_host.py), refused for the list-wise match loss
  cfg = config_util.get_configs_from_pipeline_file(MINI.replace(b'label_fields: "label"', b'label_fields: "label" sample_weight: "F1"'))
  builder.check_scope(cfg)
  cfg = config_util.get_configs_from_pipeline_file(
      MINI.replace(b'label_fields: "label"', b'label_fields: "label" sample_weight: "F1"').replace(b'model_class: "DeepFM"', b'model_class: "DSSM"'))
  with pytest.raises(NotImplementedError, match='sample_weight'):
    builder.check_scope(cfg)
  cfg = config_util.get_configs_from_pipeline_file(MINI.replace(
      b'label_fields: "label"', b'label_fields: "label" negative_sampler { input_path: "x" num_sample: 4 }'))
  il, _, _ = builder.build_model(cfg, 2, 'cpu', cpu_generator=torch.Generator().manual_seed(0))   # the model builds
  with pytest.raises(NotImplementedError, match='negative_sampler'):                                 # its input does not
    readers.make_input(cfg, il, str(tmp_path / 'x.csv'))
  cfg = config_util.get_configs_from_pipeline_file(MINI.replace(b'batch_size: 32', b'batch_size: 2 with_header: true'))
  il, _, _ = builder.build_model(cfg, 2, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  open(tmp_path / 'h.csv', 'w').write('label\tF1\tC1\n1\t2.5\t7\n0\t3.5\t8\n')
  for engine in ('native', 'python'):
    (feats, labels), = list(readers.CSVInput(cfg, il, str(tmp_path / 'h.csv'), engine=engine))
    assert labels.tolist() == [1.0, 0.0] and feats['sparse_fea'].tolist() == [7, 8]


def test_tower_options_that_are_not_implemented_are_refused():
  for new, word in ((b'dnn { hidden_units: [32, 16] activation: "softmax" }', 'activation'),):
    cfg = config_util.get_configs_from_pipeline_file(MINI.replace(b'dnn { hidden_units: [32, 16] }', new))
    with pytest.raises(NotImplementedError, match=word):
      builder.check_scope(cfg)
  # use_bn: false and dropout_ratio are built (dense + bias -> [bn] -> relu -> dropout per layer, layers/dnn.py:62-82)
  cfg = config_util.get_configs_from_pipeline_file(MINI.replace(
      b'dnn { hidden_units: [32, 16] }', b'dnn { hidden_units: [32, 16] use_bn: false dropout_ratio: [0.1, 0.1] }'))
  builder.check_scope(cfg)


def test_every_config_embedded_in_the_gpu_tests_builds_without_a_gpu():
  """the GPU tests cannot run in the build container; at least their configs must pass every host-side check
  (scope, feature plan, optimizer settings, backbone dry run) here."""
  import importlib
  import sys
  sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
  n = 0
  for mod in ('test_gpu_models', 'test_gpu_estimator'):
    m = importlib.import_module(mod)
    for name in dir(m):
      v = getattr(m, name)
      if isinstance(v, str) and 'model_config' in v:
        text = v % dict(dir='/tmp/m', kind='CSVInput') if '%(' in v else v
        cfg = config_util.get_configs_from_pipeline_file(text.encode())
        il, model, opt = builder.build_model(cfg, 16, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
        assert callable(opt['lr_fn']) and sum(p.numel() for p in model.parameters()) > 0, name
        n += 1
  assert n >= 10


def test_reference_avazu_combo_config_reads_synthetic_lines(tmp_path):
  """samples/model_config/deepfm_combo_on_avazu_ctr.config, the DeepFM config of the reference's own train tests
  (STRING hashed ids, bucketized RawFeatures, a ComboFeature): it builds unmodified and its reader turns text lines
  into the buckets the TF graph would compute - checked per feature against the scalar restatements."""
  import numpy as np
  from easyrec_b200 import _lib
  from easyrec_b200.input import readers
  from oracle import oracle as O
  cfg = config_util.get_configs_from_pipeline_file(REF_CONFIGS['samples/model_config/deepfm_combo_on_avazu_ctr.config'])
  cfg = config_util.edit_config(cfg, {'data_config.batch_size': 8})
  il, model, _ = builder.build_model(cfg, 8, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  types = builder.input_field_types(cfg)
  fields = [f.input_name for f in cfg.data_config.input_fields]
  rng = np.random.default_rng(11)
  rows = []
  for i in range(8):
    row = []
    for f in fields:
      if f in cfg.data_config.label_fields:
        row.append(str(i % 2))
      elif types[f] == 'STRING':
        row.append('' if rng.uniform() < 0.15 else '%08x' % rng.integers(0, 2**32))
      elif types[f] in ('INT32', 'INT64'):
        row.append(str(rng.integers(0, 30)))
      else:
        row.append('%.3f' % rng.uniform(0, 30))
    rows.append(row)
  sep = cfg.data_config.separator
  open(tmp_path / 'avazu.csv', 'w').write(''.join(sep.join(r) + '\n' for r in rows))
  (feats, labels), = list(readers.make_input(cfg, il, str(tmp_path / 'avazu.csv')))
  ids = feats['sparse_fea'].reshape(len(il.sparse_names), 8).numpy()
  by_name = {(fc.feature_name if fc.HasField('feature_name') else fc.input_names[0]): fc
             for fc in config_util.get_feature_configs(cfg)}
  defaults = {f.input_name: f.default_val for f in cfg.data_config.input_fields}
  kinds = set()
  for k, name in enumerate(il.sparse_names):
    fc = by_name[name]
    ftype = fc.DESCRIPTOR.fields_by_name['feature_type'].enum_type.values_by_number[fc.feature_type].name
    cols = [[r[fields.index(f)] or defaults.get(f, '') for r in rows] for f in fc.input_names]
    if ftype == 'ComboFeature':
      want = readers.cross_hash([np.array([O.fingerprint64(v) for v in col], np.uint64) for col in cols],
                                fc.hash_bucket_size).tolist()
    elif ftype == 'RawFeature':
      want = readers.bucketize_raw([float(v or 0) for v in cols[0]], fc).tolist()
    elif types[fc.input_names[0]] == 'STRING':
      want = [O.fingerprint64(v) % fc.hash_bucket_size if v != '' else -1 for v in cols[0]]
    else:
      continue          # integer ids go to the device untouched
    kinds.add(ftype)
    assert ids[k].tolist() == want, name
  assert kinds == {'ComboFeature', 'RawFeature', 'IdFeature'}


def test_in_group_sequence_feature_options_that_are_not_built_are_refused():
  """feature_groups { sequence_features { ... } } = target attention inside a plain group (built:
  tests/test_round2_host.py); its key-transform / auxiliary-history / negative-sampler variants would train
  something else and are refused."""
  for extra in (b'allow_key_transform: true', b'transform_dnn: true'):
    cfg = config_util.get_configs_from_pipeline_file(MINI.replace(
        b'feature_names: "C1" wide_deep: DEEP', b'feature_names: "C1" wide_deep: DEEP sequence_features { group_name: "s" '
        b'seq_att_map { key: "C1" hist_seq: "C1" } ' + extra + b' }'))
    with pytest.raises(NotImplementedError, match='sequence_features'):
      builder.check_scope(cfg)


def test_non_binary_task_towers_are_refused():
  import sys
  sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
  import test_gpu_models as G
  cfg = config_util.get_configs_from_pipeline_file(G.MMOE_CFG.replace('loss_type: CLASSIFICATION weight: 0.5', 'loss_type: L2_LOSS weight: 0.5').encode())
  builder.check_scope(cfg)    # a tower may be a regressor (L2_LOSS / SIGMOID_L2_LOSS on its one output)
  cfg = config_util.get_configs_from_pipeline_file(G.MMOE_CFG.replace('loss_type: CLASSIFICATION weight: 0.5', 'loss_type: PAIR_WISE_LOSS weight: 0.5').encode())
  with pytest.raises(NotImplementedError, match='PAIR_WISE_LOSS'):
    builder.check_scope(cfg)
  builder.check_scope(config_util.get_configs_from_pipeline_file(G.MMOE_CFG.encode()))


def test_no_model_or_optimizer_field_is_silently_dropped_for_configs_that_build(monkeypatch):
  """The subset schema skips fields it does not know.  For every reference sample config that BUILDS here, parse it
  with the reference's full schema as well and diff the set fields: anything under model_config, the optimizer, the
  label / input-field declarations that the subset dropped would mean training a different model in silence.
  (Control plane - export, kafka / odps inputs, extra eval metrics - may be dropped.)  The full schema's field paths
  are the ones recorded with the stored configs."""
  full = reference_configs.recorded_field_paths()
  # (only the plan matters here: the 10M-row tables of the criteo configs are allocated but not randomised)
  monkeypatch.setenv('ER_PLAN_ONLY', '1')
  guarded = ('.model_config', '.train_config.optimizer_config', '.train_config.gradient_clipping_by_norm',
             '.data_config.input_fields', '.data_config.label_fields', '.data_config.separator', '.data_config.sample_weight')
  built, dropped = 0, {}
  for p, text in REF_CONFIGS.items():
    try:
      cfg = config_util.get_configs_from_pipeline_file(text)
      builder.build_model(cfg, 4, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
    except (NotImplementedError, ValueError, KeyError, AssertionError):
      continue          # refused loudly: fine
    built += 1
    a, b = full[p], reference_configs.field_paths(cfg)
    bad = sorted(f for f in a - b if f.startswith(guarded))
    if bad:
      dropped[os.path.basename(p)] = bad
  assert built >= 40
  assert not dropped, dropped


def test_shared_names_and_name_patterns_expand_like_the_reference():
  """utils/config_util.py:81-135 auto_expand_share_feature_configs / auto_expand_names and
  feature_column/feature_group.py:46-60: a FeatureConfig with shared_names stands for one more feature per shared name
  (same settings, its own input), and `field[1-3]` in a feature group names field1, field2, field3."""
  cfg = config_util.get_configs_from_pipeline_file(b"""
data_config { batch_size: 8 input_type: CSVInput label_fields: "label" auto_expand_input_fields: true
  input_fields { input_name: "label" input_type: FLOAT } input_fields { input_name: "field1" input_type: INT64 }
  input_fields { input_name: "field2" input_type: INT64 } input_fields { input_name: "field3" input_type: INT64 } }
feature_config { features { input_names: "field1" shared_names: "field[2-3]" feature_type: IdFeature embedding_dim: 8
                            hash_bucket_size: 100 embedding_name: "shared" } }
model_config { model_class: "DeepFM"
  feature_groups { group_name: "deep" feature_names: "field[1-3]" wide_deep: DEEP }
  feature_groups { group_name: "wide" feature_names: ["field1", "field[2-3]"] wide_deep: WIDE }
  deepfm { dnn { hidden_units: [8] } final_dnn { hidden_units: [4] } } }
""")
  feats = config_util.get_feature_configs(cfg)
  assert [list(f.input_names) for f in feats] == [['field1'], ['field2'], ['field3']]
  assert all(len(f.shared_names) == 0 and f.embedding_name == 'shared' and f.hash_bucket_size == 100 for f in feats)
  assert list(cfg.model_config.feature_groups[0].feature_names) == ['field1', 'field2', 'field3']
  assert list(cfg.model_config.feature_groups[1].feature_names) == ['field1', 'field2', 'field3']
  assert config_util.auto_expand_names('c[9-11]') == ['c9', 'c10', 'c11'] and config_util.auto_expand_names('plain') == ['plain']
  il, _, _ = builder.build_model(cfg, 8, 'cpu', cpu_generator=torch.Generator().manual_seed(0))
  assert il.sparse_names == ['field1', 'field2', 'field3'] and list(il.arenas[8].tables) == ['shared']
