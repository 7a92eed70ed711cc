"""Synthetic workloads of BASELINE.json `configs` (shapes from SURVEY.md section 8d).

C2 = DeepFM Criteo-shape: 13 RawFeature (embedding_dim 16, min/max of
examples/configs/deepfm_on_criteo.config:241-330) + 26 IdFeature hashed into ONE shared
table of V rows (embedding_name 'embedding', as samples/model_config/
dlrm_on_criteo_parquet_ep.config:319-324), emb 16, batch 8192, DNN [256,128,64] +
final_dnn [256,128,64], wide_output_dim 1.
"""
import collections

import numpy as np
import torch

from easyrec_b200 import _lib
from easyrec_b200 import input_layer as IL
from easyrec_b200.model.deepfm import DeepFM

CRITEO_MAX = [5775.0, 257675.0, 65535.0, 969.0, 23159456.0, 431037.0, 56311.0, 6047.0, 29019.0,
              46.0, 231.0, 4008.0, 7393.0]
CRITEO_MIN = [0.0, -3.0] + [0.0] * 11


def criteo_features(vocab, emb_dim=16, shared_table=True):
  feats = []
  for i in range(13):
    feats.append(IL.raw_feature('F%d' % (i + 1), emb_dim, CRITEO_MIN[i], CRITEO_MAX[i]))
  per = vocab if shared_table else max(vocab // 26, 1)
  for i in range(26):
    feats.append(IL.id_feature('C%d' % (i + 1), emb_dim, hash_bucket_size=per,
                               embedding_name='embedding' if shared_table else ''))
  names = [f.name for f in feats]
  groups = collections.OrderedDict([('deep', dict(features=names, wide=False)),
                                    ('wide', dict(features=names, wide=True))])
  return feats, groups


def build_deepfm_criteo(batch_size, vocab, device, emb_dim=16, shared_table=True, seed=20240,
                        emb_opt=_lib.OPT_ADAGRAD, dnn=(256, 128, 64), final=(256, 128, 64),
                        l2_reg=1e-5, emb_reg=1e-5):
  feats, groups = criteo_features(vocab, emb_dim, shared_table)
  gen = torch.Generator(device=device).manual_seed(seed)
  il = IL.InputLayer(feats, groups, batch_size, device, wide_output_dim=1,
                     embedding_optimizer=emb_opt, generator=gen)
  cpu_gen = torch.Generator().manual_seed(seed)
  model = DeepFM(il, list(dnn), list(final), l2_reg=l2_reg, embedding_reg=emb_reg,
                 generator=cpu_gen).to(device)
  return il, model


def criteo_batch(batch_size, seed, zipf_alpha=1.05, uniform=False):
  """Host-side synthetic batch: ids int64 [26*B] feature-major, dense fp32 [B,13], labels [B].

  ids ~ Zipf(alpha) over [0, 2^40) (uniform variant: worst case, U ~= L); dense ~ lognormal
  clipped to the config's [min, max]; labels ~ Bernoulli(0.25)."""
  rng = np.random.default_rng(seed)
  n = 26 * batch_size
  if uniform:
    ids = rng.integers(0, 2**40, n, dtype=np.int64)
  else:
    ids = (rng.zipf(zipf_alpha, n).astype(np.int64) - 1) % (2**40)
    # decorrelate slots: each slot sees its own permutation of the id space
    ids = ids * 26 + np.repeat(np.arange(26, dtype=np.int64), batch_size)
  dense = rng.lognormal(1.0, 2.0, (batch_size, 13)).astype(np.float32)
  dense = np.minimum(dense, np.array(CRITEO_MAX, np.float32))
  labels = (rng.uniform(size=batch_size) < 0.25).astype(np.float32)
  return ids, dense, labels


# ---- the same workloads as pipeline configs (protobuf text): what EasyRecEstimator is handed ---------------------
def c2_config_text(vocab, batch_size, optimizer='adagrad_optimizer', lr=0.01, input_type='CSVInput', model_dir='/tmp/er_c2',
                   dnn=(256, 128, 64), final=(256, 128, 64)):
  """C2 as a pipeline config in the reference's schema: the feature / model sections of
  examples/configs/deepfm_on_criteo.config with the 26 id features sharing one `vocab`-row table (embedding_name
  "embedding", as samples/model_config/dlrm_on_criteo_parquet_ep.config:319-324).  Columns: label, f1..f13, c1..c26
  (TSV) / is_click, f1..f13, c1..c26 (Parquet, tools/criteo/convert_data.py:29-39)."""
  label = 'is_click' if input_type.startswith('Parquet') else 'label'
  fields = ['  input_fields { input_name: "%s" input_type: FLOAT }' % label]
  feats = []
  for i in range(13):
    fields.append('  input_fields { input_name: "f%d" input_type: FLOAT }' % (i + 1))
    feats.append('  features { input_names: "f%d" feature_type: RawFeature embedding_dim: 16 min_val: %r max_val: %r }'
                 % (i + 1, CRITEO_MIN[i], CRITEO_MAX[i]))
  for i in range(26):
    fields.append('  input_fields { input_name: "c%d" input_type: INT64 }' % (i + 1))
    feats.append('  features { input_names: "c%d" feature_type: IdFeature embedding_dim: 16 hash_bucket_size: %d '
                 'embedding_name: "embedding" }' % (i + 1, vocab))
  names = ', '.join('"f%d"' % (i + 1) for i in range(13)) + ', ' + ', '.join('"c%d"' % (i + 1) for i in range(26))
  text = '\n'.join([
      'model_dir: "%s"' % model_dir,
      'train_config { log_step_count_steps: 1000000',
      '  optimizer_config { %s { learning_rate { constant_learning_rate { learning_rate: %r } } } } }' % (optimizer, lr),
      'data_config { batch_size: %d input_type: %s separator: "\\t" label_fields: "%s"' % (batch_size, input_type, label),
      '\n'.join(fields) + ' }',
      'feature_config {', '\n'.join(feats) + ' }',
      'model_config { model_class: "DeepFM"',
      '  feature_groups { group_name: "deep" feature_names: [%s] wide_deep: DEEP }' % names,
      '  feature_groups { group_name: "wide" feature_names: [%s] wide_deep: WIDE }' % names,
      '  deepfm { dnn { hidden_units: %s } final_dnn { hidden_units: %s } l2_regularization: 1e-5 }' % (list(dnn), list(final)),
      '  embedding_regularization: 1e-5 }', ''])
  return text.encode()


def c3_config_text(batch_size=4096, item_vocab=1_000_000, seq_len=50, optimizer='adagrad_optimizer', lr=0.01):
  """C3: DIN, the shape of samples/model_config/din_on_taobao.config - user / item towers, two behaviour sequences
  (item ids over `item_vocab`, categories over 10K) attended by their keys, attention MLP [128, 64, 32, 1]
  (layers/sequence_feature_layer.py:158-165), final DNN [256, 128, 64]."""
  seq = 'feature_type: SequenceFeature embedding_dim: 16 max_seq_len: %d separator: "|"' % seq_len
  text = '\n'.join([
      'train_config { log_step_count_steps: 1000000',
      '  optimizer_config { %s { learning_rate { constant_learning_rate { learning_rate: %r } } } } }' % (optimizer, lr),
      'data_config { batch_size: %d input_type: DummyInput label_fields: "clk"' % batch_size,
      '  input_fields { input_name: "clk" input_type: FLOAT } input_fields { input_name: "user_id" input_type: INT64 }',
      '  input_fields { input_name: "age" input_type: INT64 } input_fields { input_name: "item_id" input_type: INT64 }',
      '  input_fields { input_name: "cate_id" input_type: INT64 } input_fields { input_name: "price" input_type: FLOAT }',
      '  input_fields { input_name: "hist_items" input_type: STRING } input_fields { input_name: "hist_cates" input_type: STRING } }',
      'feature_config {',
      '  features { input_names: "user_id" feature_type: IdFeature embedding_dim: 16 hash_bucket_size: 1000000 }',
      '  features { input_names: "age" feature_type: IdFeature embedding_dim: 16 num_buckets: 100 }',
      '  features { input_names: "item_id" feature_type: IdFeature embedding_dim: 16 hash_bucket_size: %d }' % item_vocab,
      '  features { input_names: "cate_id" feature_type: IdFeature embedding_dim: 16 hash_bucket_size: 10000 }',
      '  features { input_names: "price" feature_type: RawFeature embedding_dim: 16 min_val: 0.0 max_val: 1.0 }',
      '  features { input_names: "hist_items" hash_bucket_size: %d %s }' % (item_vocab, seq),
      '  features { input_names: "hist_cates" hash_bucket_size: 10000 %s } }' % seq,
      'model_config { model_class: "MultiTowerDIN"',
      '  feature_groups { group_name: "user" feature_names: ["user_id", "age"] wide_deep: DEEP }',
      '  feature_groups { group_name: "item" feature_names: ["item_id", "cate_id", "price"] wide_deep: DEEP }',
      '  seq_att_groups { group_name: "din" seq_att_map { key: "item_id" hist_seq: "hist_items" }',
      '                   seq_att_map { key: "cate_id" hist_seq: "hist_cates" } }',
      '  multi_tower { towers { input: "user" dnn { hidden_units: [128, 64] } } towers { input: "item" dnn { hidden_units: [128, 64] } }',
      '                din_towers { input: "din" dnn { hidden_units: [128, 64, 32, 1] } } final_dnn { hidden_units: [256, 128, 64] }',
      '                l2_regularization: 1e-5 }',
      '  embedding_regularization: 1e-5 }', ''])
  return text.encode()


def c3_batch(batch_size, seq_len, seed, vocab, cate_buckets=10000, zipf_alpha=1.05):
  """host batch in c3_config_text's InputLayer form: ids feature-major (user_id, age, item_id, cate_id), price,
  histories padded to seq_len with lengths ~ U[1, seq_len], label Bernoulli(0.25).

  The two histories are STRING fields with a hash_bucket_size in the config, so - like the file readers
  (input/readers.py) - the batch carries them host-hashed: Fingerprint64(decimal text) % buckets, the same
  rule the device applies to the INT64 id fields."""
  from .input.readers import fingerprint_i64
  rng = np.random.default_rng(seed)
  B = batch_size

  def z(n):
    return (rng.zipf(zipf_alpha, n).astype(np.int64) - 1) % (2**40)
  ids = np.concatenate([z(B), rng.integers(0, 100, B), z(B), z(B) % 100000]).astype(np.int64)
  dense = rng.uniform(0, 1, (B, 1)).astype(np.float32)
  lens = rng.integers(1, seq_len + 1, B).astype(np.int32)

  def hashed(raw, buckets):
    return (fingerprint_i64(raw) % np.uint64(buckets)).astype(np.int64).reshape(B, seq_len)
  seq = {'hist_items': (torch.from_numpy(hashed(z(B * seq_len), vocab)), torch.from_numpy(lens)),
         'hist_cates': (torch.from_numpy(hashed(z(B * seq_len) % 100000, cate_buckets)), torch.from_numpy(lens.copy()))}
  labels = (rng.uniform(size=B) < 0.25).astype(np.float32)
  return {'sparse_fea': torch.from_numpy(ids), 'dense_fea': torch.from_numpy(dense), 'seq_fea': seq}, torch.from_numpy(labels)


def write_c2_files(prefix, n_batches, batch_size, seed=20240, uniform=False):
  """The C2 batches of `criteo_batch` as a TSV and a Parquet file (same rows): returns (tsv path, parquet path)."""
  import pyarrow as pa
  import pyarrow.parquet as pq
  ids, dense, labels = [], [], []
  for i in range(n_batches):
    x, d, l = criteo_batch(batch_size, seed + i, uniform=uniform)
    ids.append(x.reshape(26, batch_size).T)
    dense.append(d)
    labels.append(l)
  ids, dense, labels = np.concatenate(ids), np.concatenate(dense), np.concatenate(labels)
  cols = [labels.astype(np.int64).astype(str)] + [np.char.mod('%.9g', dense[:, j]) for j in range(13)]
  cols += [ids[:, j].astype(str) for j in range(26)]
  lines = cols[0]
  for c in cols[1:]:
    lines = np.char.add(np.char.add(lines, '\t'), c)
  with open(prefix + '.tsv', 'w') as f:
    f.write('\n'.join(lines.tolist()) + '\n')
  tab = {'is_click': labels.astype(np.int32)}
  for j in range(13):
    tab['f%d' % (j + 1)] = dense[:, j].astype(np.float32)
  for j in range(26):
    tab['c%d' % (j + 1)] = ids[:, j].astype(np.int64)
  pq.write_table(pa.table(tab), prefix + '.parquet', row_group_size=batch_size)
  return prefix + '.tsv', prefix + '.parquet'


def c4_config_text(batch_size=4096, item_vocab=200_000_000, user_vocab=10_000_000, emb_dim=16, lr=0.01,
                   embedding_parallel=True):
  """C4 of BASELINE.json as a pipeline config: DSSM two towers (samples/model_config/dssm_on_taobao.config's shape:
  user side = user id + 4 profile ids, item side = item id + category + brand + price), cosine similarity with
  in-batch negatives (loss_type SOFTMAX_CROSS_ENTROPY, model/dssm.py + match_model.py:95-165), the item table
  row-sharded (train_distribute: EmbeddingParallelStrategy)."""
  return ('''
train_config { log_step_count_steps: 1000000 %s
  optimizer_config { adagrad_optimizer { learning_rate { constant_learning_rate { learning_rate: %g } } } } }
data_config { batch_size: %d input_type: DummyInput label_fields: "clk"
  input_fields { input_name: "clk" input_type: FLOAT } input_fields { input_name: "user_id" input_type: INT64 }
  input_fields { input_name: "age" input_type: INT64 } input_fields { input_name: "gender" input_type: INT64 }
  input_fields { input_name: "city" input_type: INT64 } input_fields { input_name: "level" input_type: INT64 }
  input_fields { input_name: "item_id" input_type: INT64 } input_fields { input_name: "cate_id" input_type: INT64 }
  input_fields { input_name: "brand" input_type: INT64 } input_fields { input_name: "price" input_type: FLOAT } }
feature_config {
  features { input_names: "user_id" feature_type: IdFeature embedding_dim: %d hash_bucket_size: %d }
  features { input_names: "age" feature_type: IdFeature embedding_dim: %d num_buckets: 100 }
  features { input_names: "gender" feature_type: IdFeature embedding_dim: %d num_buckets: 3 }
  features { input_names: "city" feature_type: IdFeature embedding_dim: %d hash_bucket_size: 10000 }
  features { input_names: "level" feature_type: IdFeature embedding_dim: %d num_buckets: 10 }
  features { input_names: "item_id" feature_type: IdFeature embedding_dim: %d hash_bucket_size: %d }
  features { input_names: "cate_id" feature_type: IdFeature embedding_dim: %d hash_bucket_size: 10000 }
  features { input_names: "brand" feature_type: IdFeature embedding_dim: %d hash_bucket_size: 1000000 }
  features { input_names: "price" feature_type: RawFeature embedding_dim: %d min_val: 0.0 max_val: 1.0 } }
model_config { model_class: "DSSM"
  feature_groups { group_name: "user" feature_names: ["user_id", "age", "gender", "city", "level"] wide_deep: DEEP }
  feature_groups { group_name: "item" feature_names: ["item_id", "cate_id", "brand", "price"] wide_deep: DEEP }
  dssm { user_tower { id: "user_id" dnn { hidden_units: [256, 128, 64, 32] } }
         item_tower { id: "item_id" dnn { hidden_units: [256, 128, 64, 32] } }
         simi_func: COSINE temperature: 0.05 scale_simi: true l2_regularization: 1e-6 }
  loss_type: SOFTMAX_CROSS_ENTROPY embedding_regularization: 5e-5 }
''' % ('train_distribute: EmbeddingParallelStrategy' if embedding_parallel else '', lr, batch_size,
       emb_dim, user_vocab, emb_dim, emb_dim, emb_dim, emb_dim, emb_dim, item_vocab, emb_dim, emb_dim, emb_dim)).encode()


def c4_batch(batch_size, seed, zipf_alpha=1.05):
  """host batch in c4_config_text's InputLayer form: ids feature-major (user_id, age, gender, city, level, item_id,
  cate_id, brand), price; the label column is ignored by the in-batch softmax (every row is its own positive)."""
  rng = np.random.default_rng(seed)
  B = batch_size

  def z(n):
    return (rng.zipf(zipf_alpha, n).astype(np.int64) - 1) % (2**40)
  item = z(B)
  ids = np.concatenate([z(B), rng.integers(0, 100, B), rng.integers(0, 3, B), z(B) % 100000, rng.integers(0, 10, B),
                        item, z(B) % 100000, z(B) % 10_000_000]).astype(np.int64)
  dense = rng.uniform(0, 1, (B, 1)).astype(np.float32)
  return {'sparse_fea': torch.from_numpy(ids), 'dense_fea': torch.from_numpy(dense),
          'item_ids': torch.from_numpy(item.copy())}, torch.ones(B, dtype=torch.float32)


def c5_config_text(batch_size=16384, vocab=100_000_000, n_feat=40, emb_dim=32, lr=0.02, embedding_parallel=True):
  """C5 of BASELINE.json as a pipeline config: 3-task MMoE over a DCN-style backbone (deep MLP next to three Cross
  layers on the same input, samples/model_config/dcn_backbone_on_taobao.config + mmoe_backbone_on_taobao.config), `n_feat`
  id slots over ONE shared `vocab` x `emb_dim` table (as dlrm_on_criteo_parquet_ep.config:319-324 shares its table),
  row-sharded (train_distribute: EmbeddingParallelStrategy), three binary labels."""
  feats = '\n'.join('  features { input_names: "c%d" feature_type: IdFeature embedding_dim: %d hash_bucket_size: %d '
                    'embedding_name: "shared" }' % (i, emb_dim, vocab) for i in range(n_feat))
  fields = ' '.join('input_fields { input_name: "c%d" input_type: INT64 }' % i for i in range(n_feat))
  names = ', '.join('"c%d"' % i for i in range(n_feat))
  return ('''
train_config { log_step_count_steps: 1000000 %s
  optimizer_config { adagrad_optimizer { learning_rate { constant_learning_rate { learning_rate: %g } } } } }
data_config { batch_size: %d input_type: DummyInput label_fields: ["l0", "l1", "l2"]
  input_fields { input_name: "l0" input_type: FLOAT } input_fields { input_name: "l1" input_type: FLOAT }
  input_fields { input_name: "l2" input_type: FLOAT } %s }
feature_config {
%s
}
model_config { model_class: "MultiTaskModel"
  feature_groups { group_name: "all" feature_names: [%s] wide_deep: DEEP }
  backbone {
    blocks { name: "deep" inputs { feature_group_name: "all" } keras_layer { class_name: "MLP" mlp { hidden_units: [256, 128] } } }
    blocks { name: "cross" inputs { feature_group_name: "all" input_fn: "lambda x: [x, x]" }
             recurrent { num_steps: 3 fixed_input_index: 0 keras_layer { class_name: "Cross" } } }
    blocks { name: "both" inputs { block_name: "deep" } inputs { block_name: "cross" } merge_inputs_into_list: true
             keras_layer { class_name: "Concatenate" } }
    blocks { name: "mmoe" inputs { block_name: "both" }
             keras_layer { class_name: "MMoE" mmoe { num_task: 3 num_expert: 4 expert_mlp { hidden_units: [128, 64] } } } }
  }
  model_params { l2_regularization: 1e-6
    task_towers { tower_name: "t0" label_name: "l0" dnn { hidden_units: [64] } }
    task_towers { tower_name: "t1" label_name: "l1" dnn { hidden_units: [64] } }
    task_towers { tower_name: "t2" label_name: "l2" dnn { hidden_units: [64] } } }
  embedding_regularization: 1e-6 }
''' % ('train_distribute: EmbeddingParallelStrategy' if embedding_parallel else '', lr, batch_size, fields, feats,
       names)).encode()


def c5_batch(batch_size, seed, n_feat=40, zipf_alpha=1.05):
  """host batch in c5_config_text's InputLayer form: `n_feat` id columns feature-major, three Bernoulli labels"""
  rng = np.random.default_rng(seed)
  ids = (rng.zipf(zipf_alpha, n_feat * batch_size).astype(np.int64) - 1) % (2**40)
  labels = (rng.uniform(size=(batch_size, 3)) < 0.25).astype(np.float32)
  return {'sparse_fea': torch.from_numpy(ids)}, torch.from_numpy(labels)
