"""GPU parity through the layer glue (not only kernel by kernel): TensorFlow's SafeEmbeddingLookupSparseTest case
table (invalid ids, empty rows, non-positive weights under mean) replayed on the KERNEL through a TagFeature group of
InputLayer - lookup and the backward row update.

The training steps of the BASELINE.json configs C3, C4 and C5 at config shape are compared with float64 in
test_gpu_config_step_parity.py.
"""
import json
import os

import numpy as np
import pytest
import torch

from easyrec_b200 import builder
from easyrec_b200.config import config_util

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
KATS = json.load(open(os.path.join(os.path.dirname(__file__), 'golden', 'reference_kats.json')))


TAG_CFG = b'''
train_config { optimizer_config { adagrad_optimizer { learning_rate { constant_learning_rate { learning_rate: 0.1 } } } } }
data_config { batch_size: 5 input_type: CSVInput separator: "," label_fields: "label"
  input_fields { input_name: "label" input_type: FLOAT } input_fields { input_name: "t" input_type: STRING }
  input_fields { input_name: "u" input_type: INT64 } }
feature_config {
  features { input_names: "t" feature_type: TagFeature embedding_dim: 4 num_buckets: 5 separator: "|" kv_separator: ":" combiner: "mean" }
  features { input_names: "u" feature_type: IdFeature embedding_dim: 4 num_buckets: 7 } }
model_config { model_class: "DeepFM"
  feature_groups { group_name: "deep" feature_names: ["t", "u"] wide_deep: DEEP }
  feature_groups { group_name: "wide" feature_names: ["t", "u"] wide_deep: WIDE }
  deepfm { dnn { hidden_units: [8] } final_dnn { hidden_units: [4] } } }
'''


@pytest.mark.parametrize('weighted', [True, False])
def test_safe_lookup_case_table_through_a_tag_group_on_the_gpu(weighted):
  """embedding_ops_test.py SafeEmbeddingLookupSparseTest: row 0 = valid ids + one invalid id, weighted mean; row 1 all
  invalid; row 2 empty; row 3 a single id; row 4 only non-positive weights - through InputLayer.lookup (CSR tag slot,
  mean combiner, kv weights) and back through the fused row update."""
  k = KATS['safe_embedding_lookup_sparse']
  cfg = config_util.get_configs_from_pipeline_file(TAG_CFG)
  il, model, _ = builder.build_model(cfg, 5, DEV, generator=torch.Generator(device=DEV).manual_seed(2),
                                     cpu_generator=torch.Generator().manual_seed(2))
  n_rows = k['dense_shape'][0]
  lens = np.bincount([i[0] for i in k['indices']], minlength=n_rows).astype(np.int32)
  ids = torch.tensor(k['ids'], dtype=torch.int64, device=DEV)
  w = torch.tensor(k['weights'], dtype=torch.float32, device=DEV) if weighted else None
  feats = {'sparse_fea': torch.arange(5, dtype=torch.int64, device=DEV),
           'tag_fea': {'t': (ids, torch.from_numpy(lens).to(DEV), w)}}
  a = il.arenas[4]
  off, _, _ = a.tables['t_embedding']
  e = a.weight[off:off + 5].detach().cpu().numpy().copy()
  groups = il.lookup(feats)
  deep, per_feature = groups['deep']
  got = per_feature[0].detach().cpu().numpy()
  for r, spec in enumerate(k['expected_weighted' if weighted else 'expected_no_weights']):
    want = np.zeros(4, np.float32) if spec is None else sum(wt * e[i] for i, wt in spec['terms']) / spec['div']
    np.testing.assert_allclose(got[r], want, rtol=1e-6, atol=1e-6)
  # backward: only ids that contributed move, by the mean-combiner coefficient w_i / sum(w)
  gsum = torch.zeros_like(deep)
  gsum[:, :4] = 1.0
  before = a.weight.detach().clone()
  deep.backward(gsum)
  il.set_optimizer_step(0.1, 0)
  il.backward_update()
  moved = (a.weight[off:off + 5] != before[off:off + 5]).any(1).cpu().numpy()
  used = sorted({i for spec in k['expected_weighted' if weighted else 'expected_no_weights'] if spec for i, _ in spec['terms']})
  assert sorted(np.flatnonzero(moved).tolist()) == used
