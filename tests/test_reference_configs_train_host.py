"""CPU, kernel doubles: every reference sample config that the scope check accepts (and whose tables are small enough to
materialise here) is built through EasyRecEstimator, trains two steps on a DummyInput batch and evaluates its
eval_config.metrics_set - the reference's own train_eval tests are exit-code smoke runs over the same files
(easy_rec/python/test/train_eval_test.py).  The configs are the ones stored under tests/golden (reference_configs.py)."""
import os
import sys

import numpy as np
import pytest
import torch

import host_doubles
from easyrec_b200 import builder
from easyrec_b200.config import config_util
from easyrec_b200.input import readers

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
import reference_configs  # noqa: E402


@pytest.mark.timeout(900)
def test_every_accepted_small_reference_config_trains_and_evaluates(monkeypatch):
  from easyrec_b200.estimator import EasyRecEstimator
  host_doubles.install_all(monkeypatch.setattr)
  trained, failed = [], {}
  for p, text in reference_configs.load().items():
    try:
      cfg = config_util.get_configs_from_pipeline_file(text)
      builder.check_scope(cfg)
      builder.feature_specs(cfg)
    except Exception:
      continue                    # refused configs are test_config.py's subject
    rows = sum(max(fc.hash_bucket_size, fc.num_buckets, 1) for fc in config_util.get_feature_configs(cfg))
    if rows > 2_000_000:
      continue
    name = os.path.basename(p)
    try:
      est = EasyRecEstimator(cfg, device='cpu', seed=1, batch_size=8)
    except (NotImplementedError, KeyError, AssertionError, ValueError):
      continue                    # refused at build time (model class, block type, ...)
    try:
      feats, labels = readers.DummyInput(est.input_layer, n_labels=max(1, len(cfg.data_config.label_fields)), seed=3).batch()
      l0, _ = est.trainer.train_step(feats, labels)
      l1, _ = est.trainer.train_step(feats, labels)
      assert np.isfinite(float(l0)) and np.isfinite(float(l1))
      ev = est.evaluate(lambda: [(feats, labels)])
      assert all(np.isfinite(v) or np.isnan(v) for v in ev.values())
      trained.append(name)
    except Exception as e:   # noqa: BLE001 - collected and reported together
      failed[name] = '%s: %s' % (type(e).__name__, str(e)[:200])
  assert not failed, failed
  assert len(trained) >= 60, len(trained)
  # the configs behind this round's additions are among them
  for must in ('dbmtl_on_multi_numeric_hash_bucket_sequence_feature_taobao.config', 'ple_on_taobao.config',
               'wide_and_deep_on_avazau_ctr.config', 'din_on_taobao.config', 'dssm_on_taobao.config'):
    assert must in trained, must
