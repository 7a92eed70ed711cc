"""CPU: no pipeline-config text this repository writes itself loses a field to the lenient parser.

The subset schema parses with allow_unknown_field (config/config_util.py), so a misspelt or misplaced field in a config
is skipped without a word and the model is built without it.  That is right for the reference's own configs, which
may use fields the port does not consume; for the configs written here (the BASELINE workloads of
easyrec_b200.workloads and every pipeline config embedded in tests/*.py) it hides mistakes.  Each field path of those
texts must either be declared by the subset schema or be a path the reference's complete schema parses out of its
sample configs (`field_paths` of tests/golden/reference_schema.json).

Texts embedded in the tests may be %-templates; a placeholder counts as a value, or is skipped where it stands for
whole fields.
"""
import ast
import glob
import json
import os
import re

import pytest

from easyrec_b200 import workloads
from easyrec_b200.config import proto_loader

HERE = os.path.dirname(os.path.abspath(__file__))
RECORD = json.load(open(os.path.join(HERE, 'golden', 'reference_schema.json')))
REF_PATHS = set(RECORD['field_paths'])

# (file, field path) pairs that are wrong on purpose
DELIBERATE = {
    # test_config.MINI shows that the subset parser skips a field it does not know
    ('test_config.py', '.feature_config.features.unknown_future_field'),
}

_TOKEN = re.compile(r'''\s+|\#[^\n]*|"(?:[^"\\\n]|\\.)*"|'(?:[^'\\\n]|\\.)*'|%(?:\(\w+\))?[-#0 +]*[\d.]*[a-zA-Z]'''
                    r'''|[{}\[\]<>:,;]|[^\s{}\[\]<>:,;"'#%]+''')


def _is_string(t):
  return t[:1] in ('"', "'")


def _fields(toks, i, prefix, out):
  """the field paths of one text-format message body starting at toks[i]; returns the index after its closing brace"""
  while i < len(toks):
    t = toks[i]
    if t in ('}', '>'):
      return i + 1
    if t in (',', ';'):
      i += 1
      continue
    path = prefix + (t,)
    i += 1
    if t.startswith('%'):
      if i >= len(toks) or toks[i] not in (':', '{', '<'):
        continue            # a template slot standing for whole fields
      out = set()           # a slot standing for a field name: what it holds cannot be checked
    else:
      out.add(path)
    if i < len(toks) and toks[i] == ':':
      i += 1
    if i >= len(toks):
      break
    if toks[i] in ('{', '<'):
      i = _fields(toks, i + 1, path, out)
    elif toks[i] == '[':
      i += 1
      while i < len(toks) and toks[i] != ']':
        i = _fields(toks, i + 1, path, out) if toks[i] in ('{', '<') else i + 1
      i += 1
    else:
      i += 1
      while _is_string(toks[i - 1]) and i < len(toks) and _is_string(toks[i]):   # "a" "b" is one string
        i += 1
  return i


def field_paths(text):
  if isinstance(text, bytes):
    text = text.decode('utf-8', errors='replace')
  toks = [t for t in _TOKEN.findall(text) if t.strip() and not t.startswith('#')]
  out = set()
  _fields(toks, 0, (), out)
  return out


def dropped_fields(text):
  """field paths of `text` that the subset schema lacks and the reference record does not know either (sorted
  '.a.b.c' strings; below an unknown field nothing more is reported)"""
  root = proto_loader.default_schema().EasyRecConfig.DESCRIPTOR
  bad = set()
  for path in field_paths(text):
    desc = root
    for k, name in enumerate(path):
      f = desc.fields_by_name.get(name) if desc is not None else None
      if f is None:
        dotted = '.' + '.'.join(path[:k + 1])
        if desc is not None and dotted not in REF_PATHS:
          bad.add(dotted)
        break
      desc = f.message_type
  return sorted(bad)


def _workload_texts():
  out = [('c2', workloads.c2_config_text(1000, 64)), ('c3', workloads.c3_config_text(64, 1000, 5))]
  for ep in (True, False):
    out.append(('c4 embedding_parallel=%s' % ep, workloads.c4_config_text(64, 1000, 1000, embedding_parallel=ep)))
    out.append(('c5 embedding_parallel=%s' % ep, workloads.c5_config_text(64, 1000, n_feat=4, embedding_parallel=ep)))
  return out


def _embedded_texts():
  """every string constant in tests/*.py that holds a pipeline config (a `model_config { ... }` message)"""
  out = []
  for path in sorted(glob.glob(os.path.join(HERE, '*.py'))):
    with open(path) as f:
      tree = ast.parse(f.read())
    for node in ast.walk(tree):
      if isinstance(node, ast.Constant) and isinstance(node.value, (str, bytes)):
        text = node.value.decode('utf-8', errors='replace') if isinstance(node.value, bytes) else node.value
        if re.search(r'(^|[\s{])model_config\s*\{', text):
          out.append(('%s:%d' % (os.path.basename(path), node.lineno), text))
  return out


EMBEDDED = _embedded_texts()


@pytest.mark.parametrize('name,text', _workload_texts(), ids=lambda v: v if isinstance(v, str) else '')
def test_workload_config_texts_lose_no_field(name, text):
  assert dropped_fields(text) == [], '%s: fields neither the subset schema nor the reference declares' % name


def test_config_texts_embedded_in_the_tests_lose_no_field():
  assert len(EMBEDDED) >= 40, 'the scan of tests/*.py found only %d pipeline configs' % len(EMBEDDED)
  problems = []
  for where, text in EMBEDDED:
    for path in dropped_fields(text):
      if (where.split(':')[0], path) not in DELIBERATE:
        problems.append('%s: %s' % (where, path))
  assert not problems, 'fields neither the subset schema nor the reference declares:\n' + '\n'.join(problems)


def test_the_check_finds_a_misplaced_field_and_accepts_reference_only_fields():
  # a DNN under a message that has no field of that name: the mistake the C5 task towers once carried
  bad = workloads.c5_config_text(64, 1000, n_feat=2).replace(b'dnn { hidden_units: [64] }', b'mlp { hidden_units: [64] }')
  assert dropped_fields(bad) == ['.model_config.model_params.task_towers.mlp']
  # fields the reference declares but the subset does not parse are not mistakes
  root = proto_loader.default_schema().EasyRecConfig.DESCRIPTOR
  skipped = [p for p in sorted(REF_PATHS) if p.count('.') == 1 and p[1:] not in root.fields_by_name]
  assert skipped, 'the reference record names no top-level field the subset skips'
  assert dropped_fields('%s { }\nmodel_config { model_class: "DeepFM" }' % skipped[0][1:]) == []
  # template slots stand for values or for whole fields; comments and strings hold no fields
  tpl = 'train_config { %s num_steps: %(n)d }  # hidden_units: 3\ndata_config { separator: "a { b: 1 }" "c" }'
  assert field_paths(tpl) == {('train_config',), ('train_config', 'num_steps'), ('data_config',),
                              ('data_config', 'separator')}
