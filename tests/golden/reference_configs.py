"""The reference's sample pipeline configs (alibaba/EasyRec samples/model_config/*.config and examples/configs/*.config,
Apache-2.0), stored as data in reference_configs.tar.xz, and what its full proto schema made of them, stored in
reference_schema.json.  Both are written by make_config_golden.py from a checkout of the reference."""
import json
import os
import tarfile

HERE = os.path.dirname(os.path.abspath(__file__))
ARCHIVE = os.path.join(HERE, 'reference_configs.tar.xz')
RECORD = os.path.join(HERE, 'reference_schema.json')
DIRS = ('samples/model_config', 'examples/configs')


def load():
  """{relative path: config bytes}, samples/model_config first, each directory in sorted order."""
  with tarfile.open(ARCHIVE, 'r:xz') as tar:
    texts = {m.name: tar.extractfile(m).read() for m in tar.getmembers() if m.isfile()}
  return {p: texts[p] for d in DIRS for p in sorted(texts) if os.path.dirname(p) == d}


def record():
  with open(RECORD) as f:
    return json.load(f)


def recorded_field_paths():
  """{relative path: set of the field paths the reference's full schema parses out of that config}"""
  r = record()
  names = r['field_paths']
  return {p: {names[i] for i in idx} for p, idx in r['config_fields'].items()}


def field_paths(msg, prefix=''):
  """every set field of a parsed config as a dotted path ('.model_config.deepfm.dnn.hidden_units'); map entries are
  not descended into."""
  from easyrec_b200 import builder
  out = set()
  for fd, v in msg.ListFields():
    p = prefix + '.' + fd.name
    out.add(p)
    if fd.type == fd.TYPE_MESSAGE and not fd.message_type.GetOptions().map_entry:
      for it in (list(v) if builder._is_repeated(fd) else [v]):
        out |= field_paths(it, p)
  return out
