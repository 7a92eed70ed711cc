"""Cross-check easyrec_b200/config/easyrec_subset.proto against the reference's full schema:
every message/field/enum value of the subset must exist in alibaba/EasyRec's protos with the same
number, type, label and default.

  python tools/check_subset_schema.py [PROTO_DIR]

PROTO_DIR is the reference's easy_rec/python/protos; without it the subset is checked against the record of those
protos in tests/golden/reference_schema.json (written by tests/golden/make_config_golden.py)."""
import glob
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from easyrec_b200.config import proto_loader as PL  # noqa: E402

RECORD = os.path.join(ROOT, 'tests', 'golden', 'reference_schema.json')


def _subset_file():
  sub = PL.load_schema([os.path.join(ROOT, 'easyrec_b200', 'config', 'easyrec_subset.proto')], virtual_name='sub.proto')
  return sub._pool.FindFileByName('sub.proto')


def _label(fd):
  if hasattr(fd, 'is_repeated'):     # protobuf >= 5.29 deprecates FieldDescriptor.label
    rep, req = fd.is_repeated, fd.is_required
    rep, req = (rep() if callable(rep) else rep), (req() if callable(req) else req)
    return 'repeated' if rep else 'required' if req else 'optional'
  return {fd.LABEL_REPEATED: 'repeated', fd.LABEL_REQUIRED: 'required'}.get(fd.label, 'optional')


def _field(fd):
  return {'number': fd.number, 'type': fd.type, 'label': _label(fd),
          'default': repr(fd.default_value) if fd.has_default_value else None,
          'message_type': fd.message_type.name if fd.message_type is not None else None,
          'oneof': fd.containing_oneof.name if fd.containing_oneof else None}


def _enum(se, re_):
  rv = {v.name: v.number for v in re_.values}
  return {v.name: rv.get(v.name) for v in se.values}


def _msg(sd, rd):
  """the reference message rd as far as the subset message sd names it (None where the reference lacks a name)"""
  rf = {f.name: f for f in rd.fields}
  rn = {x.name: x for x in rd.nested_types}
  re_ = {x.name: x for x in rd.enum_types}
  return {'fields': {f.name: _field(rf[f.name]) if f.name in rf else None for f in sd.fields},
          'nested': {n.name: _msg(n, rn[n.name]) if n.name in rn else None for n in sd.nested_types},
          'enums': {e.name: _enum(e, re_[e.name]) if e.name in re_ else None for e in sd.enum_types}}


def describe_reference(ref_dir):
  """what the check compares against: the reference protos' counterpart of every message, field and enum value
  the subset declares, as plain data (JSON-able)"""
  ref = PL.load_schema(sorted(glob.glob(os.path.join(ref_dir, '*.proto'))), virtual_name='ref.proto')
  fd = _subset_file()
  out = {'messages': {}, 'enums': {}}
  for name, sd in fd.message_types_by_name.items():
    try:
      out['messages'][name] = _msg(sd, ref._pool.FindMessageTypeByName('protos.' + name))
    except KeyError:
      out['messages'][name] = None
  for name, se in fd.enum_types_by_name.items():
    try:
      out['enums'][name] = _enum(se, ref._pool.FindEnumTypeByName('protos.' + name))
    except KeyError:
      out['enums'][name] = None
  return out


def check(reference=None):
  """reference: a directory of the reference's .proto files, or describe_reference()'s record of them (default: the
  record committed under tests/golden).  Returns the list of problems, empty when the subset is consistent."""
  if reference is None:
    with open(RECORD) as f:
      reference = json.load(f)['schema']
  elif isinstance(reference, str):
    reference = describe_reference(reference)
  problems = []
  unrecorded = 'not in the recorded reference schema (re-record it: tests/golden/make_config_golden.py)'

  def cmp_enum(se, rec, where):
    for v in se.values:
      if v.name not in rec:
        problems.append('%s: enum value %s %s' % (where, v.name, unrecorded))
      elif rec[v.name] != v.number:
        problems.append('%s: enum value %s=%d, reference %r' % (where, v.name, v.number, rec[v.name]))

  def cmp_msg(sd, rec):
    for f in sd.fields:
      if f.name not in rec['fields']:
        problems.append('%s.%s: %s' % (sd.full_name, f.name, unrecorded))
        continue
      r = rec['fields'][f.name]
      if r is None:
        problems.append('%s.%s: not in reference' % (sd.full_name, f.name))
        continue
      a = _field(f)
      for attr in ('number', 'type', 'label'):
        if a[attr] != r[attr]:
          problems.append('%s.%s: %s %r != reference %r' % (sd.full_name, f.name, attr, a[attr], r[attr]))
      if a['default'] != r['default']:
        problems.append('%s.%s: default %s != reference %s' % (sd.full_name, f.name, a['default'], r['default']))
      if a['message_type'] is not None and r['message_type'] is not None and a['message_type'] != r['message_type']:
        problems.append('%s.%s: message type %s != %s' % (sd.full_name, f.name, a['message_type'], r['message_type']))
      if a['oneof'] != r['oneof']:
        problems.append('%s.%s: oneof %r != %r' % (sd.full_name, f.name, a['oneof'], r['oneof']))
    for n in sd.nested_types:
      if n.name not in rec['nested']:
        problems.append('%s: nested message %s' % (n.full_name, unrecorded))
      elif rec['nested'][n.name] is None:
        problems.append('%s: nested message missing in reference' % n.full_name)
      else:
        cmp_msg(n, rec['nested'][n.name])
    for e in sd.enum_types:
      if e.name not in rec['enums']:
        problems.append('%s: nested enum %s' % (e.full_name, unrecorded))
      elif rec['enums'][e.name] is None:
        problems.append('%s: nested enum missing in reference' % e.full_name)
      else:
        cmp_enum(e, rec['enums'][e.name], e.full_name)

  fd = _subset_file()
  for name, sd in fd.message_types_by_name.items():
    if name not in reference['messages']:
      problems.append('message %s %s' % (name, unrecorded))
    elif reference['messages'][name] is None:
      problems.append('message %s missing in reference' % name)
    else:
      cmp_msg(sd, reference['messages'][name])
  for name, se in fd.enum_types_by_name.items():
    if name not in reference['enums']:
      problems.append('enum %s %s' % (name, unrecorded))
    elif reference['enums'][name] is None:
      problems.append('enum %s missing in reference' % name)
    else:
      cmp_enum(se, reference['enums'][name], name)
  return problems


if __name__ == '__main__':
  ps = check(sys.argv[1] if len(sys.argv) > 1 else None)
  print('\n'.join(ps) if ps else 'subset schema is consistent with the reference schema')
  sys.exit(1 if ps else 0)
