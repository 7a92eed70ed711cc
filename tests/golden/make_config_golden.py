"""Writes reference_configs.tar.xz and reference_schema.json from a checkout of the reference (alibaba/EasyRec):

  python tests/golden/make_config_golden.py REFERENCE_CHECKOUT

  reference_configs.tar.xz  every samples/model_config/*.config and examples/configs/*.config, unmodified
  reference_schema.json     schema: the reference protos' counterpart of everything easyrec_subset.proto declares
                            (tools/check_subset_schema.py compares the subset with it);
                            config_fields: per config, the field paths the reference's full schema parses out of it
                            (strict: a config that does not parse there stops this script), as indices into
                            field_paths.
"""
import glob
import io
import json
import os
import sys
import tarfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
sys.path.insert(0, HERE)

import check_subset_schema  # noqa: E402
import reference_configs as RC  # noqa: E402
from easyrec_b200.config import config_util, proto_loader  # noqa: E402


def main(ref):
  protos = os.path.join(ref, 'easy_rec', 'python', 'protos')
  paths = [os.path.relpath(p, ref) for d in RC.DIRS for p in sorted(glob.glob(os.path.join(ref, d, '*.config')))]
  buf = io.BytesIO()
  with tarfile.open(fileobj=buf, mode='w') as tar:   # fixed metadata: the archive depends on the files alone
    for p in paths:
      data = open(os.path.join(ref, p), 'rb').read()
      info = tarfile.TarInfo(p)
      info.size, info.mode, info.mtime = len(data), 0o644, 0
      tar.addfile(info, io.BytesIO(data))
  import lzma
  with open(RC.ARCHIVE, 'wb') as f:
    f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))
  full = proto_loader.load_schema(sorted(glob.glob(os.path.join(protos, '*.proto'))), virtual_name='full_ref.proto')
  per_config = {p: RC.field_paths(config_util.get_configs_from_pipeline_file(os.path.join(ref, p), schema=full))
                for p in paths}
  names = sorted(set().union(*per_config.values()))
  index = {n: i for i, n in enumerate(names)}
  out = {'_provenance': 'written by tests/golden/make_config_golden.py from alibaba/EasyRec (Apache-2.0): '
                        'easy_rec/python/protos and the sample configs',
         'schema': check_subset_schema.describe_reference(protos),
         'field_paths': names,
         'config_fields': {p: sorted(index[n] for n in per_config[p]) for p in paths}}
  with open(RC.RECORD, 'w') as f:
    json.dump(out, f, indent=None, separators=(',', ':'), sort_keys=True)
    f.write('\n')
  print('%d configs, %d field paths' % (len(paths), len(names)))


if __name__ == '__main__':
  main(sys.argv[1])
