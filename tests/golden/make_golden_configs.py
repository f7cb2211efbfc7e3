"""Generate tests/golden/configs/*.gin and tests/golden/configs.json from a multinerf checkout.

    python tests/golden/make_golden_configs.py <path to a google-research/multinerf checkout>

configs/*.gin are copied byte for byte: tests/test_host_cpu.py feeds these unmodified files to the product's
gin parser.  configs.json records, for each file, its `include` lines and its `Class.attr = value`
bindings in file order, the values the parser is expected to produce.  Values are JSON literals; gin
references such as `@jnp.reciprocal` are recorded as {"ref": "jnp.reciprocal"}.

This reading does not import multinerf_b200.configs, but it uses the same method (comments cut at '#',
literals read with ast.literal_eval, '@' read as a reference).  It therefore checks that the parser handles
the files' structure and applies every binding, not that it reads a literal differently from Python.
"""
import ast
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def parse(text):
  includes, bindings = [], []
  for raw in text.splitlines():
    line = raw.split('#', 1)[0].strip()       # the shipped files have no '#' inside string values
    if not line:
      continue
    if line.startswith('include '):
      includes.append(ast.literal_eval(line[len('include '):].strip()))
      continue
    lhs, rhs = (s.strip() for s in line.split('=', 1))
    value = {'ref': rhs[1:]} if rhs.startswith('@') else ast.literal_eval(rhs)
    bindings.append([lhs, value])
  return {'include': includes, 'bindings': bindings}


def main(checkout):
  cfg_dir = os.path.join(checkout, 'configs')
  out_dir = os.path.join(HERE, 'configs')
  os.makedirs(out_dir, exist_ok=True)
  out = {}
  for name in sorted(os.listdir(cfg_dir)):
    if name.endswith('.gin'):
      shutil.copyfile(os.path.join(cfg_dir, name), os.path.join(out_dir, name))
      with open(os.path.join(cfg_dir, name)) as f:
        out[name] = parse(f.read())
  with open(os.path.join(HERE, 'configs.json'), 'w') as f:
    json.dump(out, f, indent=1)
    f.write('\n')


if __name__ == '__main__':
  main(sys.argv[1])
