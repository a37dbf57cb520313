"""Store the reference's rule tables (crafter/data.yaml, parsed) as tests/golden/data_yaml.json, so that
tests/test_rules_table.py diffs crafter_b200/rules.py against them wherever it runs.

    python tools/make_rules_golden.py
"""
import json
import pathlib
import sys

import yaml

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from oracle import ref_harness as rh  # noqa: E402

data = yaml.safe_load((rh.REFERENCE / 'crafter' / 'data.yaml').read_text())
path = ROOT / 'tests' / 'golden' / 'data_yaml.json'
path.write_text(json.dumps(data, indent=1) + '\n')
print(path, sorted(data))
