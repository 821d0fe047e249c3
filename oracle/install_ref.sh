#!/usr/bin/env bash
# Copies the UNMODIFIED reference (zgcr/SimpleAICV_pytorch_training_examples) into oracle/_ref (git-ignored)
# so that baseline/ref_import.py can import it.  The reference is pure Python: its two import roots
# (SimpleAICV, tools) are copied as they are; no source file is edited.  Only the golden-data generators
# (tests/golden/make_*.py) and the torch baselines use it; the tests, smoke() and bench.py never do.
#
#   oracle/install_ref.sh <path to a checkout of the reference>
set -euo pipefail
REF=${1:?usage: oracle/install_ref.sh <reference checkout>}
HERE="$(cd "$(dirname "$0")" && pwd)"
rm -rf "$HERE/_ref"
mkdir -p "$HERE/_ref"
cp -r "$REF/SimpleAICV" "$REF/tools" "$HERE/_ref/"
python - <<PY
import sys; sys.path.insert(0, "$HERE/_ref")
from SimpleAICV.classification import backbones
print('reference installed:', len([k for k in backbones.__dict__ if not k.startswith('_')]), 'backbone symbols')
PY
