#!/bin/bash
# Installs the unmodified reference (UCSC-VLAA/CLIPA clipa_torch: its `open_clip` and `training` packages, with the
# BPE vocabulary and JSON model configs they load at import time) into oracle/_ref, where baseline/ref_loader.py
# imports it from.  oracle/_ref is git-ignored.  Only the golden-data generators and bench.py's library-baseline
# leg use it; tests and smoke() read the committed vectors under tests/golden instead.
#   usage: oracle/install_reference.sh <path to a clipa_torch checkout>
set -euo pipefail
src=${1:?usage: oracle/install_reference.sh <path to a clipa_torch checkout>}
dst="$(cd "$(dirname "$0")" && pwd)/_ref"
rm -rf "$dst"
mkdir -p "$dst"
cp -r "$src/open_clip" "$src/training" "$dst/"
chmod -R u+w "$dst"
find "$dst" -name __pycache__ -prune -exec rm -rf {} +
du -sh "$dst"
