#!/bin/sh
# Stage the UNMODIFIED reference (its two Python packages and the three model YAMLs) under the git-ignored
# baseline/_ref/ so that the reference's own model and wrappers can run next to the B200 backend
# (tools/model_bench.py, the wrapper / model tests in tests/test_recurrent_and_wrappers_gpu.py and
# tests/test_cabi_cpu.py, bench.py's model_train block, the golden generators under tests/golden/).
# Without it those tests skip and bench.py reports "unavailable"; the product never imports it.
#
#   sh tools/stage_reference.sh <checkout of xlstm-yolo-clean>
set -e
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
SRC="${1:?usage: sh tools/stage_reference.sh <checkout of xlstm-yolo-clean>}"
DST="$ROOT/baseline/_ref"
[ -d "$SRC/mlstm_kernels" ] || { echo "no reference at $SRC" >&2; exit 1; }
rm -rf "$DST"
mkdir -p "$DST"
cp -r "$SRC/mlstm_kernels" "$SRC/ultralytics" "$DST/"
cp "$SRC"/640-base*.yaml "$DST/"
find "$DST" -name __pycache__ -type d -prune -exec rm -rf {} +
echo "staged $(du -sh "$DST" | cut -f1) into $DST"
