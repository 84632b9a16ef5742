#!/usr/bin/env bash
# Stage the UNMODIFIED reference checkout under baseline/_ref/ (git-ignored).  The reference is pure
# Python with no setup.py / pyproject, so "installing" it is a copy of its tree; nothing is edited.
#   - bench.py --impl reference imports baseline/_ref/utils/rendering.py as the CPU arm
#   - tests/test_gpu_reference_cli.py runs baseline/_ref/train.py and test.py unchanged on the engine
# Usage: scripts/stage_reference.sh /path/to/Nerf-Simple      (default: $NERF_REFERENCE)
set -euo pipefail
SRC="${1:-${NERF_REFERENCE:?usage: scripts/stage_reference.sh /path/to/Nerf-Simple}}"
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
DST="$ROOT/baseline/_ref"
if [ ! -f "$SRC/train.py" ] || [ ! -d "$SRC/utils" ]; then
  echo "stage_reference: $SRC does not look like a Nerf-Simple checkout" >&2
  exit 1
fi
rm -rf "$DST"
mkdir -p "$DST"
cp -r "$SRC/train.py" "$SRC/test.py" "$SRC/utils" "$SRC/configs" "$SRC/README.md" "$SRC/requirements.txt" "$DST/"
find "$DST" -name '__pycache__' -type d -prune -exec rm -rf {} +
( cd "$SRC" && find train.py test.py utils configs -type f ! -path '*__pycache__*' -print0 | sort -z | xargs -0 sha256sum ) > "$DST/SHA256SUMS"
echo "staged $(wc -l < "$DST/SHA256SUMS") files from $SRC into $DST"
