#!/usr/bin/env bash
# Install the UNMODIFIED reference (kurtosis/mat_mul, a flat set of Python scripts with no packaging) from a checkout of
# it into the git-ignored baseline/_ref/.  The reference is third-party code and is not shipped with this repository.
# Used by
#   tests/test_reference_unchanged_gpu.py  (the reference's training.py / model.py run on the drop-in modules)
#   bench.py --impl reference              (times the reference's own step expression beside the C port)
# tests/golden/ref_sha256.json pins the file contents, so the test can prove the copy is unmodified.
#   usage: scripts/install_ref.sh <path to a kurtosis/mat_mul checkout>
set -euo pipefail
[ $# -eq 1 ] || { echo "usage: $0 <path to a kurtosis/mat_mul checkout>" >&2; exit 2; }
SRC="$1"
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
DST="$ROOT/baseline/_ref"
[ -f "$SRC/training.py" ] || { echo "no reference at $SRC" >&2; exit 1; }
mkdir -p "$DST"
cp "$SRC"/*.py "$DST"/
python - "$DST" "$ROOT/tests/golden/ref_sha256.json" <<'PY'
import hashlib, json, sys
from pathlib import Path
dst, out = Path(sys.argv[1]), Path(sys.argv[2])
digest = {p.name: hashlib.sha256(p.read_bytes()).hexdigest() for p in sorted(dst.glob("*.py"))}
if out.exists() and json.loads(out.read_text()) != digest:
    print("WARNING: reference files differ from the pinned hashes; rewriting", out, file=sys.stderr)
out.write_text(json.dumps(digest, indent=1, sort_keys=True) + "\n")
print("installed", ", ".join(digest), "->", dst)
PY
