#!/bin/sh
# oracle/make_ref.sh -- stage the UNMODIFIED reference step loop under oracle/_ref/ so that the CPU
# legs of bench.py can time the reference itself (kind "reference") instead of the restatement in
# oracle/py_loop.py. Usage: make_ref.sh <checkout of the original project> (default
# $INVERSUS_REFERENCE_ROOT); oracle/_ref/ is git-ignored, like the built .so files.
# Only the pure-Python files of the step path are staged: the engine package and
# the wrapper module (numpy + stdlib only). Nothing in the product imports it
# (tests/test_capi_surface.py::test_product_never_imports_the_oracle).
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
REF="${1:-$INVERSUS_REFERENCE_ROOT}"
if [ ! -d "$REF/inversus" ] || [ ! -f "$REF/inversus_rl/env_wrappers.py" ]; then
    echo "make_ref: no reference at $REF (nothing staged)"; exit 0
fi
rm -rf "$HERE/_ref"
mkdir -p "$HERE/_ref/inversus" "$HERE/_ref/inversus_rl"
for f in __init__.py core.py game_types.py config.py; do cp "$REF/inversus/$f" "$HERE/_ref/inversus/$f"; done
cp "$REF/inversus_rl/env_wrappers.py" "$HERE/_ref/inversus_rl/env_wrappers.py"
# the reference's own inversus_rl/__init__.py pulls in torch-based modules that are not on this path
: > "$HERE/_ref/inversus_rl/__init__.py"
( cd "$REF" && git rev-parse HEAD 2>/dev/null || echo unknown ) > "$HERE/_ref/SOURCE_COMMIT"
echo "make_ref: staged $(find "$HERE/_ref" -name '*.py' | wc -l) files from $REF into $HERE/_ref"
