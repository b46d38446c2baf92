#!/usr/bin/env bash
# Installs the UNMODIFIED reference (DRCL-USC/isaac) from a checkout of it into baseline/_ref (git-ignored).
# bench.py --impl reference, the runner test and the live oracle-pinning tests import `humanoid` from there.
#
#     baseline/install_ref.sh [checkout of DRCL-USC/isaac]     (default: $ISAAC_REFERENCE, else /root/reference)
#
# setup.py writes build/ + egg-info next to itself, so pip installs from a copy under a temporary directory (the
# checkout may be read-only).  The reference's setup.py uses find_packages(), which skips the directories that have no
# __init__.py (humanoid/envs/base, humanoid/envs/custom: the reference is meant to be used with `pip install -e .`); the
# same source files are added to the installed tree afterwards so that baseline/_ref holds the whole package.
# --no-deps: the declared dependencies (isaacgym preview4, mujoco, opencv, numpy==1.23.5, ...) are not needed by the hot
# path (isaacgym is stubbed by oracle/ref_harness.py).
set -euo pipefail
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
SRC="${1:-${ISAAC_REFERENCE:-/root/reference}}"
TMP="$(mktemp -d)"
cp -r "$SRC/humanoid" "$SRC/setup.py" "$TMP/"
find "$TMP" -name __pycache__ -type d -prune -exec rm -rf {} +
rm -rf "$ROOT/baseline/_ref"
python -m pip install --no-index --no-build-isolation --no-deps --find-links /opt/wheelhouse \
    --target "$ROOT/baseline/_ref" "$TMP"
for d in envs/base envs/custom; do
    mkdir -p "$ROOT/baseline/_ref/humanoid/$d"
    cp "$SRC/humanoid/$d"/*.py "$ROOT/baseline/_ref/humanoid/$d/"
done
rm -rf "$TMP"
echo "installed: $(find "$ROOT/baseline/_ref/humanoid" -name '*.py' | wc -l) python files"
