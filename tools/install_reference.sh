#!/bin/bash
# Copies the reference's PPO consumer (IsaacGymEnvs/algorithms/: ppo_asymmetry.py, nets_asymmetry.py, buffer_asymmetry.py)
# UNMODIFIED into the git-ignored baseline/_ref/, next to the project, so that it can be used on a machine without the reference tree.
# Used by tools/run_reference_ppo.py: the reference's own PPO.run drives FpvVecTask.
# Needs a copy of the reference (TACO_REFERENCE points to it).
set -e
REF=${TACO_REFERENCE:-/root/reference}
ROOT=$(cd "$(dirname "$0")/.." && pwd)
[ -d "$REF/IsaacGymEnvs/algorithms" ] || { echo "reference tree not found at $REF"; exit 0; }
mkdir -p "$ROOT/baseline/_ref"
rm -rf "$ROOT/baseline/_ref/algorithms"
cp -r "$REF/IsaacGymEnvs/algorithms" "$ROOT/baseline/_ref/algorithms"
find "$ROOT/baseline/_ref/algorithms" -name "__pycache__" -prune -exec rm -rf {} +
[ -f "$ROOT/baseline/_ref/algorithms/__init__.py" ] || touch "$ROOT/baseline/_ref/algorithms/__init__.py"
( cd "$REF/IsaacGymEnvs/algorithms" && sha256sum *.py ) > "$ROOT/baseline/_ref/algorithms.sha256"
echo "installed: $(ls "$ROOT/baseline/_ref/algorithms" | tr '\n' ' ')"
