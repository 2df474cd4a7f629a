#!/bin/sh
# Installs the UNMODIFIED rsl_rl of the original project (PPO, ActorCritic, RolloutStorage: the update half of the hot path) into
# baseline/_ref (git-ignored), copied from the checkout of the original Deep-Whole-Body-Control repository that DWBC_REFERENCE names
# (the directory holding legged_gym/ and rsl_rl/).
# The env half (legged_gym's WidowGo1) imports the closed-source isaacgym package at module import and cannot be installed or run
# unmodified; tests/golden/ref_harness.py drives it through a fake isaacgym for the golden vectors only.
set -e
: "${DWBC_REFERENCE:?set DWBC_REFERENCE to a checkout of the original Deep-Whole-Body-Control repository}"
REF=$(cd "$DWBC_REFERENCE" && pwd)
cd "$(dirname "$0")/.."
rm -rf baseline/_ref
mkdir -p baseline/_ref
cp -r "$REF/rsl_rl/rsl_rl" baseline/_ref/rsl_rl
diff -rq -x __pycache__ "$REF/rsl_rl/rsl_rl" baseline/_ref/rsl_rl && echo "baseline/_ref/rsl_rl is identical to the reference tree"
