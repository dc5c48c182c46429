#!/usr/bin/env bash
# Builds the original project's CPU CLI (b4rtaz/distributed-llama), unmodified and with its own Makefile, into
# oracle/_ref/distributed-llama (not part of the repository).
#
#   bash oracle/build_reference.sh <distributed-llama checkout>
#
# From there oracle/golden_reference_parity.py regenerates tests/golden/reference_parity.json, and
# `bench.py --impl reference` rebuilds it on the machine it runs on (the Makefile uses -march=native).
set -euo pipefail
src=${1:?usage: oracle/build_reference.sh <distributed-llama checkout>}
dst="$(cd "$(dirname "$0")" && pwd)/_ref/distributed-llama"
rm -rf "$dst"
mkdir -p "$(dirname "$dst")"
cp -r "$src" "$dst"
chmod -R u+w "$dst"
make -C "$dst" clean > /dev/null
make -C "$dst" dllama -j"$(nproc)"
