#!/bin/bash
# Builds and runs tools/cluster_exchange_probe.cu (needs a GPU); prints one JSON line per cluster size and exchange form.
# PROBE_BIN=<path> runs a binary built beforehand; otherwise it is built in a temporary directory.
cd "$(dirname "$0")/.." || exit 1
BIN=${PROBE_BIN:-}
if [ -z "$BIN" ] || [ ! -x "$BIN" ]; then
  BIN=$(mktemp -d)/cluster_exchange_probe
  /usr/local/cuda/bin/nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o "$BIN" tools/cluster_exchange_probe.cu || exit 1
fi
exec "$BIN"
