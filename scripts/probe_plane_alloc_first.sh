#!/bin/bash
# the allocation probe (with the slot sweep), then the arm comparison of plane_alloc_round.sh; output in the directory given
# as the first argument (default: a new temporary one)
cd "$(dirname "$0")/.." || exit 1
O=${1:-$(mktemp -d)}
mkdir -p "$O"
python __graft_entry__.py > "$O/build.log" 2>&1 || { tail -30 "$O/build.log"; exit 1; }
python scripts/probe_plane_compression.py --sweep 2>&1 | tee "$O/probe_plane_compression.log"
bash scripts/plane_alloc_round.sh "$O"
