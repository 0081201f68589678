#!/bin/bash
# quick probe of the scan kernels after a change: parity subset, C3 shape (K2/K4, 1 and 2 populations), C4 bench line.
# Logs land in the directory given as the first argument (default: a new temporary one), named after the second (tag).
O=${1:-$(mktemp -d)}
tag=${2:-r2x}
mkdir -p "$O"
echo "output in $O"
timeout 600 python -m pytest tests/test_gpu_parity.py tests/test_gpu_xchg.py -m gpu -x -q > $O/${tag}_gpu_tests.log 2>&1; echo "tests rc=$?" >> $O/${tag}_gpu_tests.log; tail -4 $O/${tag}_gpu_tests.log
for m in 0 4; do echo "== m=$m"; if [ "$m" = "0" ]; then python scripts/probe_c3_c5.py --c3-only; else PFA_SITE_TMA_M=$m PFA_CDS_TMA_M=$m python scripts/probe_c3_c5.py --c3-only; fi; done > $O/${tag}_probe_c3.log 2>&1; cat $O/${tag}_probe_c3.log
python bench.py --steps 20 --warmup 3 --no-cpu --no-e2e > $O/${tag}_bench_c4.json 2> $O/${tag}_bench_c4.err; python - <<PY
import json
d=json.load(open("$O/${tag}_bench_c4.json"))
print("C4: ms/step %.4f kernel_ms %.4f frac %.4f of read-only %.4f" % (d["ms_per_step"], d["roofline"]["kernel_ms"], d["roofline"]["frac"], d["roofline"]["frac_of_read_only_peak"]))
PY
