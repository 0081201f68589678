#!/bin/bash
# pool planes against the default (compressible) planes, alternated in one run: C4 three times each, then C3, C5, C4 with
# gaps and with the whole validity plane once each; the dumped outputs of both arms compared byte for byte; then the suite
# and the smoke run.  Everything lands in the directory given as the first argument (default: a new temporary one).
cd "$(dirname "$0")/.." || exit 1
O=${1:-$(mktemp -d)}
echo "output in $O"
D=$(mktemp -d)   # the dumped outputs (up to 64 MB per workload) stay out of the output directory
mkdir -p $O
python __graft_entry__.py > $O/build.log 2>&1 || { tail -30 $O/build.log; exit 1; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,driver_version --format=csv,noheader -i 0 | tee $O/card.txt
arm() {  # arm <pool|default> <tag> <bench args...>
    local a=$1 t=$2; shift 2
    if [ "$a" = pool ]; then env PFA_PLANE_ALLOC=pool python bench.py --gpus 1 --no-cpu "$@" > $O/bench_${t}_$a.json 2> $O/bench_${t}_$a.err
    else python bench.py --gpus 1 --no-cpu "$@" > $O/bench_${t}_$a.json 2> $O/bench_${t}_$a.err; fi
    echo "$t $a rc=$? $(python -c "import json,sys; r=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); print('ms_per_step=%.4f kernel_ms=%.4f e2e_ms=%s kernel=%s' % (r['ms_per_step'], r['roofline']['kernel_ms'], (r.get('e2e') or {}).get('ms_per_step'), r['roofline']['kernel']))" $O/bench_${t}_$a.json 2>&1 | tail -1)"
}
for i in 1 2 3; do
    arm pool c4_$i --dump-outputs $D/dump_c4_pool
    arm default c4_$i --dump-outputs $D/dump_c4_default
done
arm pool c3 --workload c3 --dump-outputs $D/dump_c3_pool
arm default c3 --workload c3 --dump-outputs $D/dump_c3_default
arm default c5 --workload c5 --dump-outputs $D/dump_c5_default
arm pool c5 --workload c5 --dump-outputs $D/dump_c5_pool
arm pool c4_gaps10 --gaps-ppm 10
arm default c4_gaps10 --gaps-ppm 10
arm default c4_forcev --force-validity
arm pool c4_forcev --force-validity
for w in c4 c3 c5; do
    for f in $D/dump_${w}_pool/*.npy; do cmp "$f" "$D/dump_${w}_default/$(basename $f)" && echo "identical $w $(basename $f)"; done
done
python -m pytest -q -m gpu tests 2>&1 | tee $O/gpu_tests.log | tail -15
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tee $O/smoke.log | tail -3
rm -rf "$D"
