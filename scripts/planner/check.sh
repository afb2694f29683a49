#!/bin/bash
# Planner without a GPU: digests of the plans of every case x ranks x schedule (phi, sparse_phi, its symmetric variant,
# gen.f's, gen.phi_pairs') with 1..N threads must agree
# (and agree with a digest file of an earlier build, if one is given), then ThreadSanitizer on a few.
#   bash scripts/planner/check.sh /tmp/plancases [reference_digests.txt]
set -e
D=${1:-/tmp/plancases}; REF=$2
HERE=$(cd "$(dirname "$0")" && pwd); SRC="$HERE/../../genlib.jl_b200/csrc/plan.cpp"
[ -f "$D/geneaJi.bin" ] || python "$HERE/dump_cases.py" "$D"
g++ -O3 -std=c++17 -Wall -Wextra -DPLAN_CPP="\"$SRC\"" "$HERE/plan_harness.cpp" -o "$D/harness" -lpthread
g++ -O1 -g -fsanitize=thread -std=c++17 -DPLAN_CPP="\"$SRC\"" "$HERE/plan_harness.cpp" -o "$D/harness_tsan" -lpthread
run() { for f in "$D"/*.bin; do for w in 1 2 3 8; do for s in 0 1 2 3 4; do for st in 0 1; do "$D/harness" "$f" $w $s 1 $st 2>/dev/null; done; done; done; done; }
GENLIB_PLAN_THREADS=1 run > "$D/digests_1.txt"
for t in 2 3 5; do GENLIB_PLAN_THREADS=$t run > "$D/digests_$t.txt"; cmp "$D/digests_1.txt" "$D/digests_$t.txt"; done
[ -z "$REF" ] || cmp "$REF" "$D/digests_1.txt"
for f in "$D"/genea140.bin "$D"/rand303.bin; do for w in 1 3; do for s in 0 3 4; do
  GENLIB_PLAN_THREADS=3 "$D/harness_tsan" "$f" $w $s 2 1 2>&1 | grep -E "WARNING|SUMMARY" && exit 1
done; done; done
echo "planner: $(wc -l < "$D/digests_1.txt") plans identical with 1, 2, 3, 5 threads; ThreadSanitizer clean"
