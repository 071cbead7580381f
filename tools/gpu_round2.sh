# round-2 evidence run (one GPU): tests, bench (both arms), forward-latency curves, timelines, ncu launch list + full captures
# usage: bash tools/gpu_round2.sh OUTPUT_DIR   (from the repository root)
set -x
OUT=${1:?output directory}
mkdir -p "$OUT"
python -m pytest tests -m gpu -q > "$OUT"/t_gpu_r2.log 2>&1
python __graft_entry__.py --smoke > "$OUT"/smoke_r2.log 2>&1
python bench.py --impl reference --steps 3 --warmup 1 > "$OUT"/bench_ref_r2.json 2> "$OUT"/bench_ref_r2.err
python bench.py > "$OUT"/bench_r2.json 2> "$OUT"/bench_r2.err
python bench.py --numerics bf16x3 --steps 3 > "$OUT"/bench_x3_r2.json 2> "$OUT"/bench_x3_r2.err
for n in 16 64 148 222 296 370 400 444 500 518 592 740; do python tools/fwd_loop.py $n 200; done 2>&1 | grep "^n=" > "$OUT"/fwd_curve_r2.log
for n in 16 148 370 500 740; do python tools/fwd_loop.py $n 100 bf16x3; done 2>&1 | grep "^n=" >> "$OUT"/fwd_curve_r2.log
python tools/pp_timeline.py 500 > "$OUT"/tl_pp_r2.log 2>&1
python tools/trunk_timeline.py 345 > "$OUT"/tl_r2.log 2>&1
python tools/trunk_timeline.py 40 > "$OUT"/tl40_r2.log 2>&1
UTTT_PROFILE=2 python tools/prof_selfplay.py --games 500 --reps 3 > "$OUT"/plain_r2.log 2>&1
python tools/determinism_check.py 500 > "$OUT"/determinism_r2.log 2>&1
echo '`ncu --metrics gpu__time_duration.sum --clock-control none -s 2600 -c 800 python bench.py --steps 2 --warmup 3 --no-extras --no-cpu-baseline --saturated-games 0` (launches 2600..3399 of the bench command: inside its warm-up / timed self-play cycles)' > "$OUT"/launches_r2.cmd
ncu --metrics gpu__time_duration.sum --clock-control none -s 2600 -c 800 --csv --log-file "$OUT"/launches_r2.csv python bench.py --steps 2 --warmup 3 --no-extras --no-cpu-baseline --saturated-games 0 > "$OUT"/ncu_launch_r2.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:trunk_auto -s 200 -c 1 -f -o "$OUT"/prof_trunkpp_r2 python tools/prof_selfplay.py --games 500 > "$OUT"/ncu_pp_r2.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:trunk_auto -s 3 -c 1 -f -o "$OUT"/prof_trunk2_r2 python tools/trunk_timeline.py 345 > "$OUT"/ncu2_r2.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:trunk_x3 -s 3 -c 1 -f -o "$OUT"/prof_trunkx3_r2 python tools/fwd_loop.py 500 6 bf16x3 > "$OUT"/ncu_x3_r2.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:tree_round -s 200 -c 1 -f -o "$OUT"/prof_tree_r2 python tools/prof_selfplay.py --games 500 > "$OUT"/ncu4_r2.log 2>&1
# rules kernels (plain runs: 2^22 and 2^24 positions) and the micro-benchmarks behind DESIGN.md section 9
python tools/prof_rules.py 22 > "$OUT"/rules_plain22.log 2>&1; cp "$OUT"/rules_points.json "$OUT"/rules_points22.json
python tools/prof_rules.py 24 > "$OUT"/rules_plain24.log 2>&1; cp "$OUT"/rules_points.json "$OUT"/rules_points24.json
mkdir -p build
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o build/mma_shapes tools/micro/mma_shapes.cu && build/mma_shapes > "$OUT"/mma_shapes.txt 2>&1
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o build/nt_skeleton tools/micro/nt_skeleton.cu && build/nt_skeleton > "$OUT"/nt_skeleton.txt 2>&1
tail -3 "$OUT"/t_gpu_r2.log
