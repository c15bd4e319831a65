#!/bin/bash
# One gpurun call's worth of measurements; everything lands in gpurun_out/<tag>/.
#   gpurun --timeout 1500 -- 'bash tools/gpu_round.sh r02a tests bench sanitize probe'
tag=$1; shift
out=gpurun_out/$tag
mkdir -p $out
for what in "$@"; do
case $what in
tests)
  python -m pytest tests -m gpu -x -q 2>&1 | tail -25 > $out/pytest.log
  tail -3 $out/pytest.log ;;
bench)
  for m in 1 2 3 4; do
    python bench.py --steps 6 --warmup 3 --inflight $m --no-extras --no-cpu-baseline --no-parity > $out/bench_inflight$m.json 2> $out/bench_inflight$m.err
    python - <<PY
import json
try:
    l=json.loads(open("$out/bench_inflight$m.json").read().strip().splitlines()[-1])
    print("inflight $m value", round(l["value"],1), "e2e", round(l["e2e"]["value"],1), "lat", l["latency"])
except Exception as e:
    print("inflight $m failed", e, open("$out/bench_inflight$m.err").read()[-1500:])
PY
  done ;;
benchfull)
  python bench.py > $out/bench.json 2> $out/bench.err; tail -c 3000 $out/bench.json; tail -5 $out/bench.err
  python bench.py --impl reference --steps 3 --warmup 1 > $out/bench_ref.json 2> $out/bench_ref.err; tail -c 600 $out/bench_ref.json ;;
sanitize)
  for tool in memcheck racecheck synccheck; do
    timeout 900 compute-sanitizer --tool $tool --kernel-name kns=vb --print-limit 20 python tools/sanitize_target.py > $out/sanitizer_$tool.log 2>&1
    echo "$tool rc=$?"; grep -E "ERROR SUMMARY|RACECHECK SUMMARY|sanitize_target" $out/sanitizer_$tool.log | tail -3
  done ;;
sanitizebig)
  timeout 900 compute-sanitizer --tool memcheck --kernel-name kns=vb --print-limit 20 python tools/sanitize_target.py --big > $out/sanitizer_memcheck_big.log 2>&1
  echo "memcheck big rc=$?"; grep -E "ERROR SUMMARY|sanitize_target" $out/sanitizer_memcheck_big.log | tail -3 ;;
golden)
  python tests/make_golden.py > $out/make_golden.log 2>&1; tail -3 $out/make_golden.log ;;
p3ptime)
  # per-launch time of the hypothesis sampler, quad-lane vs one thread per hypothesis (legacy), 4-iteration C2 window
  for v in quad legacy; do
    if [ $v = legacy ]; then export VB_P3P_LEGACY=1; else unset VB_P3P_LEGACY; fi
    ncu --metrics gpu__time_duration.sum --clock-control none -k regex:solve_p3p --csv --log-file $out/p3p_$v.csv python tools/profile_window.py --iters 4 > $out/p3p_$v.log 2>&1
    python tools/summarize_launches.py $out/p3p_$v.csv | tail -4
  done; unset VB_P3P_LEGACY ;;
inflight)
  for m in ${INFLIGHT_LIST:-4 6 8}; do
    python bench.py --steps 6 --warmup 3 --inflight $m --no-extras --no-cpu-baseline --no-parity > $out/bench_inflight$m.json 2> $out/bench_inflight$m.err
    python - <<PY
import json
try:
    l=json.loads(open("$out/bench_inflight$m.json").read().strip().splitlines()[-1])
    print("inflight $m value", round(l["value"],1), "e2e", round(l["e2e"]["value"],1), "lat", l["latency"]["ms_per_window_in_flight"])
except Exception as e:
    print("inflight $m failed", e, open("$out/bench_inflight$m.err").read()[-1500:])
PY
  done ;;
conns)
  # hardware work queues: 6+ contexts x 2 streams alias onto the default 8 connections; A/B on one box, two rounds
  for rep in 1 2; do for c in 8 32; do for m in ${INFLIGHT_LIST:-6 8 12}; do
    CUDA_DEVICE_MAX_CONNECTIONS=$c python bench.py --steps 6 --warmup 3 --inflight $m --no-extras --no-cpu-baseline --no-parity > $out/bench_conn${c}_m${m}_$rep.json 2> $out/bench_conn${c}_m${m}_$rep.err
    python - <<PY
import json
try:
    l=json.loads(open("$out/bench_conn${c}_m${m}_$rep.json").read().strip().splitlines()[-1])
    print("round $rep connections $c inflight $m value", round(l["value"],1), "e2e", round(l["e2e"]["value"],1))
except Exception as e:
    print("connections $c inflight $m failed", e, open("$out/bench_conn${c}_m${m}_$rep.err").read()[-800:])
PY
  done; done; done ;;
weights)
  tools/_build/tex_probe weights $out/tex_weights.bin > $out/tex_weights.json 2>&1; cat $out/tex_weights.json ;;
profile)
  # (1) top kernels, full sections, one launch each (one window of the benchmarked shape); raw + source pages are
  #     exported on the box, only the search-kernel report itself travels back (gpurun_out/ is capped at 64 MiB)
  ncu --set full --clock-control none --import-source on -k regex:k_cost_and_random_search -s 1 -c 1 -f -o $out/search python tools/profile_window.py --iters 3 > $out/ncu_search.log 2>&1
  ncu --set full --clock-control none -k regex:k_local_propagation_group -s 4 -c 4 -f -o $out/localprop python tools/profile_window.py --iters 3 > $out/ncu_local.log 2>&1
  ncu --set full --clock-control none -k regex:k_solve_p3p_quad -s 8 -c 1 -f -o $out/p3p_quad python tools/profile_window.py --iters 3 > $out/ncu_p3p.log 2>&1
  ncu --set full --clock-control none -k regex:k_update_rigidness -s 1 -c 1 -f -o $out/estep python tools/profile_window.py --iters 3 > $out/ncu_estep.log 2>&1
  for r in search localprop p3p_quad estep; do
    ncu -i $out/$r.ncu-rep --page raw --csv > $out/${r}_raw.csv 2>/dev/null
  done
  ncu -i $out/search.ncu-rep --page source --csv > $out/search_source.csv 2>/dev/null
  rm -f $out/localprop.ncu-rep $out/p3p_quad.ncu-rep $out/estep.ncu-rep
  ls -la $out/*.ncu-rep $out/*_raw.csv
  # (2) every launch of one full 30-iteration window: duration + executed warp instructions
  ncu --metrics gpu__time_duration.sum,smsp__inst_executed.sum --clock-control none --csv --log-file $out/window_launches.csv python tools/profile_window.py --iters 30 > $out/ncu_window.log 2>&1
  echo "window launches rc=$?"; wc -l $out/window_launches.csv
  # (3) launch list of the bench command itself
  ncu --metrics gpu__time_duration.sum --clock-control none -c 12000 --csv --log-file $out/launches_bench.csv python bench.py --steps 1 --warmup 3 --no-extras --no-cpu-baseline --no-parity > $out/bench_under_ncu.log 2>&1
  echo "bench launches rc=$?"; wc -l $out/launches_bench.csv ;;
localsrc)
  # source-level view of one local-propagation launch in the middle of a window (iteration 16 of 20)
  ncu --set full --clock-control none --import-source on -k regex:k_local_propagation_group -s 60 -c 1 -f -o $out/localsrc python tools/profile_window.py --iters 20 > $out/ncu_localsrc.log 2>&1
  ncu -i $out/localsrc.ncu-rep --page source --csv > $out/localprop_source.csv 2>/dev/null
  ncu -i $out/localsrc.ncu-rep --page raw --csv > $out/localsrc_raw.csv 2>/dev/null
  rm -f $out/localsrc.ncu-rep; ls -la $out/localprop_source.csv ;;
gpus2)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29517 bench.py --gpus 2 --steps 4 --warmup 3 --no-extras --no-cpu-baseline > $out/bench_gpus2.json 2> $out/bench_gpus2.err
  tail -c 1500 $out/bench_gpus2.json; tail -3 $out/bench_gpus2.err ;;
gpus8)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29518 bench.py --gpus 8 --steps 4 --warmup 3 --no-extras --no-cpu-baseline > $out/bench_gpus8.json 2> $out/bench_gpus8.err
  tail -c 1500 $out/bench_gpus8.json; tail -3 $out/bench_gpus8.err ;;
probe)
  tools/_build/tex_probe 27 > $out/tex_probe.json 2>&1; cat $out/tex_probe.json ;;
launches)
  ncu --metrics gpu__time_duration.sum --clock-control none -c 4000 --csv --log-file $out/launches.csv python bench.py --steps 2 --warmup 3 --no-extras --no-cpu-baseline --no-parity > $out/bench_under_ncu.log 2>&1
  echo "ncu launches rc=$?"; wc -l $out/launches.csv ;;
esac
done
