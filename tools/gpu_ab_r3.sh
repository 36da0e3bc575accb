# On a B200: render-gather A/B. Expects next to the product library (python -c "import __graft_entry__ as g; g.build()"):
#   procgen_b200/libprocgen_b200_base.so  the parent commit's product library (the "old" arm)
#   procgen_b200/libprocgen_b200_rb7.so   build_variant("rb7", ["-DPG_RENDER_MIN_BLOCKS=7"])
#   procgen_b200/libprocgen_b200_phase.so build_variant("phase", ["-DPG_PHASE_TIMING"])
# Writes $AB_OUT (default ab_out/). One part per invocation, each under 10 minutes: bench = card, smoke, alternating default-bench
# runs; dump = byte comparison of --dump-outputs + render phase cycles; tests = the GPU suite;
# games1 / games2 = grid games old / new.
part=${1:-bench}
O=${AB_OUT:-ab_out}
mkdir -p $O
L=$PWD/procgen_b200
declare -A LIB=([old]=$L/libprocgen_b200_base.so [new]=$L/libprocgen_b200.so [rb7]=$L/libprocgen_b200_rb7.so)
summ() { python -c "
import json,sys
j=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); r=j['roofline']
print('%-4s %-10s %-5s %6d  %7.3f M/s  step %6.3f  logic %6.3f  setup %6.3f  render %6.3f' % (sys.argv[2], j['config']['game'][:10], j['config']['distribution_mode'], j['config']['envs_per_gpu'], j['value']/1e6, j['ms_per_step'], r['logic_kernel_ms_avg'], r['setup_kernel_ms_avg'], r['kernel_ms_avg']))" $1 $2; }
if [ $part = bench ]; then
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm,clocks.mem --format=csv > $O/card.csv 2>&1
python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke.txt 2>&1; echo "smoke exit $?" >> $O/smoke.txt; tail -2 $O/smoke.txt

# 1. the flagship (bench.py defaults: coinrun easy, 65536 envs), arms alternated
for i in 1 2 3; do
  for v in old new $([ $i -lt 3 ] && echo rb7); do
    PROCGEN_B200_LIB=${LIB[$v]} timeout 600 python bench.py --no-cpu-baseline > $O/bench_${v}_$i.json 2> $O/bench_${v}_$i.err
    summ $O/bench_${v}_$i.json $v | tee -a $O/ab_coinrun.txt
  done
done

fi

# 2. same outputs: --dump-outputs of both arms, byte for byte
dump() {  # name, args...
  local n=$1; shift
  for v in old new; do
    PROCGEN_B200_LIB=${LIB[$v]} timeout 600 python bench.py --no-cpu-baseline --no-e2e "$@" --dump-outputs $O/dump_${n}_$v > /dev/null 2> $O/dump_${n}_$v.err
  done
  if diff -r $O/dump_${n}_old $O/dump_${n}_new > /dev/null && [ -n "$(ls $O/dump_${n}_new 2>/dev/null)" ]; then echo "$n identical ($(ls $O/dump_${n}_new | tr '\n' ' '))"; else echo "$n DIFFERENT"; fi | tee -a $O/dump_compare.txt
}
if [ $part = dump ]; then
dump coinrun_easy_65536
for g in maze heist chaser ninja; do dump ${g}_hard_32768 --game $g --mode hard --envs-per-gpu 32768 --steps 30; done

# 5. render phase cycles (profiling variant)
PROCGEN_B200_LIB=$L/libprocgen_b200_phase.so timeout 300 python tools/gpu_render_phases.py coinrun easy 65536 300 > $O/render_phases.txt 2>&1
PROCGEN_B200_LIB=$L/libprocgen_b200_phase.so timeout 300 python tools/gpu_render_phases.py maze hard 32768 300 >> $O/render_phases.txt 2>&1
tail -20 $O/render_phases.txt
rm -rf $O/dump_*_old $O/dump_*_new
fi

# 3. the GPU suite on the product library
if [ $part = tests ]; then timeout 560 python -m pytest tests -q -m gpu -p no:cacheprovider > $O/pytest_gpu.txt 2>&1; tail -3 $O/pytest_gpu.txt; fi

# 4. grid games (32768 envs, hard), arms alternated, two runs each
games1="caveflyer chaser climber coinrun dodgeball fruitbot"; games2="heist jumper leaper maze miner ninja"
[ $part = games1 ] && games=$games1; [ $part = games2 ] && games=$games2
for g in $games; do
  for i in 1 2; do
    for v in old new; do
      PROCGEN_B200_LIB=${LIB[$v]} timeout 300 python bench.py --game $g --mode hard --envs-per-gpu 32768 --steps 30 --warmup 5 --desync-steps 300 --no-e2e --no-cpu-baseline > $O/games_${g}_${v}_$i.json 2>/dev/null
      summ $O/games_${g}_${v}_$i.json $v | tee -a $O/ab_games.txt
    done
  done
done

