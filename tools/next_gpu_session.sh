#!/bin/bash
# Everything round 2 could not measure after it lost its GPU access (DESIGN.md "What round 2 could not measure", section 8 item 0), as ONE
# command for a single `gpurun` call on a 1-GPU box, memory-bounded (largest store: 16 GiB + one segment) and time-bounded (every step under
# its own `timeout`; the whole script < 25 min).  Outputs go to gpurun_out/next_*; copy what is worth judging into profiles/.
#
#   /usr/local/graft/bin/gpurun --timeout 1700 -- 'bash tools/next_gpu_session.sh'
#   /usr/local/graft/bin/gpurun --timeout 1500 --gpus 2 -- 'bash tools/next_gpu_session.sh multi'      # two-device test, N=2 bench, C4
set +e
ROOT="$(cd "$(dirname "$0")/.." && pwd)"; cd "$ROOT"
O=gpurun_out; mkdir -p $O
run() { name=$1; t=$2; shift 2; echo "== $name"; timeout "$t" "$@" > $O/next_$name.log 2>&1; echo "   rc=$? $(tail -1 $O/next_$name.log | cut -c1-160)"; }

if [ "$1" = "multi" ]; then
  run pytest_multi 600 python -m pytest tests/test_zzzz_multi_gpu.py -m gpu -q
  run bench_n2 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29531 bench.py --gpus 2 --steps 3 --warmup 3
  run c4_n2 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29532 bench.py --config c4 --gpus 2 --gib-per-gpu 4
  exit 0
fi

nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,memory.total --format=csv > $O/next_box.txt 2>&1
grep -E "MemTotal|MemAvailable" /proc/meminfo >> $O/next_box.txt; cat /sys/fs/cgroup/memory.max >> $O/next_box.txt 2>/dev/null; df -h /dev/shm >> $O/next_box.txt
# 1. the parity gate, including the late-sorting files no B200 has run yet
run pytest_gpu 900 python -m pytest tests -m gpu -q --durations=15
# 2. headline + side legs (framed after the Open/Running/Complete pipelining is in e2e_framed / e2e_framed_unix)
run bench_n1 600 python bench.py --gpus 1 --steps 5 --warmup 3
run bench_ref 400 python bench.py --impl reference --gpus 1 --steps 3 --warmup 1
run c5 400 python bench.py --config c5 --gpus 1
# 3. kernel rates: defaults, then the copy walker with 4-row tiles (candidate for the 4 KiB-page scatter), then the staged walk
run kbench_default 300 python tools/kbench.py --gib 4
run kbench_copy_tile4 300 python tools/kbench.py --gib 4 --tile-copy 4
run kbench_staged 300 python tools/kbench.py --gib 4 --staged 1
# 4. SSD tier: GDS (where the box has nvidia-fs; else the pinned ring) against the pinned ring, and the HBM tier over it
run c3_gds 600 python tools/c3_ssd_tier.py --gib 8 --gds auto --hbm 2
# 5. one ncu capture of the K2 walker and the launch list of a short bench (never a bench value)
run ncu_launches 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/next_launches.csv python bench.py --gpus 1 --steps 2 --warmup 1 --side-steps 0 --legs resident
run ncu_k2 600 ncu --set full --clock-control none --import-source on -k regex:walk_kernel -c 4 -o $O/next_k2 python tools/kbench.py --gib 1 --only k2 --iters 2 --warm-sec 0
# 6. device-side sanitizers over the kernel parity files (the round-2 kernels have only the host-side shim's equivalents so far)
run memcheck 600 compute-sanitizer --tool memcheck python -m pytest tests/test_kernels_gpu.py tests/test_zzz_new_kernels_gpu.py -m gpu -q -x -k "not hypothesis and not linearity"
run racecheck 600 compute-sanitizer --tool racecheck python -m pytest tests/test_zzz_new_kernels_gpu.py -m gpu -q -x -k "small_inputs or multi_cta"
grep -h "^   rc=\|passed\|failed" $O/next_*.log | tail -30
