#!/bin/bash
# Round-2 multi-GPU session on N GPUs: drift/race parity of the fused halo, NCCL-halo parity, then bench lines
# at the requested rank counts.   bash scripts/gpu_multi2.sh <label> <N> [bench args]
set -u
LABEL=${1:-multi}; N=${2:-2}; shift 2 || true
EXTRA=${*:-}
OUT=gpurun_out/$LABEL
mkdir -p "$OUT"
nvidia-smi --query-gpu=index,name,clocks.sm,clocks.max.sm,power.draw --format=csv > "$OUT/gpu.csv" 2>&1
run_check() {  # name, env...
  local name=$1; shift
  env "$@" timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port $((29600 + RANDOM % 300)) \
      scripts/multigpu_check.py > "$OUT/check_$name.log" 2>&1
  echo "check $name rc=$?" | tee -a "$OUT/rc.log"; grep '^{' "$OUT/check_$name.log" | tail -1; grep -E "Error|error" "$OUT/check_$name.log" | tail -2 | cut -c1-300
}
run_check p2p WAFER_P2P=1
run_check nccl WAFER_P2P=0
if [ "${EXCITED:-1}" = 1 ]; then
  timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29555 \
      scripts/multigpu_excited.py > "$OUT/excited_$N.log" 2>&1
  echo "excited rc=$?" | tee -a "$OUT/rc.log"; grep '^{' "$OUT/excited_$N.log" | tail -1
fi
for n in ${NLIST:-$N}; do
  if [ $n -eq 1 ]; then
    timeout 900 python bench.py --gpus 1 --steps 3 --warmup 3 --no-cpu --no-512 $EXTRA > "$OUT/scale_$n.json" 2> "$OUT/scale_$n.err"
  else
    timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port $((29700+n)) \
      bench.py --gpus $n --steps 3 --warmup 3 $EXTRA > "$OUT/scale_$n.json" 2> "$OUT/scale_$n.err"
  fi
  echo "scale $n rc=$?" | tee -a "$OUT/rc.log"; grep '^{' "$OUT/scale_$n.json" | python -c "
import sys, json
for l in sys.stdin:
    d = json.loads(l); print('N=%d value=%.1f GLUPS e2e=%s E=%s parity=%s' % (d['n_gpus'], d['value'], d['e2e'] and round(d['e2e']['value'],1), d['e2e'] and d['e2e']['last_energy'], d['parity'] and (d['parity']['ok'], d['parity']['energy_rel_diff'])))"
  tail -2 "$OUT/scale_$n.err"
done
