#!/bin/bash
# drift over three loop bodies under the Morton-domain decomposition: 16M particles on 1/2/4/8 GPUs, 64M on 8
# (rank counts above the visible GPU count are skipped); one JSON line per run in OUT/drift_domains.jsonl
# usage: scripts/evidence/drift_domains.sh [OUT]   (OUT defaults to drift_out)
OUT=${1:-drift_out}
mkdir -p "$OUT"
export OUT
NGPU=$(python -c "import torch; print(torch.cuda.device_count())")
: > "$OUT/drift_domains.jsonl"
for run in "1 16000000" "2 16000000" "4 16000000" "8 16000000" "8 64000000"; do
  set -- $run
  if [ "$1" -gt "$NGPU" ]; then echo "skip N=$1 P=$2 ($NGPU GPUs)"; continue; fi
  TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node $1 --master-addr 127.0.0.1 --master-port 29513"
  timeout 900 $TR scripts/drift_domains.py --particles $2 --steps 3 > "$OUT/drift_$1_$2.out" 2> "$OUT/drift_$1_$2.err"
  echo "N=$1 P=$2 rc=$?"
  grep "^{" "$OUT/drift_$1_$2.out" | tail -n 1 >> "$OUT/drift_domains.jsonl"
done
python - <<'PY'
import json, os
rows = [json.loads(l) for l in open(os.path.join(os.environ["OUT"], "drift_domains.jsonl"))]
for r in rows:
    print(r["ranks"], r["particles"], "E0", r["first"]["e_total"], "dE/|E0|", r["energy_rel"], "calls s", r["conserved_call_s"], r["gpu"], r["power_limit"])
ref = [r for r in rows if r["particles"] == 16000000 and r["ranks"] == 1]
for r in rows:
    if ref and r["particles"] == 16000000:
        worst = max(abs(r["first"][k] - ref[0]["first"][k]) / max(abs(ref[0]["first"][k]), 1e-300) for k in ("e_kin", "e_int", "e_pot", "mass"))
        print("N", r["ranks"], "first vs 1 rank, max rel (energies, mass):", worst)
PY
