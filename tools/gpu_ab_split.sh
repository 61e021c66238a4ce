#!/bin/bash
# A/B of the fp16x3 forward's shared epilogues on one GPU, A and B alternated three times each with the default benchmark:
#   A = a library built from the parent commit, path in $1, e.g.
#         git worktree add /tmp/parent HEAD~1 && python /tmp/parent/lab4d_b200/build.py && cp /tmp/parent/lab4d_b200/libb200render.so lab4d_b200/libb200render_parent.so
#   B = the in-tree library (python lab4d_b200/build.py).
# Runs A1, A2 and B1 also dump the rendered pixels and gradients: rend.* must match exactly between A and B, and B's
# gradients may differ from A1 by no more than A2 does (the weight-gradient kernel's fp32 atomics vary run to run).
# Usage: tools/gpu_ab_split.sh lab4d_b200/libb200render_parent.so [out dir, default: a new temporary directory]
set -u
A_LIB=$(realpath "$1")
OUT=${2:-$(mktemp -d -t ab_split.XXXXXX)}
mkdir -p "$OUT"
echo "logs and output dumps: $OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"
bench() {  # $1 = run name, rest = extra bench.py arguments
  local name=$1; shift
  timeout 300 python bench.py --gpus 1 --steps 100 --warmup 10 --no-cpu-baseline "$@" > "$OUT/$name.log" 2>&1
  echo "$name rc=$? $(grep -o '"ms_per_step": [0-9.]*' "$OUT/$name.log" | head -1) $(grep -o '"forward_call": [0-9.]*, "backward_call": [0-9.]*' "$OUT/$name.log" | head -1)"
}
for rep in 1 2 3; do
  if [ "$rep" -le 2 ]; then B200R_LIB=$A_LIB bench "A$rep" --dump-outputs "$OUT/dump_A$rep"; else B200R_LIB=$A_LIB bench "A$rep"; fi
  if [ "$rep" -eq 1 ]; then bench "B$rep" --dump-outputs "$OUT/dump_B$rep"; else bench "B$rep"; fi
done
python - "$OUT" <<'EOF'
import glob, json, os, re, sys
import numpy as np
out = sys.argv[1]
ms = {}
for f in sorted(glob.glob(os.path.join(out, "[AB][0-9].log"))):
    for line in open(f):
        if line.startswith("{") and '"ms_per_step"' in line:
            ms[os.path.basename(f)[:-4]] = json.loads(line)
a = [v["ms_per_step"] for k, v in ms.items() if k[0] == "A"]
b = [v["ms_per_step"] for k, v in ms.items() if k[0] == "B"]
print("A ms_per_step", a, "B ms_per_step", b)
if a and b:
    print(f"every B at least 5 % below every A: {max(b) <= 0.95 * min(a)}  (max B / min A = {max(b) / min(a):.4f})")
load = lambda d: {os.path.basename(p)[:-4]: np.load(p) for p in glob.glob(os.path.join(out, d, "*.npy"))}
A1, A2, B1 = load("dump_A1"), load("dump_A2"), load("dump_B1")
rend_ok = all(np.array_equal(A1[k], B1[k]) for k in A1 if k.startswith("rend."))
print("rend.* identical A1 vs B1:", rend_ok, sorted(k for k in A1 if k.startswith("rend.") and not np.array_equal(A1[k], B1[k])))
rel = lambda x, y: float(np.linalg.norm((x - y).astype(np.float64)) / (np.linalg.norm(y.astype(np.float64)) + 1e-30))
worse = []
for k in sorted(A1):
    if k.startswith("grad."):
        aa, ab = rel(A2[k], A1[k]), rel(B1[k], A1[k])
        if ab > aa:
            worse.append((k, ab, aa))
print("grad.* with |B1 - A1| above |A2 - A1|:", len(worse), worse[:8])
EOF
