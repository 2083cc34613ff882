# Run-to-run reproducibility and speed of the two partial-gradient reductions of the tc SGD step, on the bench workload:
# bench.py (fixed-order sum of the per-CTA partials) and bench.py --atomic-reduce (float atomics into one L2 vector),
# alternated, each run dumping its last timed iteration (--dump-outputs); the dumps are compared and then deleted.
# usage: bash profiles/scripts/reduction_reproducibility.sh <output dir>   -> <output dir>/reduction_reproducibility.txt
O=${1:?output dir}; mkdir -p $O
for run in fixed1 atomic1 fixed2 atomic2; do
  flag=""; case $run in atomic*) flag=--atomic-reduce;; esac
  python bench.py --steps 20 --warmup 3 --no-cpu-baseline --no-supplementary $flag --dump-outputs $O/dump_$run \
    > $O/bench_$run.json 2> $O/bench_$run.err || exit 1
done
python - "$O" <<'EOF' > $O/reduction_reproducibility.txt
import json, os, subprocess, sys
import numpy as np
O = sys.argv[1]
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print(f"GPU: {gpu}")
print("bench.py --steps 20 --warmup 3 --no-cpu-baseline --no-supplementary [--atomic-reduce] --dump-outputs DIR, runs in this order:")
print(f"{'run':8s} {'M agent-steps/s':>16s} {'ms/iteration':>13s} {'us/SGD step':>12s}  reduction")
for run in ("fixed1", "atomic1", "fixed2", "atomic2"):
    d = json.loads(open(f"{O}/bench_{run}.json").read().strip().splitlines()[-1])
    print(f"{run:8s} {d['value'] / 1e6:16.2f} {d['ms_per_step']:13.3f} {d['roofline']['us_per_sgd_step']:12.2f}  "
          f"{d['impl_detail']['partial_gradient_reduce']}")
print("\ndumps of the last timed iteration (29th learner iteration of the run), max |a - b| / max |b| per file:")
for a, b in (("fixed1", "fixed2"), ("atomic1", "atomic2"), ("fixed1", "atomic1")):
    diffs = {}
    for f in sorted(os.listdir(f"{O}/dump_{a}")):
        x, y = np.load(f"{O}/dump_{a}/{f}"), np.load(f"{O}/dump_{b}/{f}")
        diffs[f[:-4]] = float(np.abs(x.astype(np.float64) - y).max() / max(np.abs(y).max(), 1e-30))
    nz = {k: v for k, v in diffs.items() if v}
    print(f"{a} vs {b}: {len(nz)} of {len(diffs)} arrays differ" + (":" if nz else " (bit-identical)"))
    for k, v in sorted(nz.items(), key=lambda kv: -kv[1]):
        print(f"    {k:24s} {v:.2e}")
EOF
rm -rf $O/dump_*
cat $O/reduction_reproducibility.txt
