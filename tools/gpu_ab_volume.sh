#!/bin/bash
# A/B of the threshold search and the final volume against an earlier build, in one GPU session:
#   * bench.py --gpus 1 --no-cpu-baseline alternating between the two libraries (RUNS runs each, default 3),
#   * per-kernel CUDA times of one pipeline pass per build (tools/kernel_times.py, torch.profiler),
#   * --dump-outputs of both builds compared with array_equal, and the report fields th / volume / bisections.
# The earlier library is rho2sdf.jl_b200/libr2s_base.so; when it is absent it is built from the git ref given as $1 (git archive, as a
# hand-built gpu_ab_libs.sh variant).  Results go to OUT_DIR.  Usage: tools/gpu_ab_volume.sh OUT_DIR [base-ref]
set -u
ROOT=$(cd "$(dirname "$0")/.." && pwd); cd "$ROOT"
[ $# -ge 1 ] || { echo "usage: $0 OUT_DIR [base-ref]"; exit 2; }
OUT=$(mkdir -p "$1" && cd "$1" && pwd); shift
LIB=rho2sdf.jl_b200/libr2s.so; BASE=rho2sdf.jl_b200/libr2s_base.so; RUNS=${RUNS:-3}
TMP=$(mktemp -d); trap 'cp $TMP/libr2s_new.so $LIB 2>/dev/null; rm -rf $TMP' EXIT
if [ ! -f $BASE ]; then
  [ $# -ge 1 ] || { echo "no $BASE and no base ref given"; exit 2; }
  mkdir -p $TMP/src && git archive "$1" | tar -x -C $TMP/src && make -C $TMP/src/rho2sdf.jl_b200/csrc -j8 > $TMP/base_build.log 2>&1 && cp $TMP/src/rho2sdf.jl_b200/libr2s.so $BASE || { tail $TMP/base_build.log; exit 2; }
fi
cp $LIB $TMP/libr2s_new.so; cp $BASE $TMP/libr2s_base.so
use() { cp $TMP/libr2s_$1.so $LIB; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee $OUT/gpu.txt
for r in $(seq 1 $RUNS); do
  for arm in base new; do
    use $arm
    timeout 600 python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline > $OUT/bench_${arm}_$r.json 2> $OUT/bench_${arm}_$r.err; echo "bench $arm $r rc=$?"
  done
done
for arm in base new; do
  use $arm
  timeout 600 python bench.py --gpus 1 --steps 1 --warmup 1 --no-cpu-baseline --dump-outputs $TMP/dump_$arm > $OUT/dump_${arm}.json 2> $OUT/dump_${arm}.err; echo "dump $arm rc=$?"
  timeout 600 python tools/kernel_times.py > $OUT/kernels_${arm}.txt 2> $OUT/kernels_${arm}.err; echo "kernel times $arm rc=$?"
done
use new
python - $OUT $TMP <<'PY'
import glob, json, os, statistics, sys
import numpy as np
out, tmp = sys.argv[1], sys.argv[2]
def last(p):
    return json.loads(open(p).read().strip().splitlines()[-1])
res = {}
for arm in ("base", "new"):
    lines = [last(p) for p in sorted(glob.glob(os.path.join(out, "bench_%s_*.json" % arm)))]
    ms = [d["ms_per_step"] for d in lines]
    st = {k: [d["stages_ms"][k] for d in lines] for k in lines[0]["stages_ms"]}
    res[arm] = {"ms_per_step": ms, "median": statistics.median(ms), "spread": max(ms) - min(ms),
                "stages_median": {k: statistics.median(v) for k, v in st.items()}, "stages_spread": {k: max(v) - min(v) for k, v in st.items()},
                "report": {k: lines[-1]["report"][k] for k in ("th", "volume", "bisections")}}
same = {}
for name in ("sdf_dists", "fine_sdf"):
    a, b = np.load(os.path.join(tmp, "dump_base", name + ".npy")), np.load(os.path.join(tmp, "dump_new", name + ".npy"))
    same[name] = bool(a.shape == b.shape and np.array_equal(a, b))
rb, rn = last(os.path.join(out, "dump_base.json"))["report"], last(os.path.join(out, "dump_new.json"))["report"]
same["report_th_volume_bisections"] = all(rb[k] == rn[k] for k in ("th", "volume", "bisections")) and res["base"]["report"] == res["new"]["report"]
summary = {"gpu": open(os.path.join(out, "gpu.txt")).read().strip(), "runs": res, "identical": same,
           "gain_ms": res["base"]["median"] - res["new"]["median"],
           "stage_gain_ms": {k: res["base"]["stages_median"][k] - res["new"]["stages_median"][k] for k in res["base"]["stages_median"]}}
json.dump(summary, open(os.path.join(out, "summary.json"), "w"), indent=1)
print(json.dumps(summary, indent=1))
PY
