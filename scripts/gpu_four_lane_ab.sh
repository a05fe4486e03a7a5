# A/B of the four-lane class <4,25> (reads of 81-100 bases) against the same tree built without it
# (-DDFB_NARROW_GROUPS=0, where those reads run at <8,13>), in one GPU session:
#   - bench.py --steps 10 --no-secondary --no-cpu-baseline, both libraries alternating, three rounds each;
#   - bench.py --dump-outputs of both builds on the bench workload, compared file for file;
#   - one full bench.py of the new build (secondary legs).
# Card name, power limit and SM clock are recorded beside the numbers.
# usage: bash scripts/gpu_four_lane_ab.sh OUT_DIR   (build the default library first; the variant is compiled into a
# temporary directory that is removed at exit)
set -u
cd "$(dirname "$0")/.."
OUT=${1:?usage: gpu_four_lane_ab.sh OUT_DIR}
mkdir -p "$OUT"
VAR=$(mktemp -d)
trap 'rm -rf "$VAR"' EXIT
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-O2,-fvisibility=hidden \
     -DDFB_NARROW_GROUPS=0 -c defuse_b200/csrc/dfb_api.cu -o "$VAR/dfb_api.o" || exit 1
g++ -shared -o "$VAR/libdefuse_b200_narrow0.so" "$VAR/dfb_api.o" defuse_b200/build/dfb_micro.o \
    -L/usr/local/cuda/lib64 -lcudart_static -ldl -lrt -lpthread || exit 1
NEW=$PWD/defuse_b200/libdefuse_b200.so
OLD=$VAR/libdefuse_b200_narrow0.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > "$OUT/gpu.csv" 2>&1
Q="--steps 10 --no-secondary --no-cpu-baseline"
for round in 1 2 3; do
  for v in old new; do
    lib=$OLD; [ $v = new ] && lib=$NEW
    DFB_LIB_PATH=$lib timeout 300 python bench.py $Q > "$OUT/bench_${v}_$round.json" 2> "$OUT/bench_${v}_$round.err"
    echo "${v}_$round rc=$?"
  done
done
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv,noheader >> "$OUT/gpu.csv" 2>&1
for v in old new; do
  lib=$OLD; [ $v = new ] && lib=$NEW
  DFB_LIB_PATH=$lib timeout 300 python bench.py --steps 1 --warmup 1 --no-secondary --no-cpu-baseline --no-sharded \
      --dump-outputs "$OUT/dump_$v" > "$OUT/dump_$v.json" 2> "$OUT/dump_$v.err"
  echo "dump_$v rc=$?"
done
python - "$OUT" <<'EOF'
import glob, json, os, sys
import numpy as np
out = sys.argv[1]
names = sorted(os.path.basename(f) for f in glob.glob(os.path.join(out, "dump_old", "*.npy")))
same = names == sorted(os.path.basename(f) for f in glob.glob(os.path.join(out, "dump_new", "*.npy")))
diff = [n for n in names if not np.array_equal(np.load(os.path.join(out, "dump_old", n)), np.load(os.path.join(out, "dump_new", n)))]
rows = {}
for v in ("old", "new"):
    for r in (1, 2, 3):
        try:
            j = json.loads(open(os.path.join(out, "bench_%s_%d.json" % (v, r))).read().strip().splitlines()[-1])
        except Exception as e:  # a failed run is reported, not hidden
            rows.setdefault(v, []).append({"error": str(e)})
            continue
        rf = j.get("roofline", {})
        rows.setdefault(v, []).append({"ms_per_step": j.get("ms_per_step"), "sweep_ms": rf.get("kernel_ms"),
                                       "probe_ms": rf.get("probe_sweep_ms"), "results": j.get("results"),
                                       "e2e": j.get("e2e"), "clocks": j.get("clocks")})
summary = {"dump_files": names, "dump_same_names": same, "dump_differing": diff, "runs": rows}
json.dump(summary, open(os.path.join(out, "summary.json"), "w"), indent=1, default=str)
print("dump files %d, same names %s, differing %s" % (len(names), same, diff))
for v, rs in rows.items():
    print(v, ["%.3f/%.3f/%.3f" % (r["ms_per_step"], r["sweep_ms"], r["probe_ms"]) if "ms_per_step" in r else r for r in rs],
          "(step / first sweep / probe sweep, ms)")
print("results equal:", len({json.dumps(r.get("results"), sort_keys=True) for rs in rows.values() for r in rs}) == 1)
EOF
DFB_LIB_PATH=$NEW timeout 900 python bench.py > "$OUT/bench_full_new.json" 2> "$OUT/bench_full_new.err"
echo "full_new rc=$?"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv,noheader >> "$OUT/gpu.csv" 2>&1
