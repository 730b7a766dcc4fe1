#!/bin/bash
# A/B of variant builds of the streaming prepass (column index layout, fill-mean division, timing-only ablations):
# c3 and c2 bench lines (optionally c4) per variant, the variants ALTERNATED round by round in one invocation so that drift of
# the shared machine spreads over all of them.  Kernel times are the bench line's `kernels` table (CUDA events).
# A variant is build_variants/libreal3d_b200_<name>.so (loaded through R3D_LIB_PATH), or a directory build_variants/<name>
# holding a whole tree, e.g. a checkout of the parent commit with its library built in place (needed when the Python
# side binds symbols the other build lacks).  Build the variants first (no GPU needed), e.g.
#   bash tools/build_variant.sh base                                  # the commit under test
#   bash tools/build_variant.sh ablA -DR3D_ABLATE_COL_IDX             # timing only: outputs are wrong
#   bash tools/build_variant.sh g1 -DR3D_COL_GROUP=1
# usage: bash tools/gpu_prepass_ab.sh "base ablA g1" [rounds=3] [configs="c3 c2"] [out=prepass_ab]
#   -> <out>/pab_<config>_<variant>_r<round>.json, one summary line per run on stdout
VARIANTS=${1:-base}
ROUNDS=${2:-3}
CONFIGS=${3:-"c3 c2"}
OUT=${4:-prepass_ab}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
for r in $(seq 1 "$ROUNDS"); do
  for c in $CONFIGS; do
    for v in $VARIANTS; do
      out=$OUT/pab_${c}_${v}_r$r
      if [ -d "build_variants/$v" ]; then           # a whole tree (e.g. the parent commit, library built in it)
        (cd "build_variants/$v" && timeout 300 python bench.py --config "$c" --side-configs '' --no-cpu-baseline) \
            > "$out.json" 2> "$out.err"
      else
        R3D_LIB_PATH=build_variants/libreal3d_b200_$v.so timeout 300 python bench.py --config "$c" --side-configs '' \
            --no-cpu-baseline > "$out.json" 2> "$out.err"
      fi
      python - "$out.json" "$c" "$v" "$r" <<'P'
import json, sys
path, c, v, r = sys.argv[1:]
try:
    d = json.loads(open(path).read().strip().splitlines()[-1])
except (IndexError, ValueError):
    print(c, v, "r" + r, "FAILED (see the .err file)")
    sys.exit(0)
k = {n: t["ms_per_step"] for n, t in d["kernels"].items()}
pick = ["ingest_spherical", "index_build", "scatter_project", "close_fill_full", "scan_walk"]
print(c, v, "r" + r, "value", round(d["value"]), "ms_per_step", round(d["ms_per_step"], 4),
      "single_batch_ms", round(d["single_batch_ms"], 4), " ".join(f"{n}={k.get(n)}" for n in pick))
P
    done
  done
done
