#!/bin/bash
# A/B of alternative builds of libcq.so on the device-resident bench line, one box, back to back.
#   build the variants here (no GPU needed), e.g.
#     make -C swift-game-engine_b200/csrc clean; make -C swift-game-engine_b200/csrc -j8 EXTRA="-DCQ_WALK_FILL=96"
#     cp swift-game-engine_b200/csrc/libcq.so swift-game-engine_b200/csrc/libcq_r2.so      (*.so travels with gpurun)
#   then on the GPU box:   bash tools/ab_variants.sh "hulls terrain" libcq.so libcq_r2.so ...
# Every run is `bench.py --mesh M --no-cpu-baseline` with CQ_LIB pointing at the build; prints value and ms/step per run.
MESHES=${1:-hulls}
shift
D=swift-game-engine_b200/csrc
mkdir -p gpurun_out
for M in $MESHES; do
  for L in "$@"; do
    tag=$(basename "$L" .so)
    CQ_LIB=$D/$L timeout 40 python bench.py --mesh "$M" --no-cpu-baseline --no-extras > "gpurun_out/ab_${M}_${tag}.json" 2> "gpurun_out/ab_${M}_${tag}.err"
  done
done
python - <<'PY'
import glob, json
for f in sorted(glob.glob("gpurun_out/ab_*.json")):
    try:
        d = json.loads(open(f).read().strip().splitlines()[-1])
        print(f, "%.1f M/s  %.3f ms/step  e2e %.1f M/s" % (d["value"] / 1e6, d["ms_per_step"], d["e2e"]["value"] / 1e6))
    except Exception as e:
        print(f, "ERR", e)
PY
