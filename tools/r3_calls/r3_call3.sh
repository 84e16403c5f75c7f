#!/bin/bash
# Round-3 GPU call 3: the shipped form (decided bisection steps + FIN reuse in the plain-walk kernels only, after calls 1-2).
# libcq_base.so = the parent commit's sources built with tools/build_variant.sh base ""; libcq.so = this tree (build());
# libcq_nofin.so / libcq_nodec.so: the call-1 sources with the FIN reuse / the decided-step loop compiled out (a temporary
# switch, not kept).  (Call 2, the same variants alone, never got a GPU slot; it is folded in here.)
# Card and power limit; parity (pytest -m gpu) and smoke on the new build; the headline's records of both builds
# (--dump-outputs) compared byte by byte; same-box A/B, alternated three times: headline (hulls), terrain, render, C2, C4.
O=$(realpath -m "${1:?usage: $0 OUTPUT_DIR}")
cd "$(dirname "$0")/../.."
export O
D=swift-game-engine_b200/csrc
mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/r3c3_gpu.txt
timeout 300 python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $O/r3c3_smoke.log 2>&1; echo "smoke rc=$?"; tail -2 $O/r3c3_smoke.log
timeout 1500 python -m pytest tests -m gpu -q -rf --no-header -p no:cacheprovider > $O/r3c3_pytest.log 2>&1
echo "pytest rc=$?"; tail -6 $O/r3c3_pytest.log
for L in base new; do
  lib=$D/libcq_$L.so; [ $L = new ] && lib=$D/libcq.so
  CQ_LIB=$lib timeout 300 python bench.py --no-cpu-baseline --no-extras --dump-outputs $O/r3c3_dump_$L > $O/r3c3_dump_$L.json 2> $O/r3c3_dump_$L.err
done
python - <<'PY'
import glob, json, os
a, b = os.environ["O"] + "/r3c3_dump_base", os.environ["O"] + "/r3c3_dump_new"
fs = sorted(os.listdir(a)) if os.path.isdir(a) else []
same = [open(f"{a}/{f}", "rb").read() == open(f"{b}/{f}", "rb").read() for f in fs]
print("dump files", len(fs), "byte-identical", sum(same), "differ", [f for f, s in zip(fs, same) if not s])
PY
rm -rf $O/r3c3_dump_base $O/r3c3_dump_new
run() { CQ_LIB=$D/$2 timeout 300 python bench.py $3 --no-cpu-baseline --no-extras > $O/r3c3_ab_$1_$4_$(basename $2 .so).json 2> /dev/null; }
for rep in 1 2 3; do
  for L in libcq_base.so libcq.so; do
    run hulls $L "--mesh hulls" $rep
    run terrain $L "--mesh terrain" $rep
    run render $L "--mesh render" $rep
    run c2 $L "--only c2" $rep
    run c4 $L "--only c4" $rep
  done
done
# the call-1 form (both halves in every kernel) with one half switched off, once each: where the staged-walk kernels lose
for L in libcq_nofin.so libcq_nodec.so; do
  for M in terrain render; do run $M $L "--mesh $M" 1; done
  run c2 $L "--only c2" 1; run c4 $L "--only c4" 1
done
python - <<'PY'
import glob, json, os
def flags(d, p=""):
    out = []
    for k, v in d.items():
        if isinstance(v, dict): out += flags(v, p + k + ".")
        elif isinstance(v, bool) and ("match" in k or "bit_identical" in k or "identical" in k): out.append((p + k, v))
    return out
for f in sorted(glob.glob(os.environ["O"] + "/r3c3_ab_*.json")) + sorted(glob.glob(os.environ["O"] + "/r3c3_dump_*.json")):
    try:
        d = json.loads(open(f).read().strip().splitlines()[-1])
        pq = d.get("roofline", {}).get("per_query", {})
        bad = [k for k, v in flags(d) if not v]
        print("%-44s %9.1f M/s %8.3f ms/step  evals/q %7.2f cands/q %6.2f nodes/q %6.2f  flags %d bad %s" % (
            f.split("/")[-1], d["value"] / 1e6, d["ms_per_step"], pq.get("distance_evals", -1), pq.get("candidates", -1),
            pq.get("nodes", -1), len(flags(d)), bad))
    except Exception as ex:
        print(f, "ERR", ex)
PY
