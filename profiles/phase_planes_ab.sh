#!/bin/bash
# Quarter-pel phase planes (X265CU_ME_PHASEPLANES) A/B on one B200, one call: alternating c3 runs of both arms with output
# dumps compared, the job order under planes, c4 per arm, the default c3 line (CPU parity + pred_cost) and the plane-build
# time.  Usage: profiles/phase_planes_ab.sh OUT_DIR (raw JSON lines and logs go there; committed copies:
# profiles/phase_planes/).  Run from the repository root on the GPU machine.
set -u
OUT=${1:?usage: profiles/phase_planes_ab.sh OUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/card.csv"
FAST="--gpus 1 --steps 10 --warmup 3 --no-cpu --no-primitives --no-pred"
for i in 1 2 3; do
  for m in 0 1; do
    rm -rf "$OUT/dump_${m}_$i"
    X265CU_ME_PHASEPLANES=$m python bench.py --config c3 $FAST --dump-outputs "$OUT/dump_${m}_$i" > "$OUT/c3_pp${m}_run$i.json" 2> "$OUT/c3_pp${m}_run$i.err"
    echo "c3 planes=$m run $i rc=$?"
  done
done
for o in 0 1; do
  X265CU_ME_PHASEPLANES=1 X265CU_ME_ORDER=$o python bench.py --config c3 $FAST > "$OUT/c3_pp1_order$o.json" 2> "$OUT/c3_pp1_order$o.err"
  echo "c3 planes=1 order=$o rc=$?"
done
for m in 0 1; do
  X265CU_ME_PHASEPLANES=$m python bench.py --config c4 $FAST > "$OUT/c4_pp$m.json" 2> "$OUT/c4_pp$m.err"
  echo "c4 planes=$m rc=$?"
done
python bench.py --gpus 1 > "$OUT/c3_default.json" 2> "$OUT/c3_default.err"
echo "c3 default rc=$?"
python - "$OUT" <<'PY'
import glob, json, os, sys
import numpy as np
out = sys.argv[1]
def last(p):
    return [json.loads(l) for l in open(p) if l.startswith("{")][-1]
# outputs of the two arms: identical
ref = None
for d in sorted(glob.glob(os.path.join(out, "dump_*"))):
    arrs = {os.path.basename(f): np.load(f) for f in sorted(glob.glob(os.path.join(d, "*.npy")))}
    if ref is None:
        ref = (d, arrs)
    assert arrs.keys() == ref[1].keys() and all(np.array_equal(arrs[k], ref[1][k]) for k in arrs), (d, ref[0])
print("dumps identical:", len(glob.glob(os.path.join(out, "dump_*"))), "runs,", len(ref[1]), "arrays each")
for cfg in ("c3",):
    for m in "01":
        v = [last(os.path.join(out, "%s_pp%s_run%d.json" % (cfg, m, i))) for i in (1, 2, 3)]
        ms = [x["ms_per_step"] for x in v]
        st = v[-1]["stages_ms"]
        print("%s planes=%s ms_per_step %s median %.3f spread %.3f | prechecks %.3f subpel %.3f search %.3f"
              % (cfg, m, ["%.3f" % x for x in ms], float(np.median(ms)), max(ms) - min(ms), st["me_prechecks"], st["me_subpel"], st["me_integer_search"]))
for o in "01":
    x = last(os.path.join(out, "c3_pp1_order%s.json" % o))
    print("c3 planes=1 X265CU_ME_ORDER=%s ms_per_step %.3f prechecks %.3f subpel %.3f" % (o, x["ms_per_step"], x["stages_ms"]["me_prechecks"], x["stages_ms"]["me_subpel"]))
for m in "01":
    x = last(os.path.join(out, "c4_pp%s.json" % m))
    print("c4 planes=%s ms_per_step %.3f prechecks %.3f subpel %.3f" % (m, x["ms_per_step"], x["stages_ms"]["me_prechecks"], x["stages_ms"]["me_subpel"]))
x = last(os.path.join(out, "c3_default.json"))
print("c3 default: ms_per_step %.3f checks_equal %s pred_cost.checks_equal %s" % (x["ms_per_step"], x.get("checks_equal"), (x.get("pred_cost") or {}).get("checks_equal")))
PY
rm -rf "$OUT"/dump_*
# plane-build time at c3 and c4 size (4 / 5 references, uniform-noise pictures, every reference's whole region)
python - <<'PY'
import sys
sys.path.insert(0, "tests")
import numpy as np
import x265_b200
from frame_helpers import make_field
cu = x265_b200.load()
for name, W, H, depth, refs in (("c3", 3840, 2160, 8, 4), ("c4", 3840, 2160, 10, 5)):
    an = x265_b200.Analyser(cu, W, H, depth=depth, numRefs=refs, method=3, subme=3, merange=57, rect=1, qp=30)
    rng = np.random.default_rng(1)
    dt = np.uint8 if depth == 8 else np.uint16
    for r in range(refs):
        an.set_ref(r, rng.integers(0, 1 << depth, (H, W)).astype(dt))
    fenc = rng.integers(0, 1 << depth, (H, W)).astype(dt)
    field = make_field(W, H, refs)
    an.load_inputs(fenc, field)
    t = []
    for i in range(6):
        an.run_resident(1)
        t.append(an.phase_planes_ms())
    print("%s plane build: %s ms (last 5 median %.3f); region ref0 %s" % (name, ["%.3f" % v for v in t], float(np.median(t[1:])), an.phase_region(0)))
    an.close()
PY
