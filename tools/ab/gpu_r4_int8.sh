#!/bin/bash
# int8 prefilter shadow vs bf16 on one GPU: the GPU suite, then `bench.py --no-cpu-baseline` alternating AUTO (int8 on
# the isotropic bench rows) with `--opt shadow=1` (bf16) three times on the headline config c4, once each on
# c2 / c3 / the common-mean rows, every pair with --dump-outputs (the two arms must agree bit for bit).
# bench.py's roofline.achieved assumes 1536 streamed bytes per row; this script reports the true rate of each arm
# from score_ms and the bytes the scoring kernel streams per row (bf16 1536, int8 768 + 4/32).
OUT=${1:?usage: bash tools/ab/gpu_r4_int8.sh OUTPUT_DIR}
export OUT
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
if [ "${SKIP_TESTS:-0}" != 1 ]; then
  timeout 900 python -m pytest tests -q -m gpu > "$OUT"/r4_tests.log 2>&1; echo "tests rc=$?"; tail -3 "$OUT"/r4_tests.log
fi
run() { tag=$1; shift
  timeout 600 python bench.py --gpus 1 --no-cpu-baseline --dump-outputs "$OUT"/dump_$tag "$@" > "$OUT"/r4_$tag.json 2> "$OUT"/r4_$tag.err
  echo "$tag rc=$?"
  TAG=$tag python - <<'PY'
import json, os
tag, out = os.environ["TAG"], os.environ["OUT"]
try:
    j = json.load(open(f"{out}/r4_{tag}.json"))
    r = j.get("roofline") or {}; c = j.get("check") or {}
    rows, bpr = r.get("rows_per_launch"), (1536 if "bf16" in tag else 768 + 4 / 32)
    ms = r.get("ms_per_launch")
    true_tbs = rows * bpr / (ms * 1e-3) / 1e12 if rows and ms else None
    print(tag, "q/s", round(j["value"]), "ms/step", round(j["ms_per_step"], 3), "score ms/launch", ms,
          "true TB/s", true_tbs and round(true_tbs, 2), "sustained", j.get("sustained"), "clocks", j.get("clocks"),
          "check", {k: c.get(k) for k in ("oracle_violations", "fallback_queries", "overflow_redo_ok",
                                          "tensor_engine_equals_simt_engine_4q")})
except Exception as e:
    print(tag, "FAILED", e); print(open(f"{out}/r4_{tag}.err").read()[-3000:])
PY
}
same() {
  python - "$1" "$2" "$OUT" <<'PY'
import sys, numpy as np
a, b, out = sys.argv[1:4]
ok = all(np.array_equal(np.load(f"{out}/dump_{a}/{f}"), np.load(f"{out}/dump_{b}/{f}")) for f in ("scores.npy", "ids.npy"))
print("outputs", a, "==", b, ok)
PY
}
for i in $(seq 1 "${REPEATS:-3}"); do
  chk=""; [ $i -gt 1 ] && chk="--no-check"
  run c4_int8_$i $chk
  run c4_bf16_$i $chk --opt shadow=1
  same c4_int8_$i c4_bf16_$i
done
run c2_int8 --config c2 --no-check; run c2_bf16 --config c2 --no-check --opt shadow=1; same c2_int8 c2_bf16
run c3_int8 --config c3 --no-check; run c3_bf16 --config c3 --no-check --opt shadow=1; same c3_int8 c3_bf16
run aniso_auto --data aniso --no-check; run aniso_bf16 --data aniso --no-check --opt shadow=1; same aniso_auto aniso_bf16
