#!/bin/bash
# A/B of the two-team (producer / consumer) CTA inflate kernel against the parent commit, in one GPU session.
# The parent tree is an untracked export at _parent/ (git archive of the parent commit).  Results go to the directory given as
# the second argument.
#   tools/gpu_pipe_ab.sh quick   parity of the CTA kernel + kernel-alone timing and phase profile of both trees, payload-size variants
#   tools/gpu_pipe_ab.sh full    whole GPU suite + smoke, bench.py config 2 alternating 3 x per tree, output dumps compared,
#                                configs 3 / 4 / 5 and FASTQ once per tree
#   tools/gpu_pipe_ab.sh all     both (stops after the parity check if it fails)
#   tools/gpu_pipe_ab.sh suite | bench | rest   the parts of `full` (GPU suite + smoke / config 2 A/B / dumps, configs, FASTQ),
#                                for sessions shorter than the whole
set -u
mode=${1:-quick}
OUT=$(realpath -m "${2:?usage: tools/gpu_pipe_ab.sh MODE OUTPUT_DIR}"); mkdir -p "$OUT"
NEW=$PWD; OLD=$PWD/_parent
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv | tee "$OUT/gpu_info.csv"
(cd "$NEW" && python -c "import __graft_entry__ as g; g.build()" > "$OUT/build_new.log" 2>&1) || { echo "new build failed"; tail -20 "$OUT/build_new.log"; exit 1; }
(cd "$OLD" && python -c "import __graft_entry__ as g; g.build()" > "$OUT/build_old.log" 2>&1) || { echo "parent build failed"; tail -20 "$OUT/build_old.log"; exit 1; }

prof() {   # tree label [env...]
  local tree=$1 label=$2; shift 2
  echo "== $label"
  (cd "$tree" && env BAMSCAN_DEBUG_FLAGS=16 "$@" timeout 300 python tools/prof_inflate.py 4000000 2>&1 | tail -2) | tee -a "$OUT/prof_$mode.log"
}

if [ "$mode" = quick ] || [ "$mode" = all ]; then
  timeout 900 python -m pytest -x -q -m gpu tests/test_inflate_batched_resolve.py tests/test_gpu_parity.py -k "cta_per_member or batched" > "$OUT/parity_quick.log" 2>&1
  rc=$?; echo "parity rc=$rc"; tail -3 "$OUT/parity_quick.log"; [ $rc = 0 ] || exit 1
  for r in 1 2; do prof "$OLD" "parent plain"; prof "$NEW" "new plain"; done
  prof "$OLD" "parent prof" BAMSCAN_ICTA_PROF=1
  prof "$NEW" "new prof" BAMSCAN_ICTA_PROF=1
  # payload buffer size alone in the parent kernel, then the new kernel's payload / list split
  for kb in 20; do
    rm -rf /tmp/pv; cp -r "$OLD" /tmp/pv
    sed -i "s/(NT <= 384 ? 29 : 27) \* 1024/$kb * 1024/" /tmp/pv/datafusion-bio-formats_b200/csrc/kernels_inflate_cta.cuh
    rm -f /tmp/pv/datafusion-bio-formats_b200/libbamscan.so; make -C /tmp/pv/datafusion-bio-formats_b200/csrc > /dev/null 2>&1 || echo "build pv $kb failed"
    prof /tmp/pv "parent PAY ${kb} KB" BAMSCAN_ICTA_PROF=1
  done
  for kb in 24; do
    rm -rf /tmp/pv; cp -r "$NEW" /tmp/pv; rm -rf /tmp/pv/_parent
    rm -f /tmp/pv/datafusion-bio-formats_b200/libbamscan.so
    make -C /tmp/pv/datafusion-bio-formats_b200/csrc CXXFLAGS="-O3 -std=c++17 -Xcompiler -fPIC,-Wall,-Wno-unused-function -lineinfo -DBAMSCAN_ICTA_PAY_KB=$kb" > /dev/null 2>&1 || echo "build nv $kb failed"
    prof /tmp/pv "new PAY ${kb} KB" BAMSCAN_ICTA_PROF=1
  done
  rm -rf /tmp/pv
  [ "$mode" = quick ] && exit 0
fi

# ---- full ----
if [ "$mode" = all ] || [ "$mode" = full ] || [ "$mode" = suite ]; then
bash tests/run_gpu_tests.sh 2>&1 | tail -3
python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke rc=$?"; tail -3 "$OUT/smoke.log" | cut -c1-200
fi
if [ "$mode" = all ] || [ "$mode" = full ] || [ "$mode" = bench ]; then
for r in 1 2 3; do
  for t in old new; do
    tree=$NEW; [ $t = old ] && tree=$OLD
    (cd "$tree" && timeout 900 python bench.py --gpus 1 --steps 5 --warmup 3 > "$OUT/bench_${t}_$r.json" 2> "$OUT/bench_${t}_$r.err")
    python - "$OUT/bench_${t}_$r.json" $t $r <<'PY'
import json, sys
d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
print(sys.argv[2], sys.argv[3], "value", round(d["value"] / 1e6, 2), "M reads/s | kernel alone",
      d["roofline"].get("kernel_alone", {}).get("ms_per_launch"), "ms | inflate stage", d.get("stage_ms_rank0", {}).get("inflate"),
      "ms | verify", d.get("verify", {}).get("result"))
PY
  done
done
fi
[ "$mode" = suite ] || [ "$mode" = bench ] && exit 0
if [ "$mode" != all ]; then
  prof "$OLD" "parent plain"; prof "$NEW" "new plain"
  prof "$OLD" "parent prof" BAMSCAN_ICTA_PROF=1; prof "$NEW" "new prof" BAMSCAN_ICTA_PROF=1
fi
for t in old new; do
  tree=$NEW; [ $t = old ] && tree=$OLD
  (cd "$tree" && timeout 900 python bench.py --gpus 1 --steps 2 --warmup 1 --dump-outputs "$OUT/dump_$t" > "$OUT/bench_dump_$t.json" 2>/dev/null)
done
python - "$OUT/dump_old" "$OUT/dump_new" <<'PY'
import sys, hashlib
from pathlib import Path
a, b = Path(sys.argv[1]), Path(sys.argv[2])
fa = sorted(p.relative_to(a) for p in a.rglob("*.npy")); fb = sorted(p.relative_to(b) for p in b.rglob("*.npy"))
same = fa == fb and all((a / f).read_bytes() == (b / f).read_bytes() for f in fa)
print("dump files", len(fa), len(fb), "byte-identical" if same else "DIFFER")
PY
for t in old new; do
  tree=$NEW; [ $t = old ] && tree=$OLD
  echo "== configs $t"; (cd "$tree" && timeout 900 python tools/measure_configs.py 2>&1 | tail -12) | tee "$OUT/configs_$t.md"
  echo "== fastq $t"; (cd "$tree" && timeout 600 python tools/measure_fastq.py 2>&1 | tail -6) | tee "$OUT/fastq_$t.md"
done
