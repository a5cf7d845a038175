# round 2, call 2: GPU tests on the rewritten fused kernels, then a ring-geometry sweep (warps x tile blocks x depth)
mkdir -p gpurun_out
( time timeout 900 python -m pytest tests -m gpu -x -q ) > gpurun_out/r2b_tests.log 2>&1; tail -6 gpurun_out/r2b_tests.log
run() {  # workload tag env...
  wl=$1; tag=$2; shift 2
  env "$@" timeout 200 python bench.py --workload $wl --no-cpu --no-e2e --steps 10 > gpurun_out/r2b_${wl}_$tag.json 2> gpurun_out/r2b_${wl}_$tag.err
  python - "$wl" "$tag" <<'PY'
import json,sys
wl,tag=sys.argv[1:3]
try:
    j=json.load(open(f"gpurun_out/r2b_{wl}_{tag}.json")); k=j["roofline"]["kernel_ms_all"]
    print(f"{wl} {tag:14s} step {j['ms_per_step']:.4f} ms  {j['value']/1e9:6.2f} G/s  k1 {k['k1_count']:.4f} fin {k['finalize']:.4f} k3 {k['k3_small']:.4f} launches {j['gpu_launches_per_step']}")
except Exception as e:
    print(wl, tag, "ERR", e, open(f"gpurun_out/r2b_{wl}_{tag}.err").read()[-300:])
PY
}
run config5 default X=1
run config4 default X=1
for w in 8 10 12 14; do for t in 1 2; do for d in 1 2; do
  run config5 w${w}t${t}d${d} TDSFS_K1_WARPS=$w TDSFS_K1_TILE=$t TDSFS_K1_DEPTH=$d
done; done; done
for w in 10 12 14 16; do for t in 1 2 4; do for d in 1 2; do
  run config4 w${w}t${t}d${d} TDSFS_K1_WARPS=$w TDSFS_K1_TILE=$t TDSFS_K1_DEPTH=$d
done; done; done
