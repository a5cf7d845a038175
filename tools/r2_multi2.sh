mkdir -p gpurun_out
( time timeout 600 python -m pytest tests/test_gpu_multi.py -m gpu -q ) > gpurun_out/r2m_tests2.log 2>&1; tail -6 gpurun_out/r2m_tests2.log
( timeout 600 python -m pytest tests/test_gpu_fused.py tests/test_gpu_capi_parity.py -m gpu -x -q ) > gpurun_out/r2m_tests_fused.log 2>&1; tail -2 gpurun_out/r2m_tests_fused.log
for wl in config5 config4; do python bench.py --workload $wl --no-cpu --no-e2e --no-extra --verify-windows 32 --steps 20 > gpurun_out/r2m_popc_$wl.json 2> gpurun_out/r2m_popc_$wl.err; done
python tools/show_bench.py gpurun_out/r2m_popc_config5.json gpurun_out/r2m_popc_config4.json
python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus 2 --steps 30 --warmup 3 --no-cpu > gpurun_out/r2m_bench_n2.json 2> gpurun_out/r2m_bench_n2.err; tail -2 gpurun_out/r2m_bench_n2.err | cut -c1-300
