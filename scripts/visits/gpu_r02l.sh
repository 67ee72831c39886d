#!/bin/bash
# 2-GPU visit: the new speculation tests + the whole 1-GPU suite (on GPU 0), sharded parity tests at world 2, C3 bench at N=2 and N=1 shard size.
TAG=${1:-r02l}
mkdir -p gpurun_out
timeout 1200 python -m pytest tests -m gpu -q -x --deselect tests/test_gpu_multi.py > gpurun_out/${TAG}_pytest.log 2>&1; echo "pytest rc=$?" | tee -a gpurun_out/${TAG}_pytest.log; tail -15 gpurun_out/${TAG}_pytest.log
bash scripts/gpu_multi.sh ${TAG} "" "2"
timeout 600 python bench.py --workload C3r8 --steps 50 --warmup 5 --no-e2e --no-cpu-baseline --no-compact > gpurun_out/${TAG}_bench_c3r8_f32.json 2> gpurun_out/${TAG}_bench_c3r8_f32.err
timeout 600 python bench.py --steps 20 --warmup 5 --no-e2e --no-cpu-baseline --no-compact > gpurun_out/${TAG}_bench_c3_f32.json 2> gpurun_out/${TAG}_bench_c3_f32.err
python - <<PY
import json
for f in ("c3r8_f32","c3_f32"):
    try:
        d=json.loads([l for l in open("gpurun_out/${TAG}_bench_%s.json"%f) if l.startswith("{")][-1])
        print(f, "it/s %.1f ms %.4f"%(d["value"], d["ms_per_step"]), {k:round(v,4) for k,v in d["roofline"]["kernel_ms"].items()}, "kl", d["check"]["kl_raw"], d["check"]["bisect_its_H"])
    except Exception as e: print(f, "parse failed", e)
PY
