#!/bin/bash
# One gpurun call, many artefacts (GPU slots are scarce): usage  tools/gpu_batch.sh "<stages>" <tag>
#   T tests   S dcn sweep   B bench (inference)   R bench --mode train   N ncu captures   C other configs   P role timing
stages="$1"; tag="${2:-r02}"
mkdir -p gpurun_out
if [[ "$stages" == *T* ]]; then
  timeout 1200 python -m pytest tests -m gpu -q 2>&1 | tail -40 > gpurun_out/${tag}_pytest_gpu.log; tail -4 gpurun_out/${tag}_pytest_gpu.log
fi
if [[ "$stages" == *S* ]]; then
  timeout 400 python tools/dcn_sweep.py --n 28 --sigmas 0.02,3,10 2>&1 | grep timing | cut -c1-220      # modes pair,fused; dcn_sweep.json
fi
if [[ "$stages" == *P* ]]; then
  timeout 200 python tools/dp_prof.py 28 0.02 0,127 2>&1 | cut -c1-400 | tee gpurun_out/${tag}_dcn_pair_role_timing.txt
fi
if [[ "$stages" == *B* ]]; then
  timeout 900 python bench.py > gpurun_out/${tag}_bench_n1.json 2> gpurun_out/${tag}_bench_n1.err; tail -c 400 gpurun_out/${tag}_bench_n1.err
  python - <<PY
import json
try:
    d=json.loads([x for x in open("gpurun_out/${tag}_bench_n1.json") if x.startswith("{")][-1])
    print("bench", d["value"], d["ms_per_step"], "e2e", d["e2e"]["value"], "b1", d.get("latency_b1",{}).get("value"), d["clocks"])
    print("cpu", d.get("cpu_baseline")); print("ref_cuda", d.get("ref_cuda")); print("dcn", d.get("roofline_dcn"))
    print("roofline", {k: d["roofline"][k] for k in ("achieved", "frac", "traffic")})
    print({k:(v["ms"],v["tflops"]) for k,v in d["kernel_shares"].items()})
except Exception as e: print("bench parse error", e)
PY
fi
if [[ "$stages" == *R* ]]; then
  timeout 900 python bench.py --mode train > gpurun_out/${tag}_bench_train_n1.json 2> gpurun_out/${tag}_bench_train_n1.err; tail -c 600 gpurun_out/${tag}_bench_train_n1.err; cut -c1-1500 gpurun_out/${tag}_bench_train_n1.json
fi
if [[ "$stages" == *N* ]]; then
  EDVR_B200_DCN_SITE=pair timeout 600 ncu --set full --clock-control none --import-source on -k regex:dcn_pair -s 3 -c 1 -o gpurun_out/${tag}_ncu_dcn_pair python tools/one_site.py 4 180 320 128 8 0.02 2>&1 | tail -2
  EDVR_BENCH_PROFILING=1 timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 1200 --csv --log-file gpurun_out/${tag}_ncu_launches_bench.csv python bench.py --steps 2 --warmup 3 > /dev/null 2>&1; wc -l gpurun_out/${tag}_ncu_launches_bench.csv
fi
if [[ "$stages" == *C* ]]; then
  timeout 900 python tools/bench_configs.py 2>&1 | tail -25; cp gpurun_out/bench_configs.json gpurun_out/${tag}_bench_configs.json 2>/dev/null
fi
