#!/bin/bash
# 8-GPU evidence: a single-GPU bench on the SAME box first (same-box scaling efficiency), then the 8-rank bench.
O=gpurun_out
python bench.py --gpus 1 --steps 20 --warmup 3 --skip-cpu --skip-shim --skip-tc --skip-kdtree > $O/r2_bench_n1_samebox.json 2> $O/bench_n1s.err
python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus 8 --steps 20 --warmup 3 > $O/r2_bench_n8.json 2> $O/bench_n8.err
tail -2 $O/bench_n8.err
python - <<'PY'
import json
a=json.loads(open("gpurun_out/r2_bench_n1_samebox.json").read())
d=json.loads(open("gpurun_out/r2_bench_n8.json").read())
print("N=1 same box: value",a["value"],"ms_per_step",a["ms_per_step"],"e2e",a["e2e"]["value"],"depth",a["e2e"]["depth_input"]["value"],"depth idx",a["e2e"]["depth_input_idx_only"]["value"], "closed depth", a["e2e_closed_loop"]["c_loop_depth_input"]["frames_per_s"])
print("N=8: value",d["value"],"ms_per_step",d["ms_per_step"], "eff", d["value"]/8/a["value"])
print("us per step per rank",[round(x*1e3,2) for x in d["timed_region"]["ms_per_step_per_rank"]])
print("e2e",d["e2e"]["value"], "depth", d["e2e"]["depth_input"]["value"], "depth idx", d["e2e"]["depth_input_idx_only"]["value"])
print("closed", {k:round(v.get("frames_per_s")) for k,v in d["e2e_closed_loop"].items()})
print("batched", d["batched_sequences"]["frames_per_s"], "nn", d["nn"]["query_ms"], d["nn"]["build_ms"], d["nn"].get("weak_scaling"))
PY
