#!/usr/bin/env python
"""BASELINE.json config 5: gym_carracing-shaped CNN encoder + DSAC-T heads, batch 1024, one B200 (reference
networks/cnn.py `type_2`, 3x96x96 observations).  Device-resident minibatches; prints one JSON line with steps/s, the
clocks during the timed region and, with --cpu, the oracle port on the host cores for the same step.

    python tools/bench_cnn.py [--batch 1024] [--steps 20] [--cpu] [--split]

--split times the split form instead of the fused call: compute_grads + apply per step (the same kernels as
dsact_cnn_step, in two calls; the path of the gradient-message seam).
"""
import argparse
import json
import os
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import torch  # noqa: E402

from bench import ClockSampler, cpu_model  # noqa: E402
from dsac_v2_b200 import synth  # noqa: E402
from dsac_v2_b200.engine_cnn import CnnEngine, make_cnn_config  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=1024)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--cpu", action="store_true")
ap.add_argument("--split", action="store_true")
a = ap.parse_args()
cfg = synth.CNN_CONFIGS["carracing"]
t = synth.CONV_TYPES[cfg["conv_type"]]
B = a.batch
c = make_cnn_config(cfg["obs_dim"], cfg["act_dim"], t["kernels"], t["channels"], t["strides"], t["heads"], max_batch=B)
lim = torch.full((cfg["act_dim"],), cfg["act_lim"])
eng = CnnEngine(c, torch.device("cuda", 0), lim, -lim)
eng.load_weights(synth.make_cnn_weights(cfg))
g = torch.Generator(device="cuda").manual_seed(3)
data = {"obs": torch.rand((B,) + tuple(cfg["obs_dim"]), device="cuda", generator=g),
        "obs2": torch.rand((B,) + tuple(cfg["obs_dim"]), device="cuda", generator=g),
        "act": (torch.rand(B, cfg["act_dim"], device="cuda", generator=g) * 2 - 1) * cfg["act_lim"],
        "rew": torch.randn(B, device="cuda", generator=g), "done": torch.zeros(B, device="cuda")}


def update(it):
    if a.split:
        eng.compute_grads(data)
        eng.apply(it)
    else:
        eng.step(data, it)


it = 0
for _ in range(a.warmup):
    update(it); it += 1
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
with ClockSampler(0) as clocks:
    e0.record()
    for _ in range(a.steps):
        update(it); it += 1
    e1.record()
    torch.cuda.synchronize()
    time.sleep(max(0.0, 1.2 - e0.elapsed_time(e1) / 1000))
ms = e0.elapsed_time(e1) / a.steps
stats = eng.read_stats()
out = {"metric": "DSAC-T gradient-steps/sec, CNN encoder (carracing type_2, 3x96x96), batch %d" % B, "value": 1000.0 / ms,
       "unit": "steps/s", "ms_per_step": ms, "steps": a.steps, "warmup": a.warmup, "dtype": "f32", "data": "synthetic",
       "call": "compute_grads + apply" if a.split else "step",
       "config": {"workload": "gym_carracing shapes, conv(4,3,3,3,3,3)/(8..256) + mean/log_std heads [256,256,256], fp32 direct convolutions",
                  "batch": B}, "finite": bool(all(v == v for v in stats.values())), "clocks": clocks.summary()}
if a.cpu:   # the CPU arm lives in bench.py (the one place outside tests/ and smoke() that may execute oracle/)
    import bench
    out["cpu_baseline"] = bench.time_cnn_cpu_port(cfg, B, {k: v.cpu().numpy() for k, v in data.items()})
print(json.dumps(out))
