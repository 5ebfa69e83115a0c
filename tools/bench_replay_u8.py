#!/usr/bin/env python
"""fp32 vs 8-bit image replay ring of the CNN configuration (gym_carracing shapes, 3x96x96, reference networks/cnn.py
`type_2`), one B200, both rings in one process:

* device memory that `CnnEngine.bind_replay` allocates for `--capacity` rows of each kind (torch.cuda.memory_allocated);
* ms per `replay_sample` (device-drawn indices) and per `replay_sample` + `step`, at each `--batches` size.

Both rings hold the same transitions (random codes; the fp32 ring holds their decoded pixels) and draw the same indices,
so the two sample the same minibatches; the script checks that before timing.  The dtypes alternate inside every round
(the order flips between rounds); the medians over the rounds are reported.  The rings are far larger than the L2, and
the indices are uniform over all rows, so the gather reads DRAM.

    python tools/bench_replay_u8.py [--capacity 200000] [--batches 256,1024] [--rounds 4]

Prints a table and one JSON line.  Needs ~56 GB of free device memory at the default capacity (44.2 GB fp32 ring +
11.1 GB 8-bit ring + two engines).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "dsac-v2_b200", "dropin")]
import torch  # noqa: E402

from dsac_v2_b200 import synth  # noqa: E402
from dsac_v2_b200.engine_cnn import CnnEngine, make_cnn_config  # noqa: E402
from training.replay_buffer import DECODE_U8  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--capacity", type=int, default=200_000)
ap.add_argument("--batches", default="256,1024")
ap.add_argument("--rounds", type=int, default=4)
ap.add_argument("--sample-reps", type=int, default=200)
ap.add_argument("--step-reps", type=int, default=20)
a = ap.parse_args()
batches = [int(x) for x in a.batches.split(",")]
if not torch.cuda.is_available():
    sys.exit("bench_replay_u8: needs a CUDA device")

cfg = synth.CNN_CONFIGS["carracing"]
t = synth.CONV_TYPES[cfg["conv_type"]]
O, A, cap = 3 * 96 * 96, cfg["act_dim"], a.capacity
dev = torch.device("cuda", 0)
lim = torch.full((A,), cfg["act_lim"])
weights = synth.make_cnn_weights(cfg)


def engine():
    e = CnnEngine(make_cnn_config(cfg["obs_dim"], A, t["kernels"], t["channels"], t["strides"], t["heads"], max_batch=max(batches)),
                  dev, lim, -lim)
    e.load_weights(weights)
    e.seed(17)
    return e


engines = {"float32": engine(), "uint8": engine()}
mem = {}
for name, dtype in (("float32", torch.float32), ("uint8", torch.uint8)):
    torch.cuda.synchronize()
    m0 = torch.cuda.memory_allocated(dev)
    engines[name].bind_replay(cap, obs_dtype=dtype)
    torch.cuda.synchronize()
    mem[name] = torch.cuda.memory_allocated(dev) - m0

# the same transitions in both rings
g = torch.Generator(device=dev).manual_seed(5)
table = torch.from_numpy(DECODE_U8).to(dev)
r8, r32 = engines["uint8"].replay, engines["float32"].replay
for lo in range(0, cap, 4096):
    hi = min(cap, lo + 4096)
    for k in ("obs", "obs2"):
        codes = torch.randint(0, 256, (hi - lo, O), generator=g, device=dev, dtype=torch.uint8)
        r8[k][lo:hi] = codes
        r32[k][lo:hi] = table[codes.long()]
for k in ("act", "rew", "done", "logp"):
    r32[k].copy_(torch.rand(r32[k].shape, generator=g, device=dev) * 2 - 1)
    r8[k].copy_(r32[k])
s32, s8 = engines["float32"].replay_sample(max(batches), cap), engines["uint8"].replay_sample(max(batches), cap)
same = all(torch.equal(s32[k], s8[k]) for k in s32)
assert same, "the two rings sampled different minibatches"

its = {"float32": 0, "uint8": 0}


def timed(name, B, reps, with_step):
    e = engines[name]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def once():
        d = e.replay_sample(B, cap)
        if with_step:
            e.step(d, its[name])
            its[name] += 1
    for _ in range(2):
        once()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        once()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


res = {(n, B, s): [] for n in engines for B in batches for s in (False, True)}
for r in range(a.rounds):
    order = ("float32", "uint8") if r % 2 == 0 else ("uint8", "float32")
    for B in batches:
        for with_step in (False, True):
            for n in order:
                res[(n, B, with_step)].append(timed(n, B, a.step_reps if with_step else a.sample_reps, with_step))

try:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError) as exc:
    q = f"nvidia-smi unavailable: {exc}"
stats = engines["uint8"].read_stats()
out = {"card": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": q, "capacity": cap, "obs_shape": [3, 96, 96],
       "bind_replay_bytes": mem, "same_minibatches": same, "rounds": a.rounds, "sample_reps": a.sample_reps,
       "step_reps": a.step_reps, "finite": bool(all(v == v for v in stats.values())), "ms": {}}
print(f"{out['card']} ({q}); capacity {cap} rows of 3x96x96; {a.rounds} alternating rounds, medians")
print(f"bind_replay: float32 {mem['float32'] / 1e9:.2f} GB, uint8 {mem['uint8'] / 1e9:.2f} GB")
print(f"{'B':>5} {'call':<22} {'float32 ms':>11} {'uint8 ms':>9} {'u8/f32':>7}   per-round float32 | uint8")
for B in batches:
    for with_step in (False, True):
        call = "replay_sample + step" if with_step else "replay_sample"
        m = {n: statistics.median(res[(n, B, with_step)]) for n in engines}
        out["ms"][f"B{B} {call}"] = {n: {"median": m[n], "rounds": res[(n, B, with_step)]} for n in engines}
        rounds = " ".join(f"{x:.4f}" for x in res[("float32", B, with_step)]) + " | " + \
            " ".join(f"{x:.4f}" for x in res[("uint8", B, with_step)])
        print(f"{B:>5} {call:<22} {m['float32']:>11.4f} {m['uint8']:>9.4f} {m['uint8'] / m['float32']:>7.3f}   {rounds}")
print(json.dumps(out))
