#!/usr/bin/env python
"""bench.py — DSAC-T gradient-steps/sec on synthetic Humanoid-shaped minibatches.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 4096] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): obs=376, act=17, MLP [256,256,256] for the policy and both
critics, batch 4096 per GPU, device replay ring of 1e6 synthetic transitions (3.09 GB, far larger
than the 126 MB L2: every step gathers fresh random rows from HBM).  One "step" = one
`DSAC_V2.local_update`-equivalent: replay gather + 8 MLP forwards + losses + 3 backward passes +
Adam + delayed Polyak.  Nothing is skipped on any iteration.

`value`   : steps/s with inputs resident in HBM (`dsact_replay_step`: index draw, gather, update
            in one CUDA-graph submission), device-timed with CUDA events, max over ranks.
`e2e`     : the same step through the reference-facing API `DSAC_V2.local_update(data, it)` with
            HOST (pinned) minibatches: H2D copies inside the timed region and the critic loss
            read back to the host every step.
`roofline`: the grouped GEMM kernel (all dense layers; tcgen05 in the default bf16x3 mode), algorithmic FLOPs / event-timed
            duration from `dsact_profile_step`, against MEASURED_PEAKS.json.
`cpu_baseline` / `--impl reference`: the torch-CPU oracle port of the reference path (the
            reference is pure PyTorch, so the port issues the same ATen ops) on the host cores.
N > 1 (torchrun): data parallel, one process per GPU, batch 4096 per GPU (weak scaling),
NCCL all-reduce of the critic-std sums and of the flat gradients; `value` counts one
4096-row minibatch update per rank per step.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "dsac-v2_b200", "dropin"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from dsac_v2_b200 import synth  # noqa: E402

FLOP_PER_SAMPLE = 2 * 3_240_448  # SURVEY.md §8(d): 6.481 MFLOP per sample per step (H dims)
METRIC = "DSAC-T gradient-steps/sec @ batch 4096 (Humanoid-dim)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--config", default="humanoid", choices=list(synth.CONFIGS))
    ap.add_argument("--replay-size", type=int, default=1_000_000)
    ap.add_argument("--gemm", default="bf16x3", choices=["fp32", "bf16x3", "bf16"],
                    help="dense-layer arithmetic; bf16x3 (default) and fp32 pass the 1e-4 parity gate, bf16 does not")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dp", default="peer", choices=["peer", "nccl"],
                    help="N > 1: exchanges inside the step's kernels over NVLink peer memory, or torch.distributed/NCCL")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them computed (the networks' weights under their "
                         "state_dict names, and tb_info.npy) to DIR/<name>.npy, so that two builds run with the same "
                         "arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def peaks():
    try:
        p = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        return p["bf16_tflops_sustained"], p["hbm_gbs"], "measured"
    except Exception:
        return 1400.0, 6650.0, "fallback"  # B200_PROFILING.md fallback (sustained)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic(mode):
    """Average dram bytes (read + write) per GEMM-class launch from the committed `ncu --set full` summary of this
    mode (profiles/), or None if no capture is committed for it."""
    path = os.path.join(REPO, "profiles", f"r2_{mode}_tc_full.txt")
    if not os.path.exists(path):
        path = os.path.join(REPO, "profiles", f"r1_{mode}_tc_full.txt")
    try:
        rows = [l.split(" | ") for l in open(path) if l.startswith("void ")]
        mb = [float(r[3]) + float(r[4]) for r in rows]
        return {"bytes_per_launch": round(1e6 * sum(mb) / len(mb)), "launches": len(mb), "source": os.path.relpath(path, REPO)}
    except Exception:
        return None


def cpu_ring_rows(cfg, want=1_000_000):
    """Replay rows of the CPU arms: the benchmarked 1e6 when the host has the memory for it (3.1 GB for Humanoid)."""
    try:
        avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    except (ValueError, OSError):
        avail = 0
    need = want * 4 * (2 * cfg["obs_dim"] + cfg["act_dim"] + 2)
    return want if avail > 4 * need else 100_000


def oracle_setup(cfg, batch, ring_rows=100_000):
    from oracle.dsact_oracle import from_config
    torch.manual_seed(0)
    orc = from_config(cfg, synth.make_weights(cfg), **synth.HYPER)
    g = np.random.default_rng(123)
    O, A, lim = cfg["obs_dim"], cfg["act_dim"], cfg["act_lim"]
    ring = {"obs": g.standard_normal((ring_rows, O), dtype=np.float32),
            "obs2": g.standard_normal((ring_rows, O), dtype=np.float32),
            "act": g.uniform(-lim, lim, (ring_rows, A)).astype(np.float32),
            "rew": g.standard_normal(ring_rows, dtype=np.float32),
            "done": (g.random(ring_rows) < 0.01).astype(np.float32)}

    def step(it):
        idx = np.random.randint(0, ring_rows, size=batch)  # training/replay_buffer.py:85-90
        data = {k: torch.as_tensor(v[idx]) for k, v in ring.items()}
        noise = [torch.randn(batch, A), torch.randn(batch, A)] + [torch.randn(batch) for _ in range(6)]
        return orc.update(data, noise, it)

    return step


def pick_threads(cfg, batch):
    """torch intra-op threads for the CPU arm: the reference pins 4 (utils/init_args.py:14); more helps up to
    a point, and a container may see far more cores than it may use.  Try a few, keep the fastest."""
    step = oracle_setup(cfg, batch)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    best, best_t = 4, None
    for n in sorted({4, 8, 16, 32, min(64, cores)}):
        if n > cores:
            continue
        torch.set_num_threads(n)
        step(0)
        t0 = time.perf_counter()
        step(1)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def time_oracle(cfg, batch, warm, max_steps, budget_s, ring_rows=100_000):
    step = oracle_setup(cfg, batch, ring_rows)
    for it in range(warm):
        step(it)
    t0, n = time.perf_counter(), 0
    while n < max_steps and (time.perf_counter() - t0 < budget_s or n < 2):
        step(warm + n)
        n += 1
    dt = time.perf_counter() - t0
    return n / dt, n, dt


def time_cnn_cpu_port(cfg, batch, host_batch, updates=3):
    """CPU arm of tools/bench_cnn.py (BASELINE config 5): the oracle port of the CNN update on the host cores."""
    import torch
    from dsac_v2_b200 import synth
    from oracle.dsact_oracle import cnn_from_config
    torch.set_num_threads(min(32, os.cpu_count() or 4))
    orc = cnn_from_config(cfg, synth.make_cnn_weights(cfg), **synth.HYPER)
    nz = synth.make_noise(cfg, batch, 0)
    orc.update(host_batch, nz, 0)
    t0 = time.perf_counter()
    for n in range(updates):
        orc.update(host_batch, nz, n + 1)
    dt = (time.perf_counter() - t0) / updates
    return {"value": 1.0 / dt, "unit": "steps/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{updates} updates of batch {batch}, {cpu_model()}"}


def time_cuda_eager(cfg, batch, dev, steps=60, warm=5, ring_rows=200_000):
    """The reference's arithmetic as eager PyTorch on THIS GPU: the oracle port with CUDA tensors issues the ATen ops the
    reference's dsac_v2.py issues (torch.distributions object churn aside); replay ring, index draw and noise on the device.
    Separates "what a B200 gives stock PyTorch" from what the hand-written kernels add."""
    from oracle.dsact_oracle import from_config
    orc = from_config(cfg, synth.make_weights(cfg), **synth.HYPER).to(dev)
    O, A, lim = cfg["obs_dim"], cfg["act_dim"], cfg["act_lim"]
    g = torch.Generator(device=dev).manual_seed(5)
    ring = {"obs": torch.randn(ring_rows, O, device=dev, generator=g), "obs2": torch.randn(ring_rows, O, device=dev, generator=g),
            "act": (torch.rand(ring_rows, A, device=dev, generator=g) * 2 - 1) * lim, "rew": torch.randn(ring_rows, device=dev, generator=g),
            "done": (torch.rand(ring_rows, device=dev, generator=g) < 0.01).float()}

    def step(it):
        idx = torch.randint(0, ring_rows, (batch,), device=dev)
        data = {k: v[idx] for k, v in ring.items()}
        noise = [torch.randn(batch, A, device=dev), torch.randn(batch, A, device=dev)] + [torch.randn(batch, device=dev) for _ in range(6)]
        return orc.update(data, noise, it)

    for it in range(warm):
        step(it)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for it in range(steps):
        step(warm + it)
    e1.record()
    torch.cuda.synchronize(dev)
    return 1000.0 * steps / e0.elapsed_time(e1)


def h2d_gbs(eng, host_batch, nbytes, busy, reps=40):
    """Host -> device bandwidth of the staging path itself (`dsact_stage_host`: five cudaMemcpyAsync calls of one pinned
    minibatch on the library's copy stream), with no update behind the copies but WHILE the GPU runs device-resident
    steps (`busy`): the ceiling of the end-to-end rate.  (An idle GPU drops its PCIe link speed and shows half of it.)"""
    dev = eng.device
    for _ in range(5):
        busy()
        eng._stage_in(host_batch); eng._mark_staged_done()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(reps):
        busy()
        eng._stage_in(host_batch); eng._mark_staged_done()
    torch.cuda.synchronize(dev)
    return nbytes * reps / (time.perf_counter() - t0) / 1e9


def check_replicas(alg, eng, cfg, B, rank, world, dev, dist, it0):
    """N > 1 only.  (1) After the timed loops every rank's params / targets / Adam moments must be bit-identical (checksums
    all-gathered).  (2) Three more data-parallel updates on host-generated shards with explicit noise; rank 0 then replays
    the same three updates on ONE GPU over the concatenated minibatch, starting from a snapshot of the same state, and the
    results must agree within the parity tolerance (the reduction order differs)."""
    def checksum():
        parts = [eng.params, eng.targets, eng.adam_m, eng.adam_v]
        return torch.stack([p.double().sum() for p in parts] + [p.double().abs().sum() for p in parts])

    cs = checksum()
    gathered = [torch.zeros_like(cs) for _ in range(world)]
    dist.all_gather(gathered, cs)
    identical = all(bool(torch.equal(g, gathered[0])) for g in gathered)
    snap = {k: getattr(eng, k).clone() for k in ("params", "targets", "adam_m", "adam_v", "state")}
    GB = B * world
    tbs = []
    for s in range(3):
        full, noise = synth.make_batch(cfg, GB, 900 + s), synth.make_noise(cfg, GB, 900 + s)
        lo, hi = rank * B, (rank + 1) * B
        shard = {k: torch.from_numpy(v[lo:hi]).to(dev) for k, v in full.items()}
        nz = tuple(torch.from_numpy(noise[i][lo:hi]).to(dev) for i in (0, 1, 4, 5))
        if getattr(alg, "_peer_dp", False):
            eng.dp_step(shard, it0 + s, GB, nz)
        else:
            from dsac_v2_b200 import dp as dpmod
            dpmod.data_parallel_gradients(eng, shard, nz, dist, B, GB)
            eng.apply(it0 + s)
        tbs.append(eng.read_stats(GB)["Loss/Critic loss-RL iter"])
    cs2 = checksum()
    dist.all_gather(gathered, cs2)
    identical = identical and all(bool(torch.equal(g, gathered[0])) for g in gathered)
    out = {"replicas_bit_identical": identical, "ranks": world}
    if rank == 0:   # single-GPU replay of the same three updates on the concatenated minibatch
        from dsac_v2_b200.engine import Engine
        from dsac_v2_b200.engine import make_config
        c = make_config(cfg["obs_dim"], cfg["act_dim"], cfg["hidden"], cfg["hidden"], max_batch=GB, gemm_mode=_lib_mode(eng))
        one = Engine(c, dev, eng.act_high, eng.act_low)
        for k, v in snap.items():
            getattr(one, k).copy_(v)
        ref = []
        for s in range(3):
            full, noise = synth.make_batch(cfg, GB, 900 + s), synth.make_noise(cfg, GB, 900 + s)
            one.step({k: torch.from_numpy(v).to(dev) for k, v in full.items()}, it0 + s,
                     tuple(torch.from_numpy(noise[i]).to(dev) for i in (0, 1, 4, 5)))
            ref.append(one.read_stats()["Loss/Critic loss-RL iter"])
        rel = max(abs(a - b) / max(abs(b), 1e-6) for a, b in zip(tbs, ref))
        dw = float((one.params - eng.params).abs().max() / one.params.abs().max())
        out.update({"critic_loss_dp": tbs, "critic_loss_one_gpu": ref, "max_rel_loss_diff": rel, "max_param_diff_rel": dw,
                    "status": "ok" if identical and rel < 1e-4 and dw < 1e-4 else "MISMATCH"})
        one.close()
    return out


def dump_outputs(eng, out_dir, global_batch):
    """What a caller of the timed update holds after its last step: every network's parameters and target parameters
    under their state_dict names (float32), and `tb_info.npy`, the 14 tb_info values in engine.STAT_KEYS order (float64).
    About 5.6 MB for the Humanoid networks."""
    from dsac_v2_b200.engine import STAT_KEYS
    os.makedirs(out_dir, exist_ok=True)
    stats = eng.read_stats(global_batch)
    np.save(os.path.join(out_dir, "tb_info.npy"), np.array([stats[k] for k in STAT_KEYS], dtype=np.float64))
    for name, t in eng.export_weights().items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.numpy().astype(np.float32))


def _lib_mode(eng):
    from dsac_v2_b200 import _lib
    return {v: k for k, v in _lib.GEMM_MODES.items()}[eng.cfg.gemm_mode]


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path (torch-CPU port, all host threads)."""
    if rank != 0:
        return
    cfg = synth.CONFIGS[args.config]
    threads = pick_threads(cfg, args.batch)
    rows = cpu_ring_rows(cfg, args.replay_size)
    step = oracle_setup(cfg, args.batch, rows)
    t0 = time.perf_counter()
    step(0)
    est = time.perf_counter() - t0
    warm = min(args.warmup, max(1, int(20.0 / max(est, 1e-3))))
    for it in range(1, warm):
        step(it)
    k = args.steps if est * args.steps <= 200.0 else max(3, int(200.0 / est))
    t0 = time.perf_counter()
    for it in range(k):
        step(warm + it)
    dt = time.perf_counter() - t0
    value = k / dt
    sample = f"{k} full updates of batch {args.batch} (+ numpy replay gather from a {rows}-row ring), {warm} warm-up"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": args.gpus,
        "steps": k, "warmup": warm, "ms_per_step": 1000 * dt / k, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"gym_humanoid-shaped synthetic, obs=376 act=17 MLP[256,256,256] batch={args.batch}, CPU torch",
                   "global_batch": args.batch, "host": cpu_model(), "replay_rows": rows},
        "cpu_baseline": {"value": value, "unit": "steps/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        # NCCL prints its version banner on stdout when the communicator is created: keep stdout for the ONE JSON line
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.all_reduce(torch.zeros(1, device=torch.device("cuda", local)))
            torch.cuda.synchronize()
        finally:
            os.dup2(saved, 1)
            os.close(saved)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    # host side of the end-to-end leg: sit on the GPU's NUMA node before any pinned allocation (hostnuma.py), and run
    # torch's CPU ops with the reference's own thread count (utils/init_args.py:14 pins 4)
    from dsac_v2_b200 import hostnuma
    numa = hostnuma.bind_to_gpu_node(local)
    torch.set_num_threads(4)

    import dsac_v2
    from training.replay_buffer import ReplayBuffer

    cfg = synth.CONFIGS[args.config]
    B, O, A = args.batch, cfg["obs_dim"], cfg["act_dim"]
    kw = synth.reference_kwargs(cfg, replay_batch_size=B, dsact_gemm=args.gemm, buffer_max_size=args.replay_size,
                                additional_info={})
    alg = dsac_v2.DSAC_V2(**kw)
    sd = alg.networks.state_dict()
    for k, v in synth.make_weights(cfg).items():
        sd[k] = torch.from_numpy(v)
    alg.networks.load_state_dict(sd)
    alg.networks.cuda()
    eng = alg.networks.engine(B)
    eng.seed(1000 + rank)
    buf = ReplayBuffer(**kw)
    buf.attach(eng)
    g = torch.Generator(device=dev).manual_seed(123 + rank)  # synthetic transitions, SURVEY §8(d)
    r = eng.replay
    r["obs"].normal_(generator=g); r["obs2"].normal_(generator=g); r["rew"].normal_(generator=g)
    r["act"].uniform_(-cfg["act_lim"], cfg["act_lim"], generator=g)
    r["done"].copy_((torch.rand(args.replay_size, device=dev, generator=g) < 0.01).float())
    buf.size, buf.ptr = args.replay_size, 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peer_dp = False
    if world > 1 and args.dp != "nccl":   # exchange buffers mapped over NVLink (CUDA IPC); NCCL path if that fails
        from dsac_v2_b200 import dp as dpmod
        peer_dp = dpmod.connect_peers(eng, dist)
        alg._peer_dp = peer_dp

    def dev_step(it):
        if world == 1:
            eng.replay_step(B, buf.size, it)
        elif peer_dp:
            eng.dp_replay_step(B, buf.size, it, B * world)   # one graph per rank, exchanges inside its kernels
        else:
            alg.local_update(buf.sample_batch(B), it)

    # ---- device-resident throughput ------------------------------------------------
    it = 0
    for _ in range(args.warmup):
        dev_step(it); it += 1
    launches_per_step = eng.last_call_launches() if world == 1 else None   # (N > 1: three phase launches + collectives)
    barrier()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        e0.record()
        for _ in range(args.steps):
            dev_step(it); it += 1
        e1.record()
        barrier()
        if args.dump_outputs and rank == 0:   # before the sampler's extra steps below, whose count depends on timing
            dump_outputs(eng, args.dump_outputs, B * world)
        extra = max(0.0, 1.2 - e0.elapsed_time(e1) / 1000)  # keep the sampler alive for a few readings
        n_extra = torch.tensor([int(extra * 1000 / max(e0.elapsed_time(e1) / args.steps, 1e-3))], device=dev)
        if world > 1:   # data-parallel steps are collective: every rank must run the same number of them
            dist.all_reduce(n_extra, op=dist.ReduceOp.MAX)
        for _ in range(int(n_extra.item())):
            dev_step(it); it += 1
        torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step = ms.item() / args.steps
    launches = eng.launch_count() - l0
    value = world * 1000.0 / ms_per_step

    # ---- end to end through DSAC_V2.local_update with host minibatches ------------------
    ring = []
    hg = torch.Generator().manual_seed(7 + rank)
    for _ in range(4):
        ring.append({"obs": torch.randn(B, O, generator=hg).pin_memory(), "obs2": torch.randn(B, O, generator=hg).pin_memory(),
                     "act": ((torch.rand(B, A, generator=hg) * 2 - 1) * cfg["act_lim"]).pin_memory(),
                     "rew": torch.randn(B, generator=hg).pin_memory(),
                     "done": (torch.rand(B, generator=hg) < 0.01).float().pin_memory()})
    sink = 0.0
    for i in range(max(3, args.warmup // 2)):
        sink += alg.local_update(ring[i % 4], it)["Loss/Critic loss-RL iter"]; it += 1
    barrier()
    e0.record()
    prev = None
    for i in range(args.steps):
        tb = alg.local_update(ring[i % 4], it); it += 1   # H2D of this step's inputs (side stream) + update
        if prev is not None:
            sink += prev["Loss/Critic loss-RL iter"]      # device -> host read of EVERY step's result, one call late so
        prev = tb                                         # that the next step's copy overlaps this step's kernels
    sink += prev["Loss/Critic loss-RL iter"]
    e1.record()
    barrier()
    ms2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = world * 1000.0 * args.steps / ms2.item()
    assert np.isfinite(sink)
    h2d_bytes = 4 * B * (2 * O + A + 2)
    h2d_rate = None
    if world == 1:
        def busy():
            nonlocal it
            dev_step(it); it += 1
        h2d_rate = h2d_gbs(eng, ring[0], h2d_bytes, busy)

    # ---- data-parallel replicas: bit-identical after the timed loops, and equal to one GPU on the concatenated batch ----
    dp_check = None
    if world > 1:
        dp_check = check_replicas(alg, eng, cfg, B, rank, world, dev, dist, it)
        it += 3

    # ---- roofline of the dominant kernel (grouped GEMM), per-launch events, eager -------------------
    peak_tf, peak_hbm, peak_src = peaks()
    roof = None
    if rank == 0:
        data = buf.sample_batch(B)
        acc = None
        for _ in range(5):
            p = eng.profile_step(data, it); it += 1
            if acc is None:
                acc = p
            else:
                acc["total_ms"] += p["total_ms"]
                for k in ("other", "gemm_fwd", "gemm_dgrad", "gemm_wgrad"):
                    for f in ("ms", "flops", "launches"):
                        acc[k][f] += p[k][f]
        gem = [acc[k] for k in ("gemm_fwd", "gemm_dgrad", "gemm_wgrad")]
        g_ms, g_fl, g_n = sum(x["ms"] for x in gem), sum(x["flops"] for x in gem), sum(x["launches"] for x in gem)
        achieved = g_fl / (g_ms * 1e-3) / 1e12
        kname = "dsact::gemm_kernel (fp32 FFMA)" if args.gemm == "fp32" else \
            "dsact::tc_chain_kernel (fused layer chains: forward, dgrad) + dsact::tc_gemm_kernel (wgrad) — tcgen05, TMA, TMEM"
        roof = {"bound": "tensor", "kernel": kname + "; all dense layers of the step",
                "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                "traffic": ncu_traffic(args.gemm),
                "peak_source": f"bf16_tflops_sustained of {peak_src}; arithmetic here is {args.gemm}"
                               + (" = 3 bf16 MMA passes per algorithmic FLOP, i.e. effective peak = peak/3" if args.gemm == "bf16x3" else ""),
                "flop_per_sample_measured": g_fl / 5 / B, "flop_per_sample_survey": FLOP_PER_SAMPLE,
                "avg_launch_us": 1000 * g_ms / g_n, "launches_per_step": g_n // 5,
                "share_of_step": g_ms / acc["total_ms"],
                "by_kind": {k: {"tflops": acc[k]["flops"] / (acc[k]["ms"] * 1e-3) / 1e12, "ms_per_step": acc[k]["ms"] / 5}
                            for k in ("gemm_fwd", "gemm_dgrad", "gemm_wgrad")},
                "other_ms_per_step": acc["other"]["ms"] / 5, "eager_step_ms": acc["total_ms"] / 5}

    # ---- CPU baseline (oracle port) on the host cores ----------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = pick_threads(cfg, B)
        rows = cpu_ring_rows(cfg, args.replay_size)
        v, n, dt = time_oracle(cfg, B, warm=3, max_steps=2000, budget_s=12.0, ring_rows=rows)
        cpu = {"value": v, "unit": "steps/s", "cores": threads, "kind": "port",
               "sample": f"{n} full updates of batch {B} incl. numpy replay gather from a {rows}-row ring ({dt:.1f} s), {cpu_model()}"}
        torch.set_num_threads(4)

    eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v = time_cuda_eager(cfg, B, dev)
        eager = {"value": v, "unit": "steps/s", "kind": "oracle port on CUDA tensors (stock eager PyTorch ops, same GPU)",
                 "sample": f"60 updates of batch {B}, device ring 200000 rows, device randint/randn"}

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if args.gemm == "fp32" else args.gemm, "data": "synthetic",
            "config": {"workload": f"gym_{args.config} shapes (obs={O} act={A}) MLP{list(cfg['hidden'])} batch_size={B} per GPU, "
                                   f"device replay ring {args.replay_size} rows, device index+noise generation",
                       "global_batch": B * world, "parallelism": (f"dp{world}" + ("-peer" if peer_dp else "-nccl")) if world > 1 else "single",
                       "l2": f"inputs exceed L2: each step gathers {B} random rows from a {4 * args.replay_size * (2 * O + A + 3) / 1e9:.2f} GB ring",
                       "gemm_mode": args.gemm, "cuda_graph": True},
            "clocks": clocks.summary(),
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 64, "api": "DSAC_V2.local_update(host pinned dict, iteration) + tb_info read "
                                                     "(dsact_step_host: staging copies on the library's copy stream)",
                    "h2d_gbs": h2d_rate, "h2d_gbs_used": e2e_value / world * h2d_bytes / 1e9,
                    "host": {"numa": numa, "torch_threads": torch.get_num_threads()}},
            "dp_check": dp_check,
            "gpu_launches": launches,
            "launches_per_step": launches_per_step,
            "tflops_algorithmic": FLOP_PER_SAMPLE * B * value / world / 1e12 if args.config == "humanoid" else None,
            "roofline": roof,
            "cpu_baseline": cpu,
            "cuda_eager_baseline": eager,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
