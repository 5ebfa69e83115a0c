"""Split form of the head-wise engine (`dsact_cnn_grad_phase1 / _phase2 / _compute_grads / _apply`, CnnEngine's
grad_phase1 / grad_phase2 / compute_grads / apply): the CNN approximators and the policy std types mlp_separated /
parameter.

* the drop-in's gradient-message seam (get_remote_update_info + remote_update) equals local_update;
* sharded phases with the data-parallel exchanges done by hand on one device (2 and 3 handles, ragged shards) equal
  one handle stepping the full minibatch, and the replicas stay bit-identical;
* the call-sequence errors;
* the drop-in under a real process group: world 2 on one device with gloo, and NCCL on 2 / 4 / 8 devices (skipped when
  the machine has fewer)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from dsac_v2_b200 import synth

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-4
TB_KEYS = ("Loss/Critic loss-RL iter", "Loss/Actor loss-RL iter", "DSAC2/critic_avg_min_std1-RL iter", "DSAC2/mean_std1")


# ---- engine-level helpers --------------------------------------------------------------------------------------------
def make_engine(variant, max_batch):
    """(engine, cfg, make_batch) for one head-wise variant on cuda:0, with the synthetic weights."""
    from dsac_v2_b200.engine_cnn import CnnEngine, make_cnn_config, make_heads_config
    h = synth.HYPER
    hyper = dict(gamma=h["gamma"], tau=h["tau"], delay_update=h["delay_update"], auto_alpha=h["auto_alpha"], alpha=h["alpha"],
                 lr_q=h["value_learning_rate"], lr_pi=h["policy_learning_rate"], lr_alpha=h["alpha_learning_rate"],
                 min_log_std=h["policy_min_log_std"], max_log_std=h["policy_max_log_std"])
    if variant == "cnn":
        cfg = synth.CNN_CONFIGS["small_t1"]
        t = synth.CONV_TYPES[cfg["conv_type"]]
        c = make_cnn_config(cfg["obs_dim"], cfg["act_dim"], t["kernels"], t["channels"], t["strides"], t["heads"],
                            max_batch=max_batch, **hyper)
        weights, batch = synth.make_cnn_weights(cfg), synth.make_cnn_batch
    else:
        std_type, dist = {"mlp_separated": ("mlp_separated", "TanhGaussDistribution"), "parameter": ("parameter", "TanhGaussDistribution"),
                          "gauss": ("mlp_separated", "GaussDistribution")}[variant]
        cfg = synth.CONFIGS["ragged"]
        c = make_heads_config(cfg["obs_dim"], cfg["act_dim"], cfg["hidden"], std_type, max_batch=max_batch, act_dist=dist, **hyper)
        weights, batch = synth.make_weights_std(cfg, std_type), synth.make_batch
    lim = torch.full((cfg["act_dim"],), cfg["act_lim"])
    eng = CnnEngine(c, torch.device("cuda", 0), lim, -lim)
    eng.load_weights(weights)
    return eng, cfg, batch


def noise_rows(cfg, B, it, lo, hi):
    n = synth.make_noise(cfg, B, it)
    return tuple(torch.from_numpy(n[i][lo:hi]).cuda() for i in (0, 1, 4, 5))


def batch_rows(make_batch, cfg, B, it, lo, hi):
    return {k: torch.from_numpy(v[lo:hi]).cuda() for k, v in make_batch(cfg, B, it).items()}


# ---- 1. the drop-in's seam equals local_update -----------------------------------------------------------------------
def build_alg(variant, B):
    import dsac_v2
    if variant == "cnn":
        cfg = synth.CNN_CONFIGS["small_t1"]
        kw = synth.cnn_reference_kwargs(cfg, replay_batch_size=B, dsact_noise="reference")
        weights, make_batch = synth.make_cnn_weights(cfg), synth.make_cnn_batch
    else:
        cfg = synth.CONFIGS["ragged"]
        kw = synth.reference_kwargs(cfg, policy_std_type=variant, replay_batch_size=B, dsact_noise="reference")
        weights, make_batch = synth.make_weights_std(cfg, variant), synth.make_batch
    alg = dsac_v2.DSAC_V2(**kw)
    sd = alg.networks.state_dict()
    for k, v in weights.items():
        sd[k] = torch.from_numpy(v)
    alg.networks.load_state_dict(sd)
    alg.networks.cuda()
    return alg, cfg, make_batch


@pytest.mark.parametrize("variant,B", [("cnn", 7), ("mlp_separated", 37), ("parameter", 37)])
def test_remote_update_seam_equals_local_update(variant, B):
    a, cfg, make_batch = build_alg(variant, B)
    b, _, _ = build_alg(variant, B)
    assert a.networks._cnn and b.networks._cnn
    for it in range(4):   # delay_update = 2: two policy / target updates on the way
        batch = batch_rows(make_batch, cfg, B, it, 0, B)
        torch.manual_seed(it)
        tb_a = a.local_update(batch, it)
        torch.manual_seed(it)
        tb_b, info = b.get_remote_update_info(batch, it)
        assert set(info) == {"q1_grad", "q2_grad", "policy_grad", "iteration", "log_alpha_grad"}
        for key, net in (("q1_grad", "q1"), ("q2_grad", "q2"), ("policy_grad", "policy")):
            assert [g.shape for g in info[key]] == [p.shape for p in getattr(b.networks, net).parameters()]
        assert info["log_alpha_grad"].shape == b.networks.log_alpha.shape
        msg = {k: ([g.clone() for g in v] if isinstance(v, list) else (v.clone() if torch.is_tensor(v) else v))
               for k, v in info.items()}
        b.remote_update(msg)
        for k in TB_KEYS:
            assert abs(tb_a[k] - tb_b[k]) <= 1e-5 * max(1.0, abs(tb_a[k])), (k, tb_a[k], tb_b[k])
    for (k, va), vb in zip(a.networks.state_dict().items(), b.networks.state_dict().values()):
        torch.testing.assert_close(va, vb, rtol=1e-5, atol=1e-7, msg=k)


# ---- 2. sharded phases on one device == one handle on the full minibatch ---------------------------------------------
GLOBAL_ROWS = 37   # ragged for 2 and 3 shards


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("variant", ["cnn", "mlp_separated", "parameter", "gauss"])
def test_sharded_phases_equal_full_batch(variant, world):
    from dsac_v2_b200 import _lib, dp
    from dsac_v2_b200.engine import STAT_KEYS
    B = GLOBAL_ROWS
    spans = [dp.shard_rows(B, r, world) for r in range(world)]
    engs = [make_engine(variant, hi - lo)[0] for lo, hi in spans]
    full, cfg, make_batch = make_engine(variant, B)
    S, A = _lib.STATE_STDSUM, _lib.STATE_ACC
    for it in range(5):
        for e, (lo, hi) in zip(engs, spans):
            e.grad_phase1(batch_rows(make_batch, cfg, B, it, lo, hi), noise_rows(cfg, B, it, lo, hi))
        std = torch.stack([e.state[S:S + 2] for e in engs]).sum(0)   # what the all-reduces compute, in rank order
        for e in engs:
            e.state[S:S + 2].copy_(std)
        for e in engs:
            e.grad_phase2(B)
        grads = torch.stack([e.grads for e in engs]).sum(0)
        sums = torch.stack([e.state[A:A + 16] for e in engs]).sum(0)
        mins = torch.stack([e.state[A + 16:A + 18] for e in engs]).min(0).values
        for e in engs:
            e.grads.copy_(grads)
            e.state[A:A + 16].copy_(sums)
            e.state[A + 16:A + 18].copy_(mins)
            e.apply(it)
        full.step(batch_rows(make_batch, cfg, B, it, 0, B), it, noise_rows(cfg, B, it, 0, B))
        ref = full.read_stats()
        for r, e in enumerate(engs):
            s = e.read_stats(B)
            np.testing.assert_allclose([s[k] for k in STAT_KEYS], [ref[k] for k in STAT_KEYS], rtol=RTOL, atol=1e-6,
                                       err_msg=f"{variant} world {world} rank {r} step {it}")
    for e in engs[1:]:   # replicas stay bit-identical
        assert torch.equal(e.params, engs[0].params) and torch.equal(e.targets, engs[0].targets)
        assert torch.equal(e.adam_m, engs[0].adam_m) and torch.equal(e.adam_v, engs[0].adam_v)
        assert torch.equal(e.state[:4], engs[0].state[:4])
    diff = (engs[0].params - full.params).abs().max().item()
    print(f"{variant} world {world}: max |param diff| vs the full batch = {diff:.2e}")
    torch.testing.assert_close(engs[0].params, full.params, rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(engs[0].targets, full.targets, rtol=2e-5, atol=2e-6)


def test_compute_grads_then_apply_equals_step():
    """compute_grads + apply runs the kernels of step; with the same inputs the results agree to the summation order of
    the gradient atomics."""
    from dsac_v2_b200.engine import STAT_KEYS
    a, cfg, make_batch = make_engine("cnn", 9)
    b, _, _ = make_engine("cnn", 9)
    for it in range(3):
        data, nz = batch_rows(make_batch, cfg, 9, it, 0, 9), noise_rows(cfg, 9, it, 0, 9)
        a.step(data, it, nz)
        b.compute_grads(data, nz)
        b.apply(it)
        sa, sb = a.read_stats(), b.read_stats()
        np.testing.assert_allclose([sb[k] for k in STAT_KEYS], [sa[k] for k in STAT_KEYS], rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(b.params, a.params, rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(b.targets, a.targets, rtol=1e-5, atol=1e-7)


# ---- 3. call-sequence errors -----------------------------------------------------------------------------------------
def test_split_entry_points_reject_bad_sequences():
    import ctypes as C
    from dsac_v2_b200 import _lib
    from dsac_v2_b200.engine_cnn import CnnEngine, make_heads_config
    eng, cfg, make_batch = make_engine("mlp_separated", 8)
    lib, s = eng.lib, eng._stream()

    def last_error():
        return lib.dsact_last_error().decode()
    assert lib.dsact_cnn_grad_phase2(eng.h, 8, s) == -3 and last_error()           # DSACT_ESTATE: no phase 1 yet
    b = eng._batch(batch_rows(make_batch, cfg, 8, 0, 0, 8))
    assert lib.dsact_cnn_grad_phase1(eng.h, C.byref(b), None, s) == 0
    assert lib.dsact_cnn_grad_phase2(eng.h, 7, s) == -1 and "global_batch" in last_error()   # DSACT_EINVAL: < local rows
    assert lib.dsact_cnn_grad_phase2(eng.h, 8, s) == 0                               # the pending phase 1 survived the refusal
    assert lib.dsact_cnn_grad_phase2(eng.h, 8, s) == -3 and last_error()            # phase 2 consumed it
    assert lib.dsact_cnn_apply(eng.h, 0, s) == 0
    torch.cuda.synchronize()
    assert torch.isfinite(eng.params).all()
    # DSAC_V1 handles have dsact_cnn_step only
    h = synth.HYPER
    v1 = make_heads_config(cfg["obs_dim"], cfg["act_dim"], cfg["hidden"], "mlp_separated", max_batch=8, algo="DSAC_V1",
                           lr_q=h["value_learning_rate"], lr_pi=h["policy_learning_rate"], lr_alpha=h["alpha_learning_rate"])
    lim = torch.full((cfg["act_dim"],), cfg["act_lim"])
    e1 = CnnEngine(v1, torch.device("cuda", 0), lim, -lim)
    b1 = e1._batch(batch_rows(make_batch, cfg, 8, 0, 0, 8))
    for rc in (lib.dsact_cnn_grad_phase1(e1.h, C.byref(b1), None, s), lib.dsact_cnn_grad_phase2(e1.h, 8, s),
               lib.dsact_cnn_compute_grads(e1.h, C.byref(b1), None, s), lib.dsact_cnn_apply(e1.h, 0, s)):
        assert rc == -1 and "DSAC_V1" in last_error()
    with pytest.raises(_lib.DsactError):
        e1.compute_grads(batch_rows(make_batch, cfg, 8, 0, 0, 8))
    eng.close(); e1.close()


# ---- 4. the drop-in under a real process group -----------------------------------------------------------------------
DP_ROWS = 10   # global minibatch of the engine-level leg: ragged for 4 and 8 ranks, 5 rows each at world 2


def _worker(rank, world, port, out_dir, backend):
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, "dsac-v2_b200", "dropin"))
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    import datetime
    import torch.distributed as dist
    dev = 0 if backend == "gloo" else rank   # gloo: every rank on cuda:0
    torch.cuda.set_device(dev)
    kw = dict(device_id=torch.device("cuda", dev)) if backend == "nccl" else {}
    dist.init_process_group(backend, rank=rank, world_size=world, timeout=datetime.timedelta(seconds=120), **kw)
    from dsac_v2_b200 import dp
    out = {}
    # (i) engine level: dp.data_parallel_gradients + apply with explicit shard noise
    eng, cfg, make_batch = make_engine("cnn", DP_ROWS)
    lo, hi = dp.shard_rows(DP_ROWS, rank, world)
    tbs = []
    for it in range(3):
        gb = dp.data_parallel_gradients(eng, batch_rows(make_batch, cfg, DP_ROWS, it, lo, hi), noise_rows(cfg, DP_ROWS, it, lo, hi),
                                        dist, hi - lo, DP_ROWS)
        eng.apply(it)
        tbs.append([eng.read_stats(gb)[k] for k in TB_KEYS])
    out["eng_params"], out["eng_targets"], out["eng_tb"] = eng.params.cpu().numpy(), eng.targets.cpu().numpy(), np.array(tbs)
    eng.close()
    # (ii) DSAC_V2.local_update on a CNN configuration, every rank with its own rows and its own noise
    B = 4
    alg, cfg, make_batch = build_alg("cnn", B)
    tbs = []
    for it in range(3):
        tb = alg.local_update(batch_rows(make_batch, cfg, B * world, it, rank * B, (rank + 1) * B), it)
        tbs.append([tb[k] for k in TB_KEYS])
    out["alg_tb"] = np.array(tbs)
    eng = alg.networks.engine()
    out["alg_params"], out["alg_targets"] = eng.params.cpu().numpy(), eng.targets.cpu().numpy()
    # (iii) get_remote_update_info: the global gradient on every rank
    torch.manual_seed(100 + rank)   # the reference noise differs between ranks; the all-reduce makes the gradient global
    _, info = alg.get_remote_update_info(batch_rows(make_batch, cfg, B * world, 3, rank * B, (rank + 1) * B), 3)
    out["msg"] = torch.cat([g.reshape(-1) for k in ("q1_grad", "q2_grad", "policy_grad") for g in info[k]]
                           + [info["log_alpha_grad"].reshape(-1)]).cpu().numpy()
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **out)
    dist.destroy_process_group()


def _run_world(tmp_path, world, backend):
    port = 29100 + (os.getpid() + 17 * world + (5 if backend == "nccl" else 0)) % 1000
    mp.spawn(_worker, args=(world, port, str(tmp_path), backend), nprocs=world, join=True)
    ranks = [np.load(tmp_path / f"rank{r}.npz") for r in range(world)]
    r0 = ranks[0]
    for r in ranks[1:]:
        for k in ("eng_params", "eng_targets", "eng_tb", "alg_params", "alg_targets", "alg_tb", "msg"):
            np.testing.assert_array_equal(r0[k], r[k], err_msg=f"ranks differ: {k}")
    assert np.isfinite(r0["alg_tb"]).all() and np.isfinite(r0["msg"]).all()
    assert not np.array_equal(r0["msg"], np.zeros_like(r0["msg"]))
    # the engine-level leg against one handle on the full minibatch
    full, cfg, make_batch = make_engine("cnn", DP_ROWS)
    tbs = []
    for it in range(3):
        full.step(batch_rows(make_batch, cfg, DP_ROWS, it, 0, DP_ROWS), it, noise_rows(cfg, DP_ROWS, it, 0, DP_ROWS))
        s = full.read_stats()
        tbs.append([s[k] for k in TB_KEYS])
    np.testing.assert_allclose(r0["eng_tb"], np.array(tbs), rtol=RTOL, atol=1e-6)
    np.testing.assert_allclose(r0["eng_params"], full.params.cpu().numpy(), rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(r0["eng_targets"], full.targets.cpu().numpy(), rtol=2e-5, atol=2e-6)


def test_dropin_data_parallel_gloo_two_ranks_one_device(tmp_path):
    _run_world(tmp_path, 2, "gloo")


@pytest.mark.parametrize("world", [2, 4, 8])
def test_dropin_data_parallel_nccl(tmp_path, world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    _run_world(tmp_path, world, "nccl")
