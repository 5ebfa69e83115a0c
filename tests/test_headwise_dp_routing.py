"""Routing of `DSAC_V2.local_update` under a multi-rank process group, without a GPU: the head-wise engine (CNN
approximators, policy std types mlp_separated / parameter) runs the torch.distributed seam (grad_phase1 -> all-reduce ->
grad_phase2 over the global batch -> all-reduce -> apply) and never the peer-memory set-up; the tcgen05 engine still
tries the peer-memory exchange first."""
import pytest
import torch

from dsac_v2_b200 import _lib, dp, synth


class _StubEngine:
    """The split API of engine.Engine / engine_cnn.CnnEngine, recording the calls."""

    def __init__(self, n_grads=10):
        self.calls = []
        self.state = torch.zeros(64)
        self.grads = torch.zeros(n_grads)

    def grad_phase1(self, data, noise=None):
        self.calls.append(("grad_phase1", int(data["obs"].shape[0])))

    def grad_phase2(self, global_batch):
        self.calls.append(("grad_phase2", int(global_batch)))

    def apply(self, iteration):
        self.calls.append(("apply", int(iteration)))

    def step(self, data, iteration, noise=None):
        self.calls.append(("step", int(iteration)))

    def dp_step(self, data, iteration, global_batch, noise=None):
        self.calls.append(("dp_step", int(iteration)))


class _FakeDist:
    """Two ranks; this one's all-reduces see an identical peer (SUM doubles, MIN keeps)."""

    class ReduceOp:
        SUM, MIN = "sum", "min"

    def __init__(self):
        self.reduced = []

    def all_reduce(self, t, op="sum"):
        self.reduced.append((t.numel(), op))
        if op == "sum":
            t.mul_(2)


def _alg(monkeypatch, kw):
    import dsac_v2
    alg = dsac_v2.DSAC_V2(**kw)
    eng = _StubEngine()
    dist = _FakeDist()
    monkeypatch.setattr(alg.networks, "engine", lambda batch=0: eng)
    monkeypatch.setattr(alg, "_world", lambda: (dist, 2))
    seen = {}

    def stats(e, global_batch, t0):
        seen["global_batch"] = global_batch
        return {}
    monkeypatch.setattr(alg, "_stats", stats)
    return alg, eng, dist, seen


def _batch(B, obs_shape):
    return {"obs": torch.zeros((B,) + tuple(obs_shape)), "obs2": torch.zeros((B,) + tuple(obs_shape)), "act": torch.zeros(B, 2),
            "rew": torch.zeros(B), "done": torch.zeros(B)}


@pytest.mark.parametrize("variant", ["cnn", "mlp_separated", "parameter"])
def test_headwise_local_update_runs_the_nccl_seam(monkeypatch, variant):
    B = 6
    if variant == "cnn":
        cfg = synth.CNN_CONFIGS["small_t1"]
        kw, obs_shape = synth.cnn_reference_kwargs(cfg, replay_batch_size=B), cfg["obs_dim"]
    else:
        cfg = synth.CONFIGS["ragged"]
        kw, obs_shape = synth.reference_kwargs(cfg, policy_std_type=variant, replay_batch_size=B), (cfg["obs_dim"],)
    alg, eng, dist, seen = _alg(monkeypatch, kw)
    assert alg.networks._cnn

    def refuse(*a, **k):
        raise AssertionError("the head-wise engine has no peer-memory exchange")
    monkeypatch.setattr(dp, "connect_peers", refuse)
    alg.local_update(_batch(B, obs_shape), 5)
    assert eng.calls == [("grad_phase1", B), ("grad_phase2", 2 * B), ("apply", 5)]
    assert seen["global_batch"] == 2 * B
    # std sums, gradients, the 16 logged sums, the 2 minima
    assert dist.reduced == [(2, "sum"), (eng.grads.numel(), "sum"), (16, "sum"), (2, "min")]


def test_tcgen05_local_update_still_tries_peer_memory_first(monkeypatch):
    cfg, B = synth.CONFIGS["ragged"], 6
    alg, eng, dist, seen = _alg(monkeypatch, synth.reference_kwargs(cfg, replay_batch_size=B))
    assert not alg.networks._cnn
    asked = []

    def connect(e, d):
        asked.append(e)
        return False     # the ranks cannot map each other's buffers: NCCL seam
    monkeypatch.setattr(dp, "connect_peers", connect)
    alg.local_update(_batch(B, (cfg["obs_dim"],)), 1)
    assert asked == [eng]
    assert eng.calls == [("grad_phase1", B), ("grad_phase2", 2 * B), ("apply", 1)]
    assert _lib.STATE_STDSUM == 4 and seen["global_batch"] == 2 * B
