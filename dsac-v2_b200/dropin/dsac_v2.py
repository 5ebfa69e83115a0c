"""`dsac_v2` of the drop-in: `ApproxContainer` and `DSAC_V2` with the reference's
names, kwargs and return values (reference dsac_v2.py:19-62, 66-347), backed by
the B200 engine (libdsact.so) instead of eager PyTorch.

* `ApproxContainer` stays an `nn.Module` with the reference's parameter names and
  53-key `state_dict`; once on a CUDA device its parameters are views into the
  engine's flat buffers (params / targets), and Adam moments live beside them.
* `DSAC_V2.local_update(data, iteration) -> tb_info` runs the whole update
  (losses, three backward passes, Adam, delayed Polyak) in the CUDA library.
  There is no CPU fallback: on a CPU module it raises.
* `get_remote_update_info` / `remote_update` keep the gradient-message seam
  (reference :107-138); with `torch.distributed` initialised the step is
  data-parallel (all-reduce of the two critic-std sums and of the flat gradients).
  Both hold for every configuration: the MLP approximators on the tcgen05 engine,
  and the CNN approximators / policy std types mlp_separated and parameter on the
  head-wise engine (whose data-parallel exchange is torch.distributed only, so
  `dsact_dp_transport="peer"` means NCCL for those configurations).

Extra kwargs (all optional): `dsact_noise` = "device" (Philox on the GPU, default)
or "reference" (draw the 8 normals of one update from torch's CPU generator in the
reference's order, SURVEY Appendix B — same seed, same numbers as the reference);
`dsact_gemm` = "bf16x3" (tcgen05 split-precision, default) | "fp32" | "bf16" (outside the parity gate); `dsact_graph` = True; `dsact_max_batch`.
"""
__all__ = ["ApproxContainer", "DSAC_V2"]

import time
import weakref
from collections.abc import Mapping
from copy import deepcopy
from typing import Dict, Tuple

import torch
import torch.nn as nn

import networks.cnn as _cnn
import networks.mlp as _mlp
from dsact_host import TB_TAGS as tb_tags
from dsact_host import net_kwargs

from dsac_v2_b200 import _lib, dp
from dsac_v2_b200.engine import STAT_KEYS, Engine, make_config
from dsac_v2_b200.engine_cnn import CnnEngine, make_cnn_config, make_heads_config

_TRAINABLE = ("q1", "q2", "policy")


class ApproxContainer(nn.Module):
    """Six networks + log_alpha (reference dsac_v2.py:19-62)."""

    def __init__(self, **kwargs):
        super().__init__()
        if kwargs.get("cnn_shared", False):
            raise NotImplementedError("cnn_shared feature nets are not part of the B200 update path")
        q_args, pi_args = net_kwargs("value", kwargs), net_kwargs("policy", kwargs)
        if q_args["apprfunc"] != pi_args["apprfunc"]:
            raise NotImplementedError("value and policy approximators must be of the same type (both MLP or both CNN)")
        self._cnn = q_args["apprfunc"] == "CNN"   # BASELINE config 5: conv encoder + separate mean / log_std heads
        self._heads_std = None
        mod = _cnn if self._cnn else _mlp
        q_cls, pi_cls = getattr(mod, q_args["name"], None), getattr(mod, pi_args["name"], None)
        if q_cls is None or pi_cls is None:
            raise NotImplementedError("This apprfunc is not properly defined")
        # construction order q1, q2, policy = the reference's consumption of torch's RNG (:31-39)
        self.q1 = q_cls(**q_args)
        self.q2 = q_cls(**q_args)
        self.q1_target = deepcopy(self.q1)
        self.q2_target = deepcopy(self.q2)
        self.policy = pi_cls(**pi_args)
        self.policy_target = deepcopy(self.policy)
        for net in (self.policy_target, self.q1_target, self.q2_target):
            for p in net.parameters():
                p.requires_grad = False
        self.log_alpha = nn.Parameter(torch.tensor(1, dtype=torch.float32))

        if pi_args["action_distribution_cls"].__name__ not in _lib.ACT_DISTS:
            raise NotImplementedError("the B200 engine implements TanhGaussDistribution and GaussDistribution")
        common = dict(gamma=kwargs.get("gamma", 0.99), tau=kwargs.get("tau", 0.005), tau_b=kwargs.get("tau_b", None),
                      delay_update=kwargs.get("delay_update", 2), auto_alpha=kwargs.get("auto_alpha", True),
                      alpha=kwargs.get("alpha", 0.2), lr_q=kwargs["value_learning_rate"], lr_pi=kwargs["policy_learning_rate"],
                      lr_alpha=kwargs["alpha_learning_rate"], min_log_std=pi_args["min_log_std"], max_log_std=pi_args["max_log_std"],
                      act_dist=pi_args["action_distribution_cls"].__name__)
        if self._cnn:
            if q_args["conv_type"] != pi_args["conv_type"] or q_args["hidden_activation"] != pi_args["hidden_activation"]:
                raise NotImplementedError("the CNN engine takes one conv_type / head activation for critics and policy")
            t = _cnn.CONV_TYPES[q_args["conv_type"]]
            self._cfg_args = dict(obs_shape=tuple(q_args["obs_dim"]), act_dim=q_args["act_dim"], kernels=t["kernels"],
                                  channels=t["channels"], strides=t["strides"], hidden=t["heads"],
                                  act_hidden=q_args["hidden_activation"], **common)
        elif pi_args["std_type"] != "mlp_shared":
            # separate mean / log_std (reference networks/mlp.py:43-72): the head-wise fp32 engine without an encoder
            if q_args["hidden_sizes"] != pi_args["hidden_sizes"] or q_args["hidden_activation"] != pi_args["hidden_activation"]:
                raise NotImplementedError("policy std_type != 'mlp_shared': critics and policy take one hidden_sizes / activation")
            self._cnn = True     # same engine class and entry points as the CNN approximators
            self._heads_std = pi_args["std_type"]
            self._cfg_args = dict(obs_dim=q_args["obs_dim"], act_dim=q_args["act_dim"], hidden=q_args["hidden_sizes"],
                                  std_type=pi_args["std_type"], act_hidden=q_args["hidden_activation"], **common)
        else:
            self._cfg_args = dict(
                obs_dim=q_args["obs_dim"], act_dim=q_args["act_dim"],
                hidden_q=q_args["hidden_sizes"], hidden_pi=pi_args["hidden_sizes"],
                act_q=q_args["hidden_activation"], act_pi=pi_args["hidden_activation"],
                gemm_mode=kwargs.get("dsact_gemm", "bf16x3"), use_graph=kwargs.get("dsact_graph", True), **common)
        if q_args["output_activation"] != "linear" or pi_args["output_activation"] != "linear":
            raise NotImplementedError("the B200 engine implements linear output activations")
        self._max_batch = int(kwargs.get("dsact_max_batch", kwargs.get("replay_batch_size", 256)))
        self._engine = None
        # seed of the device generator (noise + replay indices): the run's `seed` kwarg (reference utils/init_args.py
        # seeds torch/numpy with it) mixed with the data-parallel rank, so that seeds and ranks draw independent streams
        self._user_seed = kwargs.get("seed", None)
        self._attachments = []   # objects holding a reference to the engine (ReplayBuffer): re-bound when the engine is rebuilt
        self._register_state_dict_hook(_detach_state_dict)

    def create_action_distributions(self, logits):
        return self.policy.get_act_dist(logits)

    # ---- flat-buffer plumbing -----------------------------------------------------
    def _flat_groups(self):
        """(flat tensor name, [parameters in layout order]) — include/dsact.h layout."""
        train = [p for n in _TRAINABLE for p in getattr(self, n).parameters()] + [self.log_alpha]
        targ = [p for n in _TRAINABLE for p in getattr(self, n + "_target").parameters()]
        return train, targ

    def _apply(self, fn, recurse=True):
        super()._apply(fn, recurse)
        if self.log_alpha.device.type == "cuda":
            self._attach(self.log_alpha.device)
        return self

    def _attach(self, device):
        """Make every parameter a view into the engine's flat buffers on `device`."""
        eng = self._engine
        if eng is not None and eng.device != torch.device(device):
            self._engine = eng = None  # moved to another GPU: rebuild there
        if eng is None and self._cnn:
            make = make_heads_config if self._heads_std else make_cnn_config
            cfg = make(max_batch=self._max_batch, **self._cfg_args)
            eng = self._engine = CnnEngine(cfg, device, self.policy.act_high_lim, self.policy.act_low_lim)
            eng.seed(self.device_seed())
        elif eng is None:
            cfg = make_config(max_batch=self._max_batch, **self._cfg_args)
            eng = self._engine = Engine(cfg, device, self.policy.act_high_lim, self.policy.act_low_lim)
            eng.seed(self.device_seed())
        train, targ = self._flat_groups()
        with torch.no_grad():
            for flat, group in ((eng.params, train), (eng.targets, targ)):
                off = 0
                for p in group:
                    n = p.numel()
                    view = flat[off:off + n].view(p.shape)
                    if p.data.data_ptr() != view.data_ptr():
                        view.copy_(p.data)
                        p.data = view
                    off += n
                assert off == flat.numel(), "flat layout does not match the module"

    def device_seed(self) -> int:
        """64-bit seed of the engine's Philox generator: splitmix64 of (user seed, data-parallel rank)."""
        rank = 0
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                rank = dist.get_rank()
        except Exception:   # noqa: BLE001
            rank = 0
        base = 0x5DEECE66D if self._user_seed is None else int(self._user_seed)
        z = (base * 0x9E3779B97F4A7C15 + (rank + 1) * 0xBF58476D1CE4E5B9) & (2 ** 64 - 1)
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & (2 ** 64 - 1)
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & (2 ** 64 - 1)
        return z ^ (z >> 31)

    def engine(self, batch: int = 0) -> Engine:
        """The bound engine; raises when the module is not on a CUDA device."""
        if self.log_alpha.device.type != "cuda" or self._engine is None:
            raise _lib.DsactError(
                "DSAC_V2's update path runs only on the CUDA engine (libdsact.so, sm_100a); "
                "move the networks to the GPU first (`alg.networks.cuda()`). There is no CPU fallback.")
        if batch > self._max_batch and self._cnn:
            raise ValueError(f"batch {batch} > dsact_max_batch / replay_batch_size {self._max_batch} (the CNN engine does not regrow)")
        if batch > self._max_batch:  # grow the activation arena, keep weights / Adam state / carry
            old = self._engine
            self._max_batch = int(batch)
            cfg = make_config(max_batch=self._max_batch, **self._cfg_args)
            new = Engine(cfg, old.device, self.policy.act_high_lim, self.policy.act_low_lim)
            with torch.no_grad():
                for name in ("params", "targets", "adam_m", "adam_v", "state"):
                    getattr(new, name).copy_(getattr(old, name))
            new.seed(old._seed)            # a seed restored by load_full_state_dict survives the rebuild
            self._engine = new
            for p in self.parameters():  # force re-pointing
                p.data = p.data.clone()
            self._attach(old.device)
            for ref in list(self._attachments):   # replay rings move with their rows; peers reconnect on the next update
                obj = ref()
                if obj is not None:
                    obj.rebind(old, new)
            old.close()
        return self._engine

    def grad_views(self):
        """Per-parameter views of the flat gradient buffer, grouped like get_remote_update_info."""
        eng = self.engine()
        out, off = {}, 0
        for name in _TRAINABLE:
            views = []
            for p in getattr(self, name).parameters():
                views.append(eng.grads[off:off + p.numel()].view(p.shape))
                off += p.numel()
            out[name] = views
        out["log_alpha"] = eng.grads[off]
        return out


def _detach_state_dict(module, state_dict, prefix, local_metadata):
    # checkpoints must not alias the flat buffers (torch.save would serialise the whole storage per view)
    for k, v in list(state_dict.items()):
        if isinstance(v, torch.Tensor):
            state_dict[k] = v.detach().clone()
    return state_dict


class _LazyTbInfo(Mapping):
    """tb_info whose 14 device-computed scalars are fetched on first access (one event wait),
    so a training loop that only logs every N iterations never stalls on `.item()`."""

    def __init__(self, slot, event, alg_ms):
        self._slot, self._event, self._alg_ms, self._vals = slot, event, alg_ms, None

    def _materialise(self):
        if self._vals is None:
            self._event.synchronize()
            err = float(self._slot[14])
            if err != 0.0:   # include/dsact.h: tb_info slot 14 = 1 + rank of a peer that never arrived
                raise _lib.DsactError(f"data-parallel exchange timed out waiting for rank {int(err) - 1}")
            vals = dict(zip(STAT_KEYS, self._slot.tolist()))
            vals[tb_tags["alg_time"]] = self._alg_ms
            self._vals, self._slot = vals, None
        return self._vals

    def __getitem__(self, k):
        return self._materialise()[k]

    def __iter__(self):
        return iter(self._materialise())

    def __len__(self):
        return len(STAT_KEYS) + 1


class DSAC_V2:
    """DSAC-T (arXiv 2310.05858) on the B200 engine; interface of reference dsac_v2.py:66-138."""

    _RING = 32

    def __init__(self, **kwargs):
        self.networks = ApproxContainer(**kwargs)
        self.gamma = kwargs["gamma"]
        self.tau = kwargs["tau"]
        self.target_entropy = -kwargs["action_dim"]
        self.auto_alpha = kwargs["auto_alpha"]
        self.alpha = kwargs.get("alpha", 0.2)
        self.delay_update = kwargs["delay_update"]
        self.tau_b = kwargs.get("tau_b", self.tau)
        self.act_dim = kwargs["action_dim"]
        self.noise_source = kwargs.get("dsact_noise", "device")
        if self.noise_source not in ("device", "reference"):
            raise ValueError("dsact_noise must be 'device' or 'reference'")
        self.data_parallel = kwargs.get("dsact_data_parallel", True)
        # "peer": exchanges inside the step's kernels over NVLink peer memory (falls back to NCCL if the ranks cannot
        # map each other's buffers); "nccl": torch.distributed all-reduces between three graph launches.  The head-wise
        # engine (CNN approximators, policy std types mlp_separated / parameter) has no peer-memory exchange: for those
        # configurations both values mean torch.distributed all-reduces between its phase launches
        self.dp_transport = kwargs.get("dsact_dp_transport", "peer")
        self._peer_dp, self._peer_eng = None, None
        self._slots, self._owners, self._cursor = None, [None] * self._RING, 0

    @property
    def adjustable_parameters(self):
        return ("gamma", "tau", "auto_alpha", "alpha", "delay_update")

    @property
    def mean_std1(self):
        return float(self.networks.engine().state[0])

    @property
    def mean_std2(self):
        return float(self.networks.engine().state[1])

    # ---- helpers ------------------------------------------------------------------
    def _noise(self, batch: int):
        if self.noise_source == "device":
            return None
        A = self.act_dim
        eps1 = torch.empty(batch, A).normal_()   # rsample of pi(obs),        reference :160
        eps2 = torch.empty(batch, A).normal_()   # rsample of pi_target(obs2), reference :228
        z = [torch.normal(torch.zeros(batch), torch.ones(batch)) for _ in range(6)]  # __q_evaluate x6
        return eps1, eps2, z[2], z[3]

    def _world(self):
        return dp.world() if self.data_parallel else (None, 1)

    def _stats(self, eng, global_batch, t0):
        if self._slots is None:
            self._slots = [torch.zeros(_lib.NUM_STATS, dtype=torch.float32).pin_memory() for _ in range(self._RING)]
        i = self._cursor
        self._cursor = (i + 1) % self._RING
        prev = self._owners[i]() if self._owners[i] is not None else None
        if prev is not None:
            prev._materialise()  # its pinned slot is about to be reused
        eng.read_stats_async(global_batch, out=self._slots[i])
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(eng.device))
        info = _LazyTbInfo(self._slots[i], ev, (time.time() - t0) * 1000)
        self._owners[i] = weakref.ref(info)
        return info

    def _gradients(self, data, eng):
        """Everything up to (and including) the gradients; returns the global batch size."""
        B = data["obs"].shape[0]
        noise = self._noise(B)
        dist, world = self._world()
        if world == 1:
            eng.compute_grads(data, noise)
            return B
        # every rank holds `B` rows of the global minibatch (the trainer samples B per rank)
        return dp.data_parallel_gradients(eng, data, noise, dist, B, B * world)

    # ---- full training state (SURVEY §8f rank 3; the reference saves weights only, training/trainer.py:137-152) ----
    def full_state_dict(self) -> dict:
        """Everything a bit-for-bit resume needs beyond the 53-key `networks.state_dict()`: Adam moments and step
        counters, the mean_std EMA pair, the device generator's seed/counter."""
        eng = self.networks.engine()
        st = eng.state.detach().cpu()
        ints = st[:16].view(torch.int32)
        return {
            "format": "dsact-full-state-1",
            "networks": self.networks.state_dict(),
            "adam_m": eng.adam_m.detach().cpu().clone(),
            "adam_v": eng.adam_v.detach().cpu().clone(),
            "mean_std": [float(st[0]), float(st[1])],
            "adam_steps": [int(ints[8]), int(ints[9])],
            "rng_counter": int(ints[10]) & 0xFFFFFFFF,
            "rng_seed": int(getattr(eng, "_seed", 0)),
        }

    def load_full_state_dict(self, state: dict) -> None:
        if state.get("format") != "dsact-full-state-1":
            raise ValueError("not a dsact full-state checkpoint")
        self.networks.load_state_dict(state["networks"])
        eng = self.networks.engine()
        with torch.no_grad():
            eng.adam_m.copy_(state["adam_m"])
            eng.adam_v.copy_(state["adam_v"])
            ints = eng.state[:16].view(torch.int32)
            ints[10] = int(state["rng_counter"]) - (1 << 32 if int(state["rng_counter"]) >= (1 << 31) else 0)
        eng.set_carry(state["mean_std"][0], state["mean_std"][1], state["adam_steps"][0], state["adam_steps"][1])
        eng.seed(state["rng_seed"])

    # ---- reference interface ------------------------------------------------------
    def local_update(self, data: Dict, iteration: int) -> dict:
        t0 = time.time()
        B = data["obs"].shape[0]
        eng = self.networks.engine(B)
        dist, world = self._world()
        if world == 1:
            eng.step(data, iteration, self._noise(B))
            return self._stats(eng, B, t0)
        if not self.networks._cnn:   # the tcgen05 engine; the head-wise engine exchanges through torch.distributed only
            if self._peer_dp is None or self._peer_eng is not eng:   # first data-parallel update (or the engine was rebuilt):
                self._peer_dp = self.dp_transport != "nccl" and dp.connect_peers(eng, dist)   # map the exchange buffers (collective)
                self._peer_eng = eng
            if self._peer_dp:           # one graph launch; exchanges inside the step's kernels over NVLink peer memory
                eng.dp_step(data, iteration, B * world, self._noise(B))
                return self._stats(eng, B * world, t0)
        gb = self._gradients(data, eng)
        eng.apply(iteration)
        return self._stats(eng, gb, t0)

    def get_remote_update_info(self, data: Dict, iteration: int) -> Tuple[dict, dict]:
        t0 = time.time()
        eng = self.networks.engine(data["obs"].shape[0])
        gb = self._gradients(data, eng)
        g = self.networks.grad_views()
        update_info = {"q1_grad": g["q1"], "q2_grad": g["q2"], "policy_grad": g["policy"], "iteration": iteration}
        if self.auto_alpha:
            update_info["log_alpha_grad"] = g["log_alpha"]
        return self._stats(eng, gb, t0), update_info

    def remote_update(self, update_info: dict):
        eng = self.networks.engine()
        g = self.networks.grad_views()
        with torch.no_grad():
            for key, name in (("q1_grad", "q1"), ("q2_grad", "q2"), ("policy_grad", "policy")):
                for dst, src in zip(g[name], update_info[key]):
                    if src.data_ptr() != dst.data_ptr():
                        dst.copy_(src)
            if self.auto_alpha and update_info["log_alpha_grad"].data_ptr() != g["log_alpha"].data_ptr():
                g["log_alpha"].copy_(update_info["log_alpha_grad"])
        eng.apply(update_info["iteration"])
