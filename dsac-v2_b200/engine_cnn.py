"""Python owner of one libdsact CNN handle (`dsact_cnn_*`, include/dsact.h): the DSAC-T update with the reference's CNN
approximators (BASELINE config 5; reference networks/cnn.py).  Same division of labour as `engine.Engine`: torch owns the
flat device buffers, every arithmetic step runs in the CUDA library; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import torch

from . import _lib
from ._lib import Batch, Buffers, CnnConfig, Layout, Noise, Replay, ReplayU8, check
from .engine import STAT_KEYS


def make_cnn_config(obs_shape: Sequence[int], act_dim: int, kernels: Sequence[int], channels: Sequence[int],
                    strides: Sequence[int], hidden: Sequence[int], *, max_batch: int, act_hidden: str = "gelu", gamma=0.99,
                    tau=0.005, tau_b=None, delay_update=2, auto_alpha=True, alpha=0.2, lr_q=1e-4, lr_pi=1e-4, lr_alpha=3e-4,
                    min_log_std=-20.0, max_log_std=0.5, q_heads: int = 2, pi_std: str = "head",
                    act_dist: str = "TanhGaussDistribution", algo: str = "DSAC_V2", bound: bool = True,
                    td_bound: float = 20.0) -> CnnConfig:
    """`q_heads` / `pi_std` select the head wiring: (2, "head") = networks/cnn.py; with no conv layers and
    obs_shape = (obs_dim, 1, 1): (1, "head") = networks/mlp.py with policy std_type "mlp_separated", (1, "row") = "parameter"."""
    if len(kernels) > _lib.MAX_CONV or len(hidden) > _lib.MAX_HIDDEN:
        raise ValueError("too many layers")
    c = CnnConfig()
    c.abi_version = _lib.ABI_VERSION
    c.channels, c.height, c.width = (int(x) for x in obs_shape)
    c.act_dim, c.n_conv, c.n_hidden = int(act_dim), len(kernels), len(hidden)
    for j, (k, ch, st) in enumerate(zip(kernels, channels, strides)):
        c.conv_kernel[j], c.conv_channels[j], c.conv_stride[j] = int(k), int(ch), int(st)
    for j, v in enumerate(hidden):
        c.hidden[j] = int(v)
    c.act_hidden = _lib.ACTIVATIONS[act_hidden]
    c.max_batch, c.auto_alpha, c.delay_update = int(max_batch), int(bool(auto_alpha)), int(delay_update)
    c.gamma, c.tau, c.tau_b = float(gamma), float(tau), float(tau if tau_b is None else tau_b)
    c.alpha_fixed = float(alpha)
    c.lr_q, c.lr_pi, c.lr_alpha = float(lr_q), float(lr_pi), float(lr_alpha)
    c.min_log_std, c.max_log_std = float(min_log_std), float(max_log_std)
    c.adam_beta1, c.adam_beta2, c.adam_eps = 0.9, 0.999, 1e-8
    c.q_heads, c.pi_std = int(q_heads), {"head": 0, "row": 1, "shared": 2}[pi_std]
    c.algo, c.v1_bound, c.td_bound = {"DSAC_V2": 0, "DSAC_V1": 1}[algo], int(bool(bound)), float(td_bound)
    c.act_dist = _lib.ACT_DISTS[act_dist]
    return c


def make_heads_config(obs_dim: int, act_dim: int, hidden: Sequence[int], std_type: str, **kw) -> CnnConfig:
    """The MLP approximators on the head-wise fp32 engine: no encoder, one two-output head per critic, the policy with any
    of the reference's std types (networks/mlp.py:43-72).  DSAC-T with "mlp_shared" normally runs on `engine.Engine`
    (tcgen05); this entry is for "mlp_separated" / "parameter" and for `algo="DSAC_V1"`."""
    return make_cnn_config((int(obs_dim), 1, 1), act_dim, (), (), (), hidden, q_heads=1,
                           pi_std={"mlp_separated": "head", "parameter": "row", "mlp_shared": "shared"}[std_type], **kw)


class CnnEngine:
    """One `dsact_cnn_handle` bound to flat torch-owned buffers on one CUDA device."""

    def __init__(self, cfg: CnnConfig, device, act_high, act_low):
        if not torch.cuda.is_available():
            raise _lib.DsactError("the DSAC-T update engine needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib, self.cfg = _lib.load(), cfg
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        lay = Layout()
        check(self.lib.dsact_cnn_query_layout(C.byref(cfg), C.byref(lay)))
        self.layout = lay
        with torch.cuda.device(self.device):
            z = lambda n: torch.zeros(int(n), dtype=torch.float32, device=self.device)
            self.params, self.targets = z(lay.n_params), z(lay.n_targets)
            self.grads, self.adam_m, self.adam_v = z(lay.n_params), z(lay.n_params), z(lay.n_params)
            self.state = z(lay.state_floats)
            self.workspace = z(int(lay.workspace_bytes) // 4 + 64)
            off = (-self.workspace.data_ptr() % 256) // 4
            self._ws_view = self.workspace[off:]
            self.act_high = torch.as_tensor(act_high, dtype=torch.float32).reshape(-1).to(self.device).clone()
            self.act_low = torch.as_tensor(act_low, dtype=torch.float32).reshape(-1).to(self.device).clone()
            h = C.c_void_p()
            check(self.lib.dsact_cnn_create(C.byref(cfg), self.device.index, C.byref(h)))
            self.h = h
            b = Buffers(self.params.data_ptr(), self.targets.data_ptr(), self.grads.data_ptr(), self.adam_m.data_ptr(),
                        self.adam_v.data_ptr(), self.act_high.data_ptr(), self.act_low.data_ptr(), self.state.data_ptr(),
                        self._ws_view.data_ptr())
            check(self.lib.dsact_cnn_bind(self.h, C.byref(b)))
            check(self.lib.dsact_cnn_set_carry(self.h, -1.0, -1.0, 0, 0, self._stream()))
            self._stats_host = torch.zeros(_lib.NUM_STATS, dtype=torch.float32).pin_memory()
        self.last_batch = 0

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def close(self):
        if getattr(self, "h", None):
            self.lib.dsact_cnn_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:   # noqa: BLE001
            pass

    # ---- flat layout in the reference's state_dict schema (include/dsact.h) --------------------------------------------
    def _schema(self):
        c = self.cfg
        out, off = [], 0
        shapes = []
        cin, hh, ww = c.channels, c.height, c.width
        for j in range(c.n_conv):
            k, co, st = c.conv_kernel[j], c.conv_channels[j], c.conv_stride[j]
            shapes.append((f"conv.{2 * j}", (co, cin, k, k), (co,)))
            cin, hh, ww = co, (hh - k) // st + 1, (ww - k) // st + 1
        feat = cin * hh * ww
        hidden = [c.hidden[j] for j in range(c.n_hidden)]

        def leaf(net, name, shape):
            nonlocal off
            n = 1
            for d in shape:
                n *= int(d)
            out.append((f"{net}.{name}", f"{net}_target.{name}", off, n, shape))
            off += n

        def mlp(net, head, sizes):
            for j in range(len(sizes) - 1):
                leaf(net, f"{head}.{2 * j}.weight", (sizes[j + 1], sizes[j]))
                leaf(net, f"{head}.{2 * j}.bias", (sizes[j + 1],))

        critics = ("q",) if c.algo == 1 else ("q1", "q2")   # dsac_v1.ApproxContainer holds ONE critic named `q`
        for net, extra, width in tuple((n, c.act_dim, 1) for n in critics) + (("policy", 0, c.act_dim),):
            for name, wshape, bshape in shapes:
                leaf(net, f"{name}.weight", wshape)
                leaf(net, f"{name}.bias", bshape)
            if net != "policy" and c.q_heads == 1:          # networks/mlp.py ActionValueDistri: self.q
                mlp(net, "q", [feat + extra] + hidden + [2])
            elif net == "policy" and c.pi_std == 2:         # networks/mlp.py std_type "mlp_shared": self.policy, 2A outputs
                mlp(net, "policy", [feat] + hidden + [2 * width])
            elif net == "policy" and c.pi_std == 1:         # the module's own parameter precedes its children's
                leaf(net, "log_std", (1, width))
                mlp(net, "mean", [feat] + hidden + [width])
            else:
                for head in ("mean", "log_std"):
                    mlp(net, head, [feat + extra] + hidden + [width])
        return out, off

    def load_weights(self, weights: dict):
        schema, n = self._schema()
        assert n == self.layout.n_targets, (n, self.layout.n_targets)
        with torch.no_grad():
            for key, tkey, off, cnt, shape in schema:
                self.params[off:off + cnt].copy_(torch.as_tensor(weights[key]).reshape(-1))
                self.targets[off:off + cnt].copy_(torch.as_tensor(weights.get(tkey, weights[key])).reshape(-1))
            self.params[n] = float(weights.get("log_alpha", 1.0))

    def export_weights(self, grads: bool = False) -> dict:
        schema, n = self._schema()
        src = (self.grads if grads else self.params).detach().cpu()
        tgt = self.targets.detach().cpu()
        out = {"log_alpha": src[n].clone()}
        for key, tkey, off, cnt, shape in schema:
            out[key] = src[off:off + cnt].view(shape).clone()
            if not grads:
                out[tkey] = tgt[off:off + cnt].view(shape).clone()
        return out

    # ---- the path -------------------------------------------------------------------------------------------------------
    def _batch(self, data: Dict[str, torch.Tensor]) -> Batch:
        """Device copies of the minibatch (kept alive on the engine until the next call that reads them) as a Batch."""
        t = {k: data[k].to(device=self.device, dtype=torch.float32).contiguous() for k in ("obs", "act", "rew", "obs2", "done")}
        B = t["obs"].shape[0]
        c = self.cfg
        if t["obs"][0].numel() != self.obs_elems or t["obs2"].shape != t["obs"].shape or t["act"].shape != (B, c.act_dim):
            raise ValueError("minibatch shapes do not match the configured observation / action shape")
        self._keep = t
        return Batch(t["obs"].data_ptr(), t["act"].data_ptr(), t["rew"].data_ptr(), t["obs2"].data_ptr(), t["done"].data_ptr(), B, None)

    def _noise(self, noise):
        """eps1, eps2, z3, z4 on the device as a Noise pointer, or None (the engine draws them)."""
        if noise is None:
            return None
        nz = [torch.as_tensor(x).to(device=self.device, dtype=torch.float32).contiguous() for x in noise]
        self._keep_noise = nz
        return C.byref(Noise(*(x.data_ptr() for x in nz)))

    def step(self, data: Dict[str, torch.Tensor], iteration: int, noise=None):
        """DSAC_V2.local_update (reference dsac_v2.py:102-105) with image observations [B, C, H, W] on the device."""
        with torch.cuda.device(self.device):
            b = self._batch(data)
            check(self.lib.dsact_cnn_step(self.h, C.byref(b), self._noise(noise), int(iteration), self._stream()))
        self.last_batch = b.batch

    # ---- split form: the gradient-message seam and data-parallel steps (dp.data_parallel_gradients) -------------------
    def grad_phase1(self, data: Dict[str, torch.Tensor], noise=None):
        """Every forward of the step on the local minibatch; leaves the local critic-std sums in state[4:6]."""
        with torch.cuda.device(self.device):
            b = self._batch(data)
            check(self.lib.dsact_cnn_grad_phase1(self.h, C.byref(b), self._noise(noise), self._stream()))
        self.last_batch = b.batch

    def grad_phase2(self, global_batch: int):
        """Losses (means over `global_batch` rows) and every backward pass of the minibatch of grad_phase1."""
        with torch.cuda.device(self.device):
            check(self.lib.dsact_cnn_grad_phase2(self.h, int(global_batch), self._stream()))

    def compute_grads(self, data: Dict[str, torch.Tensor], noise=None):
        """grad_phase1 + grad_phase2 over this minibatch alone: `grads` holds the step's gradients."""
        with torch.cuda.device(self.device):
            b = self._batch(data)
            check(self.lib.dsact_cnn_compute_grads(self.h, C.byref(b), self._noise(noise), self._stream()))
        self.last_batch = b.batch

    def apply(self, iteration: int):
        """Adam + delayed Polyak with whatever `grads` holds (DSAC_V2.remote_update)."""
        with torch.cuda.device(self.device):
            check(self.lib.dsact_cnn_apply(self.h, int(iteration), self._stream()))

    # ---- device replay ring (flattened image rows) ---------------------------------------------------------------------
    @property
    def obs_elems(self) -> int:
        return self.cfg.channels * self.cfg.height * self.cfg.width

    def bind_replay(self, capacity: int, obs_dtype: torch.dtype = torch.float32):
        """Allocate and bind the device ring.  obs_dtype=torch.uint8 stores every image pixel as its code k (the pixel is
        float32(k) / 255, decoded by the gather), a quarter of the fp32 ring's image bytes; it needs a conv encoder."""
        if obs_dtype not in (torch.float32, torch.uint8):
            raise ValueError(f"obs_dtype must be torch.float32 or torch.uint8, not {obs_dtype}")
        O, A = self.obs_elems, self.cfg.act_dim
        with torch.cuda.device(self.device):
            z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=self.device)
            r = dict(obs=z(capacity, O, dtype=obs_dtype), obs2=z(capacity, O, dtype=obs_dtype), act=z(capacity, A), rew=z(capacity),
                     done=z(capacity), logp=z(capacity))
            ptrs = (r["obs"].data_ptr(), r["obs2"].data_ptr(), r["act"].data_ptr(), r["rew"].data_ptr(), r["done"].data_ptr(),
                    r["logp"].data_ptr(), int(capacity))
            if obs_dtype == torch.uint8:
                check(self.lib.dsact_cnn_replay_bind_u8(self.h, C.byref(ReplayU8(*ptrs))))
            else:
                check(self.lib.dsact_cnn_replay_bind(self.h, C.byref(Replay(*ptrs))))
        self.replay = r
        self.capacity = int(capacity)

    def replay_add(self, staging: Dict[str, torch.Tensor], n: int, ptr: int):
        """Copy n staged rows into ring rows (ptr + i) % capacity.  uint8 obs / obs2 staging goes to an 8-bit ring, fp32
        staging to an fp32 ring; the library refuses the other pairings."""
        s = staging
        add = self.lib.dsact_cnn_replay_add_u8 if s["obs"].dtype == torch.uint8 else self.lib.dsact_cnn_replay_add
        with torch.cuda.device(self.device):
            check(add(self.h, s["obs"].data_ptr(), s["obs2"].data_ptr(), s["act"].data_ptr(), s["rew"].data_ptr(),
                      s["done"].data_ptr(), s["logp"].data_ptr(), int(n), int(ptr), self._stream()))

    def replay_sample(self, batch: int, size: int, idx: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        out = Batch()
        with torch.cuda.device(self.device):
            if idx is not None:
                idx = idx.to(device=self.device, dtype=torch.int64).contiguous()
                self._keep_idx = idx
            check(self.lib.dsact_cnn_replay_sample(self.h, int(batch), int(size), None if idx is None else idx.data_ptr(), C.byref(out),
                                                   self._stream()))
        base, c, B, A = self._ws_view.data_ptr(), self.cfg, int(batch), self.cfg.act_dim

        def view(ptr, n, shape):
            off = (ptr - base) // 4
            return self._ws_view[off:off + n].view(shape)

        img = (B, c.channels, c.height, c.width) if c.n_conv else (B, self.obs_elems)
        return {"obs": view(out.obs, B * self.obs_elems, img), "obs2": view(out.obs2, B * self.obs_elems, img),
                "act": view(out.act, B * A, (B, A)), "rew": view(out.rew, B, (B,)), "done": view(out.done, B, (B,)),
                "logp": view(out.logp, B, (B,))}

    def seed(self, seed: int):
        self._seed = int(seed) & (2 ** 64 - 1)
        check(self.lib.dsact_cnn_seed(self.h, self._seed))

    def set_carry(self, mean_std1=-1.0, mean_std2=-1.0, adam_steps_q=0, adam_steps_pi=0):
        """Overwrite the carried scalars (mean_std EMA pair, Adam step counters), as `Engine.set_carry`: the drop-in's
        load_full_state_dict restores them through this."""
        with torch.cuda.device(self.device):
            check(self.lib.dsact_cnn_set_carry(self.h, float(mean_std1), float(mean_std2), int(adam_steps_q), int(adam_steps_pi),
                                               self._stream()))

    def read_stats_async(self, global_batch: Optional[int] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        out = self._stats_host if out is None else out
        with torch.cuda.device(self.device):
            check(self.lib.dsact_cnn_read_stats(self.h, int(global_batch or self.last_batch), out.data_ptr(), self._stream()))
        return out

    def read_stats(self, global_batch: Optional[int] = None) -> Dict[str, float]:
        with torch.cuda.device(self.device):
            check(self.lib.dsact_cnn_read_stats(self.h, int(global_batch or self.last_batch), self._stats_host.data_ptr(), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()
        return dict(zip(STAT_KEYS, self._stats_host.tolist()))
