"""`training.replay_buffer` of the drop-in: the reference's `ReplayBuffer`
interface (reference training/replay_buffer.py:15-90) over a DEVICE-resident ring
buffer.  Transitions are staged in pinned host memory and copied to the GPU
asynchronously; `sample_batch` is a coalesced row gather on the GPU
(libdsact `dsact_replay_sample`), so no H2D copy sits on the update step.

Uniform sampling with replacement, like `np.random.randint` (reference :86).
`index_source="numpy"` draws the indices from numpy's global generator exactly as
the reference does (same seed -> same minibatch rows); the default "device" draws
them with Philox on the GPU.

`dsact_image_dtype="uint8"` (image observations only) stores every pixel as its
8-bit code k, the pixel being float32(k) / 255: a quarter of the fp32 ring's
device memory, the same minibatches.  It is exact for environments that emit
rgb / 255 (the reference's gym_carracingraw); a pixel that has no such code is
refused with ValueError, never rounded.
"""
__all__ = ["ReplayBuffer", "DECODE_U8", "encode_u8", "decode_u8"]

import numpy as np
import torch

# float32(k) / 255 for every code k, by IEEE correctly-rounded fp32 division: equal to the float64 k / 255 cast to
# float32, which is what rgb / 255 environments produce.  (k * float32(1 / 255) differs for about half of the codes.)
DECODE_U8 = np.arange(256, dtype=np.float32) / np.float32(255)


def encode_u8(x) -> np.ndarray:
    """8-bit codes of pixels on the 1/255 grid: k = rint(x * 255), kept only if DECODE_U8[k] equals x bit for bit.
    Raises ValueError naming the first pixel that has no code (off the grid, outside [0, 1], -0.0, NaN)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    k = np.rint(x * np.float32(255))
    ok = (k >= 0) & (k <= 255)
    codes = np.where(ok, k, 0).astype(np.uint8)
    ok &= DECODE_U8[codes].view(np.uint32) == x.view(np.uint32)
    if not ok.all():
        j = int(np.flatnonzero(~ok.reshape(-1))[0])
        v = float(x.reshape(-1)[j])
        raise ValueError(f"pixel {j} = {v!r} is not k / 255 for an integer k in [0, 255]: the 8-bit replay ring "
                         "(dsact_image_dtype='uint8') stores only rgb / 255 images; use dsact_image_dtype='float32'")
    return codes


def decode_u8(codes) -> np.ndarray:
    """float32 pixels of 8-bit codes (exact inverse of encode_u8)."""
    return DECODE_U8[np.asarray(codes, dtype=np.uint8)]


class ReplayBuffer:
    _STAGE_ROWS = 4096
    _STAGES = 4

    def __init__(self, index=0, **kwargs):
        self.obsv_dim = kwargs["obsv_dim"]
        self.act_dim = kwargs["action_dim"]
        self.max_size = int(kwargs["buffer_max_size"])
        if not np.isscalar(self.act_dim):
            raise NotImplementedError("the device ring buffer stores flat action vectors")
        # image observations (CNN path, BASELINE config 5): rows hold the flattened [C*H*W] image
        self.obs_shape = None if np.isscalar(self.obsv_dim) else tuple(int(x) for x in self.obsv_dim)
        self.obs_elems = int(self.obsv_dim) if self.obs_shape is None else int(np.prod(self.obs_shape))
        if kwargs.get("additional_info"):
            raise NotImplementedError("additional_info fields are not supported by the device ring buffer")
        self.image_dtype = kwargs.get("dsact_image_dtype", "float32")
        if self.image_dtype not in ("float32", "uint8"):
            raise ValueError(f"dsact_image_dtype must be 'float32' or 'uint8', not {self.image_dtype!r}")
        if self.image_dtype == "uint8" and self.obs_shape is None:
            raise ValueError("dsact_image_dtype='uint8' stores image observations; vector observations (obsv_dim "
                             f"{self.obsv_dim}) are not on the 1/255 grid and stay float32")
        self._u8 = self.image_dtype == "uint8"
        self.index_source = kwargs.get("dsact_index_source",
                                       "numpy" if kwargs.get("dsact_noise") == "reference" else "device")
        self.ptr, self.size = 0, 0
        self.engine = None
        self._stage = None      # pinned staging buffers
        self._events = None
        self._cur, self._fill, self._flushed = 0, 0, 0
        self._pending = []      # transitions stored before an engine was attached

    # ---- wiring -------------------------------------------------------------------
    def attach(self, engine):
        """Bind the ring storage to an engine (done by the trainer once the networks are on the GPU)."""
        eng_obs = getattr(engine, "obs_elems", None) or engine.cfg.obs_dim
        if eng_obs != self.obs_elems or engine.cfg.act_dim != self.act_dim:
            raise ValueError("replay buffer and engine disagree on obs/act dimensions")
        self.engine = engine
        self._bind(engine)
        O, A = self.obs_elems, self.act_dim
        img_bytes = 1 if self._u8 else 4
        R = min(self._STAGE_ROWS if self.obs_shape is None else max(8, self._STAGE_ROWS * 1600 // (img_bytes * O)), self.max_size)   # ~6 MB per staging set
        self._rows = R
        pin = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype).pin_memory()
        img = torch.uint8 if self._u8 else torch.float32
        self._stage = [dict(obs=pin(R, O, dtype=img), obs2=pin(R, O, dtype=img), act=pin(R, A), rew=pin(R), done=pin(R), logp=pin(R))
                       for _ in range(self._STAGES)]
        self._np = [{k: v.numpy() for k, v in s.items()} for s in self._stage]
        self._events = [None] * self._STAGES
        pending, self._pending = self._pending, []
        for row in pending:
            self._store_row(*row)

    def _bind(self, engine):
        if self._u8:
            engine.bind_replay(self.max_size, obs_dtype=torch.uint8)
        else:
            engine.bind_replay(self.max_size)

    def rebind(self, old, new):
        """The engine was rebuilt (larger activation arena): give the new one a ring and move the stored rows."""
        if self.engine is not old:
            return
        self.flush()
        torch.cuda.current_stream(old.device).synchronize()
        self._bind(new)
        for k, v in old.replay.items():
            new.replay[k].copy_(v)
        self.engine = new

    def _require_engine(self):
        if self.engine is None:
            raise RuntimeError("ReplayBuffer is not attached to the CUDA engine: call buffer.attach(alg.networks.engine()) "
                               "(training.trainer.OffSerialTrainer does this). There is no CPU sampling path.")

    def __len__(self):
        return self.size

    def __get_RAM__(self):
        """MB of device memory holding valid transitions."""
        row_bytes = (1 if self._u8 else 4) * 2 * self.obs_elems + 4 * (self.act_dim + 3)
        return row_bytes * self.size / 1e6

    # ---- store ----------------------------------------------------------------------
    def _store_row(self, obs, act, rew, next_obs, done, logp):
        """Write one transition into the staging set; obs / next_obs are already 8-bit codes on a uint8 ring (store)."""
        if self._fill == self._rows:
            self.flush()
        if self._fill == 0 and self._events[self._cur] is not None:
            self._events[self._cur].synchronize()  # the async copy out of this staging buffer has finished
        s, i = self._np[self._cur], self._fill
        s["obs"][i] = obs.reshape(-1)
        s["obs2"][i] = next_obs.reshape(-1)
        s["act"][i] = act
        s["rew"][i] = rew
        s["done"][i] = done
        s["logp"][i] = logp
        self._fill += 1

    def store(self, obs, info, act, rew, next_obs, done, logp, next_info):
        obs, next_obs = np.asarray(obs, dtype=np.float32), np.asarray(next_obs, dtype=np.float32)
        if self._u8:   # encode and verify here, so that an off-grid image is refused by the call that stored it
            obs, next_obs = encode_u8(obs), encode_u8(next_obs)
        row = (obs, np.asarray(act, dtype=np.float32), float(rew), next_obs, float(done), float(np.asarray(logp)))
        if self.engine is None:
            self._pending.append(row)
        else:
            self._store_row(*row)
        self.size = min(self.size + 1, self.max_size)

    def add_batch(self, samples: list):
        for sample in samples:
            self.store(*sample)

    def flush(self):
        """Enqueue the async H2D copy of the staged rows into the ring."""
        if self.engine is None or self._fill == 0:
            return
        n = self._fill
        self.engine.replay_add(self._stage[self._cur], n, self.ptr)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.engine.device))
        self._events[self._cur] = ev
        self.ptr = (self.ptr + n) % self.max_size
        self._cur = (self._cur + 1) % self._STAGES
        self._fill = 0

    # ---- full-state checkpoint (SURVEY §8f rank 3) ---------------------------------------
    def state_dict(self, with_data: bool = True) -> dict:
        """ptr/size (+ the valid transitions, fetched from the device ring) for an exact resume.  An 8-bit ring saves its
        uint8 codes."""
        self.flush()
        out = {"ptr": self.ptr, "size": self.size, "max_size": self.max_size}
        if with_data and self.engine is not None:
            torch.cuda.current_stream(self.engine.device).synchronize()
            out["data"] = {k: v[:self.size].cpu().clone() for k, v in self.engine.replay.items()}
        return out

    def load_state_dict(self, state: dict) -> None:
        self._require_engine()
        if state["max_size"] != self.max_size:
            raise ValueError("replay capacity differs from the checkpoint")
        self.ptr, self.size, self._fill = int(state["ptr"]), int(state["size"]), 0
        if "data" in state:
            for k, v in state["data"].items():
                dst = self.engine.replay[k][:self.size]
                if k in ("obs", "obs2") and v.dtype != dst.dtype:   # a checkpoint of the other ring kind: convert 1024 rows at a time
                    for i in range(0, self.size, 1024):
                        dst[i:i + 1024].copy_(self._convert_images(v[i:i + 1024], dst.dtype))
                else:
                    dst.copy_(v)

    @staticmethod
    def _convert_images(v: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
        """fp32 rows -> verified 8-bit codes (ValueError off the grid), or 8-bit codes -> fp32 rows (exact)."""
        if dtype == torch.uint8:
            return torch.from_numpy(encode_u8(v.numpy()))
        if v.dtype != torch.uint8:
            raise ValueError(f"image rows of dtype {v.dtype} cannot be stored in a {dtype} ring")
        return torch.from_numpy(decode_u8(v.numpy()))

    # ---- sample -----------------------------------------------------------------------
    def sample_indices(self, batch_size: int):
        if self.index_source == "numpy":
            return torch.from_numpy(np.random.randint(0, self.size, size=batch_size))
        return None

    def sample_batch(self, batch_size: int):
        """dict of DEVICE fp32 tensors (views of the engine's minibatch arena, valid until the next sample)."""
        self._require_engine()
        if self.size == 0:
            raise ValueError("cannot sample from an empty replay buffer")
        self.flush()
        return self.engine.replay_sample(batch_size, self.size, self.sample_indices(batch_size))
