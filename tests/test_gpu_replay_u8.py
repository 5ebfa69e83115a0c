"""The 8-bit image replay ring on the GPU (dsact_cnn_replay_bind_u8 / _add_u8, gather_u8_kernel; CnnEngine.bind_replay
(obs_dtype=torch.uint8); ReplayBuffer(dsact_image_dtype="uint8")):

* an fp32 ring and an 8-bit ring holding the same transitions return identical minibatches, device-drawn and by index
  list, after a wrap-around add, for row lengths that are multiples of 16 bytes, of 4 bytes only, and neither;
* the drop-in trains the same with either ring (20 sample_batch + local_update iterations);
* the trainer's full checkpoint saves the 8-bit codes and resumes the ring exactly; checkpoints of either ring kind load
  into the other;
* the error codes of wrong pairings, and the device memory of a 200 000-row CarRacing ring."""
import ctypes as C

import numpy as np
import pytest
import torch

from dsac_v2_b200 import synth

pytestmark = pytest.mark.gpu

RING_CONFIGS = {
    "carracing": synth.CNN_CONFIGS["carracing"],                                      # 27 648-byte rows (16-byte loads)
    "word": dict(obs_dim=(3, 10, 10), act_dim=2, act_lim=1.0, conv_type="test_odd"),  # 300-byte rows (4-byte loads)
    "odd": synth.CNN_CONFIGS["odd"],                                                  # 429-byte rows (byte loads)
}


def make_engine(cfg, batch):
    from dsac_v2_b200.engine_cnn import CnnEngine, make_cnn_config
    t = synth.CONV_TYPES[cfg["conv_type"]]
    c = make_cnn_config(cfg["obs_dim"], cfg["act_dim"], t["kernels"], t["channels"], t["strides"], t["heads"], max_batch=batch)
    lim = torch.full((cfg["act_dim"],), cfg["act_lim"])
    return CnnEngine(c, torch.device("cuda", 0), lim, -lim)


def on_grid(g, shape):
    """float32 images as rgb / 255 environments emit them"""
    return (g.integers(0, 256, size=shape) / 255.0).astype(np.float32)


def transitions(g, cfg, n):
    return [(on_grid(g, cfg["obs_dim"]), {}, g.uniform(-1, 1, cfg["act_dim"]).astype(np.float32), float(g.standard_normal()),
             on_grid(g, cfg["obs_dim"]), bool(g.random() < 0.1), np.float32(g.standard_normal()), {}) for _ in range(n)]


# ---- 1. the same minibatches from both kinds of ring -----------------------------------------------------------------
@pytest.mark.parametrize("name", list(RING_CONFIGS))
def test_u8_ring_samples_what_the_fp32_ring_samples(name):
    from training.replay_buffer import decode_u8
    cfg, B, cap = RING_CONFIGS[name], 32, 40
    O, A = int(np.prod(cfg["obs_dim"])), cfg["act_dim"]
    f32, u8 = make_engine(cfg, B), make_engine(cfg, B)
    f32.seed(7); u8.seed(7)
    f32.bind_replay(cap)
    u8.bind_replay(cap, obs_dtype=torch.uint8)
    assert u8.replay["obs"].dtype == torch.uint8 and set(u8.replay) == set(f32.replay)
    g = np.random.default_rng(1)
    n = 65
    codes = {k: g.integers(0, 256, size=(n, O), dtype=np.uint8) for k in ("obs", "obs2")}
    rest = {"act": g.standard_normal((n, A)).astype(np.float32), "rew": g.standard_normal(n).astype(np.float32),
            "done": (g.random(n) < 0.2).astype(np.float32), "logp": g.standard_normal(n).astype(np.float32)}
    keep = []
    for lo, hi in ((0, 30), (30, 65)):   # the second add wraps: rows 30..39, then 0..24
        s8 = {k: torch.from_numpy(v[lo:hi]).cuda() for k, v in codes.items()}
        s32 = {k: torch.from_numpy(decode_u8(v[lo:hi])).cuda() for k, v in codes.items()}
        for k, v in rest.items():
            s8[k] = s32[k] = torch.from_numpy(v[lo:hi]).cuda()
        f32.replay_add(s32, hi - lo, lo % cap)
        u8.replay_add(s8, hi - lo, lo % cap)
        keep += [s8, s32]
    torch.cuda.synchronize()
    ring = np.arange(n)[-cap:][np.argsort(np.arange(n)[-cap:] % cap)]   # transition held by each ring row
    assert torch.equal(u8.replay["obs"].cpu(), torch.from_numpy(codes["obs"][ring]))
    for draw in range(20):
        a, b = f32.replay_sample(B, cap), u8.replay_sample(B, cap)
        for k in a:
            assert torch.equal(a[k], b[k]), (name, draw, k)
    assert tuple(b["obs"].shape) == (B,) + tuple(cfg["obs_dim"])
    idx = torch.tensor([0, 39, 24, 25, 3, 3, 17, 30])
    a, b = f32.replay_sample(len(idx), cap, idx), u8.replay_sample(len(idx), cap, idx)
    for k in a:
        assert torch.equal(a[k], b[k]), (name, "idx", k)
    want = decode_u8(codes["obs2"][ring[idx.numpy()]]).reshape(b["obs2"].shape)
    assert np.array_equal(b["obs2"].cpu().numpy().view(np.uint32), want.view(np.uint32))
    assert np.array_equal(b["rew"].cpu().numpy(), rest["rew"][ring[idx.numpy()]])
    f32.close(); u8.close()


# ---- 2. the drop-in trains the same with either ring -----------------------------------------------------------------
def build_alg(cfg, B, **over):
    import dsac_v2
    kw = synth.cnn_reference_kwargs(cfg, replay_batch_size=B, seed=5, **over)
    alg = dsac_v2.DSAC_V2(**kw)
    sd = alg.networks.state_dict()
    for k, v in synth.make_cnn_weights(cfg).items():
        sd[k] = torch.from_numpy(v)
    alg.networks.load_state_dict(sd)
    alg.networks.cuda()
    return alg, kw


def test_dropin_trains_the_same_with_the_u8_ring():
    from dsac_v2_b200.engine import STAT_KEYS
    from training.replay_buffer import ReplayBuffer
    cfg, B = synth.CNN_CONFIGS["small_t1"], 16
    rows = transitions(np.random.default_rng(2), cfg, 90)
    runs = []
    for dtype in ("float32", "uint8"):
        alg, kw = build_alg(cfg, B)
        buf = ReplayBuffer(**dict(kw, buffer_max_size=64, additional_info={}, dsact_image_dtype=dtype))
        buf.attach(alg.networks.engine())
        buf.add_batch(rows)              # wraps
        tbs = []
        for it in range(20):
            tb = alg.local_update(buf.sample_batch(B), it)
            tbs.append([tb[k] for k in STAT_KEYS[:14]])
        runs.append((np.array(tbs), alg.networks.engine().params.clone(), alg.networks.engine().targets.clone()))
    (tb_a, p_a, t_a), (tb_b, p_b, t_b) = runs
    assert np.isfinite(tb_a).all()
    np.testing.assert_allclose(tb_b, tb_a, rtol=1e-4, atol=1e-6)   # fp32 atomics-order differences only
    torch.testing.assert_close(p_b, p_a, rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(t_b, t_a, rtol=2e-5, atol=2e-6)


# ---- 3. checkpoints --------------------------------------------------------------------------------------------------
class _ImageSampler:
    """Stands in for training.off_sampler.OffSampler with rgb / 255 frames."""

    def __init__(self, kw, cfg):
        import dsac_v2
        self.networks = dsac_v2.ApproxContainer(**kw)
        self.cfg, self.n, self.g = cfg, 0, np.random.default_rng(0)

    def sample(self):
        self.n += 10
        return transitions(self.g, self.cfg, 10), {"Time/Sampler time [ms]-RL iter": 0.0}

    def get_total_sample_number(self):
        return self.n


class _StubEvaluator:
    networks = None

    def run_evaluation(self, it):
        return 0.0


def test_trainer_full_checkpoint_resumes_the_u8_ring(tmp_path):
    from training.trainer import create_trainer
    from training.replay_buffer import ReplayBuffer
    cfg, B = synth.CNN_CONFIGS["small_t1"], 8

    def make(folder, **extra):
        np.random.seed(3); torch.manual_seed(3)
        alg, kw = build_alg(cfg, B)
        kw = dict(kw, buffer_max_size=56, additional_info={}, buffer_name="replay_buffer", buffer_warm_size=50,
                  max_iteration=6, log_save_interval=1000, apprfunc_save_interval=3, eval_interval=1000,
                  save_folder=str(folder), ini_network_dir=None, use_gpu=True, dsact_tensorboard=False,
                  dsact_full_checkpoint=True, sample_interval=1000, dsact_image_dtype="uint8", **extra)   # no new rows after iteration 0
        buf = ReplayBuffer(**kw)
        return create_trainer(alg, _ImageSampler(kw, cfg), buf, _StubEvaluator(), **kw), alg, buf

    full, alg_full, buf_full = make(tmp_path / "full")
    full.train()
    ck = tmp_path / "full" / "apprfunc" / "trainstate_3.pkl"
    st = torch.load(ck, weights_only=False)
    data = st["buffer"]["data"]
    assert data["obs"].dtype == torch.uint8 and data["obs2"].dtype == torch.uint8 and data["act"].dtype == torch.float32
    assert st["buffer"]["size"] == 56 and st["buffer"]["ptr"] == 4   # 60 rows: the ring wrapped before the checkpoint
    resumed, alg_res, buf_res = make(tmp_path / "resumed", dsact_resume_dir=str(ck))
    assert resumed.iteration == 4
    for k, v in data.items():
        assert torch.equal(buf_res.engine.replay[k].cpu(), v), k
    resumed.train()
    for k in buf_full.engine.replay:
        assert torch.equal(buf_res.engine.replay[k], buf_full.engine.replay[k]), k
    # the resumed run made the updates of iterations 4 and 5 of the full run
    for (k, va), vb in zip(alg_full.networks.state_dict().items(), alg_res.networks.state_dict().values()):
        torch.testing.assert_close(va, vb, rtol=2e-5, atol=1e-7, msg=k)


def test_checkpoints_load_across_ring_kinds():
    from training.replay_buffer import ReplayBuffer, decode_u8
    cfg, B = synth.CNN_CONFIGS["small_t1"], 8
    alg, kw = build_alg(cfg, B)
    eng = alg.networks.engine()
    rows = transitions(np.random.default_rng(4), cfg, 30)
    bufs = {}
    for dtype in ("float32", "uint8"):
        buf = ReplayBuffer(**dict(kw, buffer_max_size=40, additional_info={}, dsact_image_dtype=dtype))
        buf.attach(eng)                  # binding a ring replaces the engine's previous one
        buf.add_batch(rows)
        bufs[dtype] = buf.state_dict()
    ck32, ck8 = bufs["float32"]["data"], bufs["uint8"]["data"]
    assert ck32["obs"].dtype == torch.float32 and ck8["obs"].dtype == torch.uint8
    assert ck8["obs"].numel() * 4 == ck32["obs"].numel() * ck32["obs"].element_size()
    for src, dtype in ((bufs["float32"], "uint8"), (bufs["uint8"], "float32")):
        buf = ReplayBuffer(**dict(kw, buffer_max_size=40, additional_info={}, dsact_image_dtype=dtype))
        buf.attach(eng)
        buf.load_state_dict(src)
        for k in ("obs", "obs2"):
            got = buf.engine.replay[k][:30].cpu()
            if dtype == "uint8":
                assert torch.equal(got, ck8[k])
            else:
                assert torch.equal(got, torch.from_numpy(decode_u8(ck8[k].numpy()))) and torch.equal(got, ck32[k])
        for k in ("act", "rew", "done", "logp"):
            assert torch.equal(buf.engine.replay[k][:30].cpu(), ck32[k])
    bad = dict(bufs["float32"], data=dict(ck32, obs=ck32["obs"] * 0.5))   # half of the codes fall between grid points
    buf = ReplayBuffer(**dict(kw, buffer_max_size=40, additional_info={}, dsact_image_dtype="uint8"))
    buf.attach(eng)
    with pytest.raises(ValueError, match="not k / 255"):
        buf.load_state_dict(bad)


# ---- 4. error codes --------------------------------------------------------------------------------------------------
def test_wrong_ring_pairings_return_error_codes():
    from dsac_v2_b200 import _lib
    from dsac_v2_b200.engine_cnn import CnnEngine, make_heads_config
    cfg = synth.CONFIGS["ragged"]
    lim = torch.full((cfg["act_dim"],), cfg["act_lim"])
    vec = CnnEngine(make_heads_config(cfg["obs_dim"], cfg["act_dim"], cfg["hidden"], "mlp_separated", max_batch=4),
                    torch.device("cuda", 0), lim, -lim)
    lib = vec.lib
    with pytest.raises(_lib.DsactError, match="n_conv = 0"):
        vec.bind_replay(8, obs_dtype=torch.uint8)
    z = torch.zeros(8 * 64, dtype=torch.uint8, device="cuda")
    f = torch.zeros(64, device="cuda")
    rb = _lib.ReplayU8(z.data_ptr(), z.data_ptr(), f.data_ptr(), f.data_ptr(), f.data_ptr(), f.data_ptr(), 8)
    assert lib.dsact_cnn_replay_bind_u8(vec.h, C.byref(rb)) == -1 and "n_conv = 0" in lib.dsact_last_error().decode()
    vec.close()

    img = RING_CONFIGS["odd"]
    eng = make_engine(img, 4)
    O, A, s = eng.obs_elems, img["act_dim"], eng._stream()
    st8 = {k: torch.zeros(2, O, dtype=torch.uint8, device="cuda") for k in ("obs", "obs2")}
    st32 = {k: torch.zeros(2, O, device="cuda") for k in ("obs", "obs2")}
    for st in (st8, st32):
        st.update(act=torch.zeros(2, A, device="cuda"), rew=torch.zeros(2, device="cuda"), done=torch.zeros(2, device="cuda"),
                  logp=torch.zeros(2, device="cuda"))
    args = lambda st: [st[k].data_ptr() for k in ("obs", "obs2", "act", "rew", "done", "logp")] + [2, 0, s]
    eng.bind_replay(8)
    assert lib.dsact_cnn_replay_add_u8(eng.h, *args(st8)) == -3 and "fp32" in lib.dsact_last_error().decode()
    assert lib.dsact_cnn_replay_add(eng.h, *args(st32)) == 0
    eng.bind_replay(8, obs_dtype=torch.uint8)
    assert lib.dsact_cnn_replay_add(eng.h, *args(st32)) == -3 and "8-bit" in lib.dsact_last_error().decode()
    with pytest.raises(_lib.DsactError, match="8-bit"):
        eng.replay_add(st32, 2, 0)
    assert lib.dsact_cnn_replay_add_u8(eng.h, *args(st8)) == 0
    eng.bind_replay(8)                   # the last bind decides
    assert lib.dsact_cnn_replay_add(eng.h, *args(st32)) == 0
    torch.cuda.synchronize()
    eng.close()


# ---- 5. device memory of a CarRacing-sized ring ----------------------------------------------------------------------
def test_u8_carracing_ring_of_200k_rows_fits_in_a_quarter():
    cap, limit = 200_000, 11.2e9
    free, _ = torch.cuda.mem_get_info(0)
    if free < limit + 2e9:
        pytest.skip(f"{free / 1e9:.1f} GB free on the shared device; the ring needs {limit / 1e9:.1f} GB")
    eng = make_engine(synth.CNN_CONFIGS["carracing"], 4)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated(0)
    eng.bind_replay(cap, obs_dtype=torch.uint8)
    grown = torch.cuda.memory_allocated(0) - before
    O = 3 * 96 * 96
    assert 2 * cap * O <= grown <= limit, grown     # fp32 would be 4 * (2 * O + 6) * cap = 44.2 GB
    eng.close()
    del eng
    torch.cuda.empty_cache()
