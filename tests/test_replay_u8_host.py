"""Host side of the 8-bit image replay ring (ReplayBuffer(dsact_image_dtype="uint8"), dsact_cnn_replay_bind_u8 /
_add_u8): the code <-> pixel mapping is exact for every code and refuses pixels off the 1/255 grid, the kwarg is refused
for vector observations, the RAM figure counts one byte per pixel, and the library exports and types the entry points.
No GPU needed."""
import ctypes as C

import numpy as np
import pytest

from dsac_v2_b200 import _lib, synth


def test_every_code_round_trips_and_matches_float64_division():
    from training.replay_buffer import DECODE_U8, decode_u8, encode_u8
    k = np.arange(256)
    x = (k / 255.0).astype(np.float32)          # what rgb / 255 environments emit: float64 divide, then cast
    assert np.array_equal(np.rint(x * np.float32(255)), k)
    assert np.array_equal(DECODE_U8.view(np.uint32), x.view(np.uint32))
    assert np.array_equal(encode_u8(x), k.astype(np.uint8))
    assert np.array_equal(decode_u8(encode_u8(x)).view(np.uint32), x.view(np.uint32))
    # the reciprocal multiply is not the same mapping; the decode table must not be built that way
    assert (k.astype(np.float32) * np.float32(1 / 255) != x).sum() > 100


@pytest.mark.parametrize("bad", [np.float32(0.5 / 255), np.float32(-1.0), np.float32(256 / 255), np.float32(np.nan),
                                 np.float32(-0.0)])
def test_off_grid_pixels_are_refused(bad):
    from training.replay_buffer import encode_u8
    img = (np.arange(12) / 255.0).astype(np.float32)
    img[7] = bad
    with pytest.raises(ValueError, match="pixel 7"):
        encode_u8(img)


def test_grey_scale_carracing_frames_are_refused():
    """The reference's gym_carracing wrapper emits gray / 128 - 1: mostly off the grid, and negative."""
    from training.replay_buffer import encode_u8
    gray = np.random.default_rng(0).integers(0, 256, size=(1, 96, 96))
    with pytest.raises(ValueError, match="not k / 255"):
        encode_u8((gray / 128.0 - 1.0).astype(np.float32))


def _kwargs(obs_dim, **over):
    return dict(obsv_dim=obs_dim, action_dim=3, buffer_max_size=200_000, additional_info={}, **over)


def test_uint8_ring_is_refused_for_vector_observations():
    from training.replay_buffer import ReplayBuffer
    with pytest.raises(ValueError, match="vector observations"):
        ReplayBuffer(**_kwargs(17, dsact_image_dtype="uint8"))
    with pytest.raises(ValueError, match="dsact_image_dtype"):
        ReplayBuffer(**_kwargs((3, 96, 96), dsact_image_dtype="float16"))
    ReplayBuffer(**_kwargs(17, dsact_image_dtype="float32"))


def test_store_refuses_an_off_grid_image_before_any_engine_is_attached():
    from training.replay_buffer import ReplayBuffer
    buf = ReplayBuffer(**_kwargs((3, 4, 5), dsact_image_dtype="uint8"))
    good = (np.random.default_rng(1).integers(0, 256, size=(3, 4, 5)) / 255.0).astype(np.float32)
    buf.store(good, {}, np.zeros(3, np.float32), 0.0, good, False, np.float32(0), {})
    assert buf.size == 1 and buf._pending[0][0].dtype == np.uint8
    bad = good.copy()
    bad[1, 2, 3] = 0.5
    with pytest.raises(ValueError, match="pixel 33 = 0.5"):
        buf.store(good, {}, np.zeros(3, np.float32), 0.0, bad, False, np.float32(0), {})
    assert buf.size == 1


def test_ram_figure_counts_one_byte_per_pixel():
    from training.replay_buffer import ReplayBuffer
    shape = synth.CNN_CONFIGS["carracing"]["obs_dim"]
    u8, f32 = ReplayBuffer(**_kwargs(shape, dsact_image_dtype="uint8")), ReplayBuffer(**_kwargs(shape))
    u8.size = f32.size = 200_000
    O = 3 * 96 * 96
    assert u8.__get_RAM__() == pytest.approx(200_000 * (2 * O + 4 * (3 + 3)) / 1e6)   # ~11.06 GB
    assert f32.__get_RAM__() == pytest.approx(200_000 * 4 * (2 * O + 3 + 3) / 1e6)    # ~44.2 GB


def test_u8_entry_points_are_exported_and_typed():
    lib = _lib.load()
    assert C.sizeof(_lib.ReplayU8) == 6 * 8 + 8
    bind = lib.dsact_cnn_replay_bind_u8
    assert bind.restype is C.c_int and bind.argtypes == [C.c_void_p, C.POINTER(_lib.ReplayU8)]
    add = lib.dsact_cnn_replay_add_u8
    assert add.restype is C.c_int and add.argtypes == [C.c_void_p] + [C.c_void_p] * 6 + [C.c_int64, C.c_int64, C.c_void_p]
    # without a handle both refuse with a message instead of touching memory
    assert bind(None, None) == -1 and lib.dsact_last_error()
    assert add(None, None, None, None, None, None, None, 0, 0, None) == -3 and lib.dsact_last_error()
