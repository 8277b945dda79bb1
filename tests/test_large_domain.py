"""The geometry contract of c2w_create (include/c2w_b200.h): a level's width is a power of two <= 128 whose rows tile
into 128-pixel row blocks, or a multiple of 128.  c2w_create checks the geometry before it looks for a device, so
on a machine without one an accepted geometry fails with "no CUDA device" and a refused one with the rule."""
import ctypes

import pytest

from climate2weather_b200 import _lib

SDA = (128, 128, 256, 384, 512)


def _lib_or_skip():
    try:
        return _lib.load()
    except Exception as e:  # the library is not built here
        pytest.skip(f"libc2w_b200 not loadable: {e}")


def _create(lib, H, W, channels=SDA):
    cfg = _lib.Config()
    cfg.frame_channels, cfg.window, cfg.height, cfg.width = 4, 13, H, W
    cfg.embedding_dim, cfg.noise_features = 512, 32
    cfg.n_levels = len(channels)
    for i, c in enumerate(channels):
        cfg.hidden_channels[i], cfg.hidden_blocks[i] = c, 3
    cfg.attention_mask = 1 << (len(channels) - 1)
    h = ctypes.c_void_p()
    rc = lib.c2w_create(ctypes.byref(cfg), ctypes.byref(h))
    msg = lib.c2w_last_error()
    msg = msg.decode() if isinstance(msg, bytes) else str(msg)
    if rc == 0:
        lib.c2w_destroy(h)
    return rc, msg


@pytest.mark.parametrize("H,W", [(128, 128), (256, 256), (128, 256), (256, 128), (512, 512), (64, 512), (16, 1024)])
def test_accepted_geometries(H, W):
    lib = _lib_or_skip()
    rc, msg = _create(lib, H, W)
    assert rc == 0 or "no CUDA device" in msg, msg


@pytest.mark.parametrize("H,W,level,bad", [(96, 96, 0, "96x96"), (160, 160, 0, "160x160"), (64, 192, 0, "64x192"),
                                           (128, 384, 1, "64x192"), (256, 320, 0, "256x320")])
def test_refused_geometries_name_level_and_rule(H, W, level, bad):
    lib = _lib_or_skip()
    rc, msg = _create(lib, H, W)
    assert rc != 0
    assert f"level {level}: {bad}" in msg, msg
    assert "power of two in [8,128]" in msg and "multiple of 128" in msg, msg


def test_guidance_geometry_refused_up_front():
    """Patches the UNet runs but the guidance kernels cannot tile are refused on the host with the reason."""
    from climate2weather_b200 import score
    assert score.guidance_tile(128, 128) == 16 and score.guidance_tile(256, 256) == 16
    assert score.guidance_tile(64, 512) == 16 and score.guidance_tile(512, 512) == 16
    with pytest.raises(NotImplementedError, match="16 x 1024"):
        score.guidance_tile(16, 1024)
    assert score.point_strip_rows(256, 256) == 8 and score.point_strip_rows(16, 2048) == 1
    with pytest.raises(NotImplementedError, match="4096 pixels"):
        score.point_strip_rows(16, 4096)
