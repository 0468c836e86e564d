"""CPU: the one-block-latency convolver's schedule (neo_b200_lowlat_layout) and configuration errors -- no device needed."""
import pytest


def layout(pkg, partitions, block=1024, frame_blocks=None, dtype="float32"):
    return pkg.LowLatencyConvolver.layout(partitions, block, frame_blocks, dtype)


def test_layout_arithmetic(pkg):
    got = layout(pkg, 1024, frame_blocks=(8, 64))
    assert got == {"frame_blocks": (8, 64), "head": (0, 16), "levels": [(16, 128), (128, 1024)]}
    got = layout(pkg, 100, block=64, frame_blocks=(2, 4, 16))
    assert got == {"frame_blocks": (2, 4, 16), "head": (0, 4), "levels": [(4, 8), (8, 32), (32, 100)]}


def test_default_schedule(pkg):
    # T_1 = 8, times 4 while the level starts inside the filter (at most 4 levels, T <= 512)
    assert layout(pkg, 1024)["frame_blocks"] == (8, 32, 128)
    assert layout(pkg, 1024)["levels"] == [(16, 64), (64, 256), (256, 1024)]
    assert layout(pkg, 1025)["frame_blocks"] == (8, 32, 128, 512)
    assert layout(pkg, 1025)["levels"][-1] == (1024, 1025)
    assert layout(pkg, 1 << 20)["frame_blocks"] == (8, 32, 128, 512)
    assert layout(pkg, 17)["frame_blocks"] == (8,)
    assert layout(pkg, 16) == {"frame_blocks": (), "head": (0, 16), "levels": []}
    assert layout(pkg, 3) == {"frame_blocks": (), "head": (0, 3), "levels": []}


def test_levels_dropped_when_the_filter_is_short(pkg):
    assert layout(pkg, 6, frame_blocks=(4,)) == {"frame_blocks": (), "head": (0, 6), "levels": []}
    assert layout(pkg, 8, frame_blocks=(4, 16)) == {"frame_blocks": (), "head": (0, 8), "levels": []}
    assert layout(pkg, 9, frame_blocks=(4, 16)) == {"frame_blocks": (4,), "head": (0, 8), "levels": [(8, 9)]}
    assert layout(pkg, 40, frame_blocks=(2, 4, 16, 64)) == {
        "frame_blocks": (2, 4, 16), "head": (0, 4), "levels": [(4, 8), (8, 32), (32, 40)]}


@pytest.mark.parametrize("frame_blocks,message", [
    ((8, 4), "frame_blocks must increase"),
    ((8, 8), "frame_blocks must increase"),
    ((6,), r"frame_blocks\[0\] must be a power of two in \[2, 512\], got 6"),
    ((4, 12), r"frame_blocks\[1\] must be a power of two"),
    ((1024,), r"power of two in \[2, 512\], got 1024"),
    ((1,), r"power of two in \[2, 512\], got 1"),
    ((2, 4, 8, 16, 32), "at most 4 levels, got 5"),
])
def test_schedule_errors(pkg, frame_blocks, message):
    with pytest.raises(RuntimeError, match=message):
        layout(pkg, 4096, frame_blocks=frame_blocks)


@pytest.mark.parametrize("block,dtype", [(96, "float32"), (1, "float32"), (0, "float32"), (16384, "float32"), (8192, "float64")])
def test_bad_block(pkg, block, dtype):
    with pytest.raises(RuntimeError, match="block size must be a power of two"):
        layout(pkg, 64, block=block, dtype=dtype)


def test_largest_blocks_accepted(pkg):
    assert layout(pkg, 7, block=8192, frame_blocks=(2,))["levels"] == [(4, 7)]
    assert layout(pkg, 7, block=4096, frame_blocks=(2,), dtype="float64")["levels"] == [(4, 7)]


def test_create_reports_configuration_errors_before_any_device_work(pkg):
    import numpy as np

    conv = pkg.LowLatencyConvolver("float32", frame_blocks=(16, 8))
    with pytest.raises(RuntimeError, match="frame_blocks must increase"):
        conv.filter(np.zeros((2, 64, 65), dtype=np.complex64))
