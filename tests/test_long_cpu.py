"""Long-utterance attention: saturation radius of the bias table and the T-based kernel selection (no GPU needed)."""
import pytest
import torch

from unispeech_b200 import build
from unispeech_b200.engine import ATTN_MAX_FRAMES, attn_kernels, bias_radius, relative_positions_bucket_lut


@pytest.mark.parametrize("T", [3073, 5000, 16384])
def test_radius_of_released_bucketing(T):
    lut = relative_positions_bucket_lut(T, 320, 800)
    R = bias_radius(lut, 320)
    assert R == 778
    d = torch.arange(-(T - 1), T)
    # constant beyond R on each side (the last bucket), and R is the smallest such radius
    assert (lut[d >= R] == 319).all() and (lut[d <= -R] == 159).all()
    assert lut[T - 1 + R - 1] != 319 or lut[T - 1 - (R - 1)] != 159


@pytest.mark.parametrize("T,max_distance", [(100, 800), (1000, 1100), (3000, 3200), (5000, 8000)])
def test_radius_unsaturated_is_whole_table(T, max_distance):
    # max_distance beyond T: no delta of the utterance reaches the last bucket (which the truncated log branch reaches a
    # few percent short of max_distance, e.g. at 778 for 800), so the whole table is used
    assert bias_radius(relative_positions_bucket_lut(T, 320, max_distance), 320) == T - 1


def test_radius_other_bucketing():
    T = 4000
    lut = relative_positions_bucket_lut(T, 64, 300)
    R = bias_radius(lut, 64)
    assert R < T - 1
    d = torch.arange(-(T - 1), T)
    assert (lut[d >= R] == 63).all() and (lut[d <= -R] == 31).all()


def test_attention_kernel_selection():
    build.build()
    from unispeech_b200 import ops
    assert ops.attn_fwd_max_frames(True) == 3072
    assert ops.attn_fwd_max_frames(False) == 16384
    for T in list(range(1, 300, 7)) + [1499, 2047, 2048, 2049, 3071, 3072, 3073, 4095, 4096, 4097, 5000, 8192, 16383, 16384]:
        for bias in (True, False):
            fwd, bwd = attn_kernels(T, bias)
            assert fwd == ("attn_fwd" if T <= (3072 if bias else 16384) else "attn_fwd_long"), (T, bias)
            assert bwd == ("attn_bwd_fused" if T <= 2048 else "attn_bwd" if T <= 4096 else "attn_bwd_long"), (T, bias)
    with pytest.raises(ValueError):
        attn_kernels(ATTN_MAX_FRAMES + 1, True)
