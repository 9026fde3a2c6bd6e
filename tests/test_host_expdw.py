"""CPU: shared-memory plan and eligibility of the fused expand + depthwise kernel (expdw_kernel, csrc/tc_expdw.cuh)."""
import ctypes as C
import os

import pytest

from metrabs_b200 import _lib
from metrabs_b200.backbones.efficientnet import stage_table


def _plan(h, w, cin, cexp):
    v = [C.c_int() for _ in range(4)]
    assert _lib.lib().mtb_debug_expdw_plan(h, w, cin, cexp, *[C.byref(x) for x in v]) == 0
    return tuple(x.value for x in v)  # pixels per tile, crops per tile, ring stages, smem bytes


def _mbconv_blocks(size, side):
    """(H, W, Cin, Cexp, stride) of every MBConv block with an expand conv, for a crop of side `side`."""
    stages, _ = stage_table(size, centered_stride=False)
    hw = side // 2  # stem stride 2
    out = []
    for st in stages:
        for bi in range(st['layers']):
            stride = st['stride'] if bi == 0 else 1
            cin = st['cin'] if bi == 0 else st['cout']
            hw_out = -(-hw // stride)
            if st['block'] != 'fused' and st['expand'] != 1:
                out.append((hw_out, hw_out, cin, cin * st['expand'], stride))
            hw = hw_out
    return out


@pytest.mark.skipif(not os.path.exists(_lib.LIB_PATH), reason='libmetrabs_b200.so not built')
@pytest.mark.parametrize('size', ['s', 'm', 'l'])
def test_expdw_plan_fits_shared_memory_for_every_effnetv2_mbconv_shape(size):
    """Every stride-1 MBConv shape of EfficientNetV2-S/M/L @256 either has a plan within the 227 KB opt-in limit (whole crops per
    tile, at least 3 weight stages) or keeps the two launches; only 16x16 / 8x8 maps are covered."""
    for h, w, cin, cexp, stride in _mbconv_blocks(size, 256):
        px, crops, ns, smem = _plan(h, w, cin, cexp)
        if px == 0:
            continue
        assert (h, w) in ((16, 16), (8, 8)), (h, w, cin, cexp)
        assert smem <= 227 * 1024 and ns >= 3, (h, w, cin, cexp, ns, smem)
        assert px == crops * h * w and px in (128, 256)
        a_bytes = (px // 128) * ((cin + 63) // 64) * 128 * 128
        assert a_bytes <= 128 * 1024


@pytest.mark.skipif(not os.path.exists(_lib.LIB_PATH), reason='libmetrabs_b200.so not built')
def test_expdw_covers_exactly_the_v2l_256_stage_4_to_7_shapes():
    """EfficientNetV2-L @256: the 53 stride-1 expand blocks on 16x16 (stage 4: 192 -> 768, stage 5: 192 -> 1152 and 224 -> 1344)
    and 8x8 (stage 6 and the first block of stage 7: 384 -> 2304) maps are eligible; stride-2 blocks and stage 7's 640 -> 3840
    blocks (a 160 KB resident input) are not."""
    eligible = {}
    for h, w, cin, cexp, stride in _mbconv_blocks('l', 256):
        if stride == 1 and _plan(h, w, cin, cexp)[0]:
            eligible[(h, cin, cexp)] = eligible.get((h, cin, cexp), 0) + 1
    assert eligible == {(16, 192, 768): 9, (16, 192, 1152): 1, (16, 224, 1344): 18, (8, 384, 2304): 25}
    assert sum(eligible.values()) == 53
    assert _plan(8, 8, 640, 3840) == (0, 0, 0, 0)
    assert _plan(24, 24, 224, 1344) == (0, 0, 0, 0)  # @384 maps keep the two launches
    assert _plan(12, 12, 384, 2304) == (0, 0, 0, 0)
