"""GPU: the fused MBConv front half (expdw_kernel, csrc/tc_expdw.cuh: 1x1 expand + SiLU -> depthwise 3x3 + SiLU -> SE squeeze
in ONE launch, the expanded tensor never leaves the SM) against

* the two launches it replaces (tc_conv_kernel + dw3x3s1_tma_kernel with SE pooling) on identical inputs: same MMA order,
  roundings, FMA chains and sum orders, so the depthwise output AND the pooled means are bit-equal;
* plain ``torch.nn.functional.conv2d`` arithmetic (oracle/port_ops.py restates the reference layers,
  metrabs_pytorch/backbones/efficientnet.py:110-173 of the reference) with the expanded activation rounded to bf16 between the
  two convs (what the unfused path stores): 1e-2 on ||.||inf/||ref||inf (a layout / pipeline bug gives O(1) errors);
* a whole forward with MTB_EXPDW=0 in a second process (the switch is read once per process): bit-identical."""
import os
import subprocess
import sys

import pytest
import torch

from oracle import port, port_ops

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def H():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    from tests import helpers
    return helpers


def _engine(H, name, side):
    pcfg = port.PathConfig(proc_side=side)
    spec = port.effnet_spec(name)
    sd = port.make_effnet_state_dict(spec, pcfg, 8, seed=0, calib_batch=1)
    return H.device_model(name, pcfg, 8, sd, precision='bf16').engine(), sd, spec


def _check_pair(eng, sd, spec, names, i, x, with_reference=True):
    out, pooled = eng.debug_run_expdw(i, x, fused=True)
    out2, pooled2 = eng.debug_run_expdw(i, x, fused=False)
    assert torch.equal(out, out2), (names[i], float((out - out2).abs().max()))
    assert torch.equal(pooled, pooled2), (names[i], float((pooled - pooled2).abs().max()))
    if with_reference:
        mid = port_ops.conv_layer_reference(sd, spec, names[i], x, precision='bf16', dtype=torch.float32).bfloat16().float()
        ref = port_ops.conv_layer_reference(sd, spec, names[i + 1], mid, precision='bf16', dtype=torch.float32)
        err = port.relative_error(out.cpu(), ref.cpu())
        perr = port.relative_error(pooled.cpu(), ref.mean(dim=(1, 2)).cpu())
        print(f'{names[i]} {tuple(x.shape)}: vs conv2d {err:.2e}, means {perr:.2e}')
        assert err < 1e-2 and perr < 1e-2


@pytest.mark.parametrize('name,side,batch', [('efficientnetv2-s', 256, 3), ('efficientnetv2-m', 256, 5), ('efficientnetv2-l', 256, 3),
                                             ('efficientnetv2-l', 128, 5),   # stages 4-5 on 8x8 maps with Cin 192 / 224
                                             ('efficientnetv2-l', 256, 5)])  # odd crop counts: the last 8x8 tile holds half a tile
def test_expdw_bit_equal_to_two_launches_and_matches_conv2d(H, name, side, batch):
    eng, sd, spec = _engine(H, name, side)
    names = eng.op_names()
    g = torch.Generator().manual_seed(7)
    seen = set()
    for i in range(len(names) - 1):
        if not eng.op_is_expdw(i):
            continue
        io = eng.op_io(i)
        key = (io['in_shape'], io['out_shape'])
        if key in seen:
            continue
        seen.add(key)
        x = torch.randn((batch,) + io['in_shape'], generator=g).bfloat16().float().cuda()
        _check_pair(eng, sd, spec, names, i, x)
    assert seen, f'{name}@{side}: no fused expand + depthwise pair'


@pytest.mark.parametrize('batch', [64, 256])
def test_expdw_bit_equal_on_multi_wave_batches(H, batch):
    """The two V2-L@256 stage-5 / stage-6 shapes at sizes where every CTA walks several tiles of its job range."""
    eng, sd, spec = _engine(H, 'efficientnetv2-l', 256)
    names = eng.op_names()
    g = torch.Generator().manual_seed(11)
    done = set()
    for i in range(len(names) - 1):
        if not eng.op_is_expdw(i):
            continue
        io = eng.op_io(i)
        if io['in_shape'] not in ((16, 16, 224), (8, 8, 384)) or io['in_shape'] in done:
            continue
        done.add(io['in_shape'])
        x = torch.randn((batch,) + io['in_shape'], generator=g).bfloat16().float().cuda()
        _check_pair(eng, sd, spec, names, i, x, with_reference=False)
    assert len(done) == 2


_DUMP = r'''
import sys, torch
sys.path.insert(0, %r)
from oracle import port
from tests import helpers
side, out = int(sys.argv[1]), sys.argv[2]
pcfg = port.PathConfig(proc_side=side)
sd = port.make_effnet_state_dict(port.effnet_spec('efficientnetv2-l'), pcfg, 8, seed=0, calib_batch=1)
eng = helpers.device_model('efficientnetv2-l', pcfg, 8, sd, precision='bf16').engine()
crops, _ = port.synthetic_inputs(5, side, seed=1)
n = sum(eng.op_is_expdw(i) for i in range(len(eng.op_names())))
torch.save((eng.backbone(crops.cuda()).float().cpu(), n), out)
''' % ROOT


def test_whole_forward_bit_identical_with_and_without_fusion(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    outs = {}
    for v in ('1', '0'):
        path = str(tmp_path / f'feat_{v}.pt')
        subprocess.run([sys.executable, '-c', _DUMP, '256', path], check=True, env=dict(os.environ, MTB_EXPDW=v), cwd=ROOT)
        outs[v] = torch.load(path)
    assert outs['1'][1] == 53 and outs['0'][1] == 0
    assert torch.equal(outs['1'][0], outs['0'][0]), float((outs['1'][0] - outs['0'][0]).abs().max())
