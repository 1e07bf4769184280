"""Tile schedule of the tcgen05 accumulate kernel: every (layer, prompt, head, 128-pixel tile) of a launch is processed
exactly once, whatever the ratio of tiles to CTAs, the partial last tiles, the number of prompts, the number of parameter
blocks a call is split into, the K-chunk mix or the operand form.

For each case:
* exactly once: softmax rows sum to 1, so after n launches into zeroed accumulators every pixel's 77-token sum is n;
  a tile dropped or processed twice moves a whole 128-pixel block by 1;
* agreement with the SIMT kernel, with the element-wise tolerances of test_parity_elementwise_gpu.py;
* determinism: one add per accumulator element per launch, so two identical launch sequences are bit-equal.

The grid is min(tiles, 2 CTAs x SMs) for 16-bit inputs and min(tiles, SMs) for fp32 (the split form), so the cases
that straddle the grid size are built from the device's SM count.
"""
import pytest
import torch

from daam_b200 import _native, ops
from tests.util import assert_elementwise

pytestmark = pytest.mark.gpu
DEV = 'cuda'
RTOL = {torch.float32: 1e-5, torch.float16: 1e-4, torch.bfloat16: 1e-4}
ATOL = {torch.float32: 1e-6, torch.float16: 1e-5, torch.bfloat16: 1e-5}       # x launches
LAUNCHES = 2
SD21 = [(256, 20, 64), (1024, 10, 64), (4096, 5, 64)]
SD15 = [(256, 8, 160), (1024, 8, 80), (4096, 8, 40)]


def _case(name, sms):
    """-> (layers [(hw, heads, head_dim)], prompts, dtype). A 128-pixel layer has one tile per head."""
    g16, g32 = 2 * sms, sms
    bf16, f16, f32 = torch.bfloat16, torch.float16, torch.float32
    return {
        'tiles_below_grid': ([(256, 5, 64)], 1, bf16),
        'tiles_grid_minus_1': ([(128, g16 - 1, 64)], 1, bf16),
        'tiles_grid_plus_1': ([(128, g16 + 1, 64)], 1, f16),
        'tiles_grid_multiple': ([(384, g16, 64)], 1, bf16),
        'split_tiles_grid_minus_1': ([(128, g32 - 1, 64)], 1, f32),
        'split_tiles_grid_plus_1': ([(128, g32 + 1, 64)], 1, f32),
        'odd_tiles_per_head_hw576': ([(576, 20, 64), (576, 3, 64)], 3, bf16),
        'hw_not_multiple_of_128': ([(144, 20, 64), (2304, 10, 64), (68, 4, 64)], 1, f16),
        'prompts_1': (SD21, 1, bf16),
        'prompts_3': (SD21, 3, bf16),
        'prompts_8': (SD21, 8, bf16),
        'layers_40_several_packs': ([(128 * (1 + i % 3) + 64 * (i % 2), 2 + i % 5, 64) for i in range(40)], 2, bf16),
        'head_dims_40_80_160': (SD15, 1, f16),
        'head_dims_40_80_160_prompts_3': (SD15, 3, bf16),
        'split_head_dims_40_80_160': (SD15, 1, f32),
        'split_fp32': ([(576, 20, 64), (2304, 10, 64), (9216, 5, 64)], 2, f32),
    }[name]


CASES = ['tiles_below_grid', 'tiles_grid_minus_1', 'tiles_grid_plus_1', 'tiles_grid_multiple',
         'split_tiles_grid_minus_1', 'split_tiles_grid_plus_1', 'odd_tiles_per_head_hw576', 'hw_not_multiple_of_128',
         'prompts_1', 'prompts_3', 'prompts_8', 'layers_40_several_packs', 'head_dims_40_80_160',
         'head_dims_40_80_160_prompts_3', 'split_head_dims_40_80_160', 'split_fp32']


def _inputs(name):
    layers, prompts, dtype = _case(name, _native.device_info()['sm_count'])
    g = torch.Generator(device=DEV).manual_seed(sum(map(ord, name)))
    qk = []
    for hw, heads, d in layers:
        q = (torch.randn(2 * prompts, hw, heads * d, generator=g, device=DEV) * 1.5).to(dtype)
        k = torch.randn(2 * prompts, 77, heads * d, generator=g, device=DEV).to(dtype)
        qk.append((q, k, heads, d))
    return qk, dtype


def _run(qk, flags, launches=LAUNCHES):
    """`launches` calls of daam_accumulate over all layers at once, into fresh zeroed accumulators."""
    accs = [ops.new_accumulator(q.shape[0] // 2, heads, q.shape[1], DEV) for q, _, heads, _ in qk]
    descs = ops.pack([ops.make_layer_desc(q, k, acc, heads, d ** -0.5) for (q, k, heads, d), acc in zip(qk, accs)])
    for _ in range(launches):
        ops.accumulate(descs, DEV, flags=flags)
    torch.cuda.synchronize()
    return accs


@pytest.mark.parametrize('name', CASES)
def test_every_tile_exactly_once(name):
    qk, _ = _inputs(name)
    for (q, _, heads, _), acc in zip(qk, _run(qk, _native.ACC_FORCE_MMA)):
        token_sums = acc.double().sum(dim=2)                    # [prompts, heads, hw]
        err = (token_sums - LAUNCHES).abs()
        worst = float(err.max())
        assert worst <= 1e-5 * LAUNCHES, \
            f'{name}: layer hw {q.shape[1]} heads {heads}: pixel sum off by {worst} at {tuple(int(i) for i in (err == err.max()).nonzero()[0])}'


@pytest.mark.parametrize('name', CASES)
def test_agrees_with_simt(name):
    qk, dtype = _inputs(name)
    mma = _run(qk, _native.ACC_FORCE_MMA | _native.ACC_EARLY_LOADS)
    simt = _run(qk, _native.ACC_FORCE_SIMT)
    for i, (a, b) in enumerate(zip(mma, simt)):
        assert_elementwise(a, b, RTOL[dtype], ATOL[dtype] * LAUNCHES, f'{name} layer {i}')


@pytest.mark.parametrize('name', CASES)
def test_deterministic(name):
    qk, _ = _inputs(name)
    first = _run(qk, _native.ACC_FORCE_MMA | _native.ACC_EARLY_LOADS, launches=3)
    second = _run(qk, _native.ACC_FORCE_MMA | _native.ACC_EARLY_LOADS, launches=3)
    for i, (a, b) in enumerate(zip(first, second)):
        assert torch.equal(a, b), f'{name} layer {i}: {int((a != b).sum())} elements differ'
