"""Shared helpers of the test-suite (oracle access, fixture loading, CPU-side recomputation of GPU inputs)."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
LAYER_FIXTURES = ['layer_hw256_h2_d64', 'layer_hw1024_h1_d64_peaky', 'layer_hw64_h2_d40', 'layer_hw576_h1_d64']


def golden(name):
    return np.load(os.path.join(GOLDEN, name + '.npz'), allow_pickle=False)


def fingerprint(t):
    """Exact, order-independent digest of a float32 tensor's bits: [sum of the bit patterns, position-weighted sum].

    Integer sums are exact in any order, so bit-equal tensors have equal fingerprints on every machine, and a change to
    any one element changes both sums. It lets a fixture pin tensors too large to store."""
    t = torch.as_tensor(t).detach().cpu().contiguous()
    assert t.dtype == torch.float32, t.dtype
    bits = t.view(torch.int32).to(torch.int64).flatten()
    weight = torch.arange(bits.numel(), dtype=torch.int64) % 251 + 1
    return [int(bits.sum()), int((bits * weight).sum())]


def oracle_layer_maps(q, k, heads, scale, steps=1):
    """Oracle rows a3+a4 (+a6 summed over `steps` identical calls) for q [B, hw, C], k [B, 77, C]: [N*H, 77, hw] fp32.

    The inputs are moved to CPU fp32 first: products of fp16/bf16 values are exact in fp32, so the oracle sees exactly
    the values the kernel reads (SURVEY.md section 8c: parity is against the fp32 oracle fed identical Q/K)."""
    from oracle import daam_oracle as O
    maps = O.port_layer_step(q.detach().float().cpu(), k.detach().float().cpu(), heads, scale)
    maps = maps.reshape(maps.shape[0], maps.shape[1], -1)
    return maps * steps if steps != 1 else maps


def rel_err(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def assert_elementwise(got, ref, rtol, atol, what=''):
    """SURVEY.md section 8c's form: |got - ref| <= atol + rtol * |ref| for EVERY element (small probabilities included),
    reporting the worst element when it fails."""
    got, ref = torch.as_tensor(got).double().cpu(), torch.as_tensor(ref).double().cpu()
    assert got.shape == ref.shape, f'{what}: shape {tuple(got.shape)} vs {tuple(ref.shape)}'
    excess = (got - ref).abs() / (atol + rtol * ref.abs())
    worst = float(excess.max())
    if not worst <= 1.0:
        i = int(excess.argmax())
        raise AssertionError(f'{what}: element {i}: got {got.flatten()[i]:.9e} ref {ref.flatten()[i]:.9e} '
                             f'= {worst:.2f} x (atol {atol:.1e} + rtol {rtol:.1e} * |ref|)')
    return worst


class HookRecorder:
    """Wraps DiffusionHeatMapHooker._enqueue to keep CPU copies of every (layer, q, k) the hook handed to the kernel, and
    replays them through the oracle (rows a3+a4+a6) -- parity on the IDENTICAL Q/K the kernel read."""

    def __init__(self, tc):
        self.calls = []
        inner = tc._enqueue

        def enqueue(layer_idx, factor, q, k, heads, scale):
            self.calls.append((layer_idx, factor, q.detach().float().cpu(), k.detach().float().cpu(), heads, scale))
            return inner(layer_idx, factor, q, k, heads, scale)

        tc._enqueue = enqueue

    def oracle_store(self, prompt_idx=0):
        from oracle import daam_oracle as O
        store = O.OracleHeatMaps()
        for layer_idx, factor, q, k, heads, scale in self.calls:
            n = q.shape[0] // 2
            pair = [prompt_idx, n + prompt_idx]
            maps = O.port_layer_step(q[pair], k[pair], heads, scale)
            for head, m in enumerate(maps):
                store.update(factor, layer_idx, head, m)
        return store
