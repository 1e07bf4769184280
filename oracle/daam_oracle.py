"""TEST INFRASTRUCTURE -- CPU restatement ("oracle") of the reference's cross-attention heat-map hot path.

Nothing in the product (``daam_b200/``) imports this file. Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may use it, and only as the checker or as the timed CPU
baseline -- never as the thing shipped.

Parity status: the reference holds no tests, golden vectors or fixtures for this path (SURVEY.md section 4 / section 8c), so
the oracle is pinned the other way the task allows: against outputs of the reference itself. ``oracle/make_golden.py``
runs the *verbatim* reference (imported behind the stubs in ``oracle/ref_loader.py``) on seeded inputs and stores what it
computed as fixtures under ``tests/golden/``; ``tests/test_oracle_vs_reference.py`` runs this restatement on the same
inputs and requires bit-equality on CPU fp32.

Two layers live here:

* ``port_*`` / :class:`OracleTrace` -- an op-for-op torch port (same torch calls in the same order as the reference), used
  for bit-equality with the reference and as the timed CPU baseline ("kind": "port").
* ``math_*`` -- an independent float64 numpy statement of the same arithmetic (explicit softmax, explicit bicubic taps
  and Keys' cubic-convolution weights), used to check the port's numerics and to bound the CUDA kernels' error.

Row labels (a1..a10) are SURVEY.md section 8a; every function cites the reference lines it follows (paths relative to
``/root/reference``).
"""
from __future__ import annotations

import functools
import math
from collections import defaultdict
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Key = Tuple[int, int, int]  # (factor, layer_idx, head_idx) -- daam/heatmap.py:145


# =================================================================================================================
# port layer: same torch ops as the reference
# =================================================================================================================
def port_locate(unet, restrict=None, locate_middle_block: bool = False):
    """a1 -- daam/hook.py:95-127. Up blocks first, then down blocks, then (optionally) the mid block; blocks whose
    class name contains 'CrossAttn'; every ``attentions[*].transformer_blocks[*].attn2``; names restart per block."""
    found, names = [], []
    groups = [(b, 'up') for b in unet.up_blocks] + [(b, 'down') for b in unet.down_blocks]
    if locate_middle_block:
        groups.append((unet.mid_block, 'mid'))
    for block, tag in groups:
        if 'CrossAttn' not in type(block).__name__:
            continue
        layers = [tb.attn2 for st in block.attentions for tb in st.transformer_blocks]
        keep = [i for i in range(len(layers)) if restrict is None or i in restrict]
        found += [layers[i] for i in keep]
        names += [f'{tag}-attn-{i}' for i in keep]
    return found, names


def port_latent_hw(unet_sample_size: int, vae_scale_factor: int) -> int:
    """daam/trace.py:32-33 -- 64x64 for 512/1024-pixel models (SDXL included), else 96x96."""
    return 4096 if unet_sample_size * vae_scale_factor in (512, 1024) else 9216


def port_factor(latent_hw: int, hw: int) -> int:
    """a5 -- daam/trace.py:285."""
    return int(math.sqrt(latent_hw // hw))


def port_traced(tokens: int, factor: int, context_size: int = 77) -> bool:
    """a5 -- daam/trace.py:289 (the ``== 77`` and ``factor != 8`` guards)."""
    return tokens == context_size and factor != 8


def port_attention_probs(attn, query, key, attention_mask=None):
    """a3 -- the call at daam/trace.py:276 into diffusers 0.21.2 ``Attention.get_attention_scores``."""
    return attn.get_attention_scores(query, key, attention_mask)


def port_unravel(probs: torch.Tensor) -> torch.Tensor:
    """a4 -- daam/trace.py:219-244. ``[B*H, hw, T]`` -> ``[H', T, h, w]`` keeping the second half of the B*H axis."""
    side = int(math.sqrt(probs.size(1)))
    per_token = []
    for tok in probs.permute(2, 0, 1):                    # T views of [B*H, hw]
        tok = tok.view(tok.size(0), side, side)
        per_token.append(tok[tok.size(0) // 2:])          # "filter out unconditional" (trace.py:240)
    return torch.stack(per_token, 0).permute(1, 0, 2, 3).contiguous()


class OracleHeatMaps:
    """a6 -- daam/heatmap.py:148-172: ``defaultdict(lambda: 0.0)`` of per-key sums, in the map's own dtype."""

    def __init__(self):
        self.store: Dict[Key, torch.Tensor] = defaultdict(lambda: 0.0)

    def update(self, factor: int, layer_idx: int, head_idx: int, heat_map: torch.Tensor):
        key = (factor, layer_idx, head_idx)
        self.store[key] = self.store[key] + heat_map

    def clear(self):
        self.store.clear()

    def __iter__(self):
        return iter(self.store.items())

    def __len__(self):
        return len(self.store)


def port_global_heat_map(heat_maps: Iterable[Tuple[Key, torch.Tensor]], latent_hw: int, n_prompt_tokens: int,
                         factors=None, head_idx=None, layer_idx=None, normalize: bool = False) -> torch.Tensor:
    """a7 -- daam/trace.py:83-132: filter keys, bicubic to (x, x), clamp_(min=0), stack, mean over keys, keep the first
    ``n_prompt_tokens + 2`` rows, optional normalisation over rows 1..-2 with 1e-6."""
    factors = {0, 1, 2, 4, 8, 16, 32, 64} if factors is None else set(factors)
    x = int(np.sqrt(latent_hw))
    merged = []
    for (factor, layer, head), hm in heat_maps:
        if factor in factors and (head_idx is None or head_idx == head) and (layer_idx is None or layer_idx == layer):
            merged.append(F.interpolate(hm.unsqueeze(1), size=(x, x), mode='bicubic').clamp_(min=0))
    if not merged:
        if head_idx is not None or layer_idx is not None:
            raise RuntimeError('No heat maps found for the given parameters.')
        raise RuntimeError('No heat maps found. Did you forget to call `with trace(...)` during generation?')
    maps = torch.stack(merged, dim=0).mean(0)[:, 0]
    maps = maps[:n_prompt_tokens + 2]
    if normalize:
        maps = maps / (maps[1:-1].sum(0, keepdim=True) + 1e-6)
    return maps


def port_token_merge_indices(tokenizer, prompt: str, word: str, word_idx: Optional[int] = None, offset_idx: int = 0):
    """a8 -- daam/utils.py:73-91: rows of the word's token pieces, +1 for the SOS row."""
    strip = lambda toks: [t.replace('</w>', '') for t in toks]
    tokens = strip(tokenizer.tokenize(prompt.lower()))
    if word_idx is not None:
        return [word_idx + 1], word_idx
    word = word.lower()
    needle = strip(tokenizer.tokenize(word))
    rows: List[int] = []
    for start in range(len(tokens)):
        if tokens[start:start + len(needle)] == needle:
            rows += [start + offset_idx + j for j in range(len(needle))]
    if not rows:
        raise ValueError(f'Search word {word} not found in prompt!')
    return [r + 1 for r in rows], word_idx


def port_word_heat_map(global_maps: torch.Tensor, tokenizer, prompt: str, word: str, word_idx=None, offset_idx=0):
    """a8 -- daam/heatmap.py:121-123."""
    rows, _ = port_token_merge_indices(tokenizer, prompt, word, word_idx, offset_idx)
    return global_maps[rows].mean(0)


def port_expand_as(word_map: torch.Tensor, size: Tuple[int, int], absolute: bool = False, threshold=None):
    """a10 -- daam/heatmap.py:77-93 (``size`` is PIL's ``image.size``; the reference passes (W, H) as (H, W))."""
    im = F.interpolate(word_map[None, None].float(), size=(size[0], size[1]), mode='bicubic')
    if not absolute:
        im = (im - im.min()) / (im.max() - im.min() + 1e-8)
    if threshold:
        im = (im > threshold).float()
    return im.squeeze()


class OracleProcessor:
    """a2 -- daam/trace.py:252-304: the whole attn2 forward with explicit probabilities, plus the capture."""

    def __init__(self, module, parent: 'OracleTrace', layer_idx: int):
        self.module, self.parent, self.layer_idx = module, parent, layer_idx
        self.saved = None

    def _path(self):
        return self.parent.data_dir / f'{self.parent.gen_idx}.pt'     # daam/trace.py:246-250

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None):
        bsz, n, _ = hidden_states.shape
        attention_mask = attn.prepare_attention_mask(attention_mask, n, bsz)
        q = attn.to_q(hidden_states)
        ctx = hidden_states if encoder_hidden_states is None else encoder_hidden_states
        if encoder_hidden_states is not None and attn.norm_cross is not None:
            ctx = attn.norm_cross(ctx)
        k, v = attn.to_k(ctx), attn.to_v(ctx)
        q, k, v = attn.head_to_batch_dim(q), attn.head_to_batch_dim(k), attn.head_to_batch_dim(v)
        probs = port_attention_probs(attn, q, k, attention_mask)
        if self.parent.save_heads:                                    # daam/trace.py:279-282
            torch.save(probs, self._path())
        elif self.parent.load_heads:
            probs = torch.load(self._path())
        factor = port_factor(self.parent.latent_hw, probs.shape[1])
        self.parent.gen_idx += 1
        if port_traced(probs.shape[-1], factor):
            for head, m in enumerate(port_unravel(probs)):
                self.parent.heat_maps.update(factor, self.layer_idx, head, m)
        out = attn.batch_to_head_dim(torch.bmm(probs, v))
        return attn.to_out[1](attn.to_out[0](out))


class OracleTrace:
    """The reference's ``trace`` context manager reduced to the hot path (daam/trace.py:22-132, 150-186): hooks every
    located attn2, clears the store at ``check_inputs``, exposes ``compute_global_heat_map``."""

    def __init__(self, pipe, low_memory: bool = False, locate_middle_block: bool = False, save_heads: bool = False,
                 load_heads: bool = False, data_dir=None):
        from pathlib import Path
        self.pipe = pipe
        self.save_heads, self.load_heads = save_heads, load_heads
        self.data_dir = Path(data_dir) if data_dir is not None else None
        locate_middle_block = locate_middle_block or save_heads or load_heads     # daam/trace.py:34-35
        self.heat_maps = OracleHeatMaps()
        self.latent_hw = port_latent_hw(pipe.unet.config.sample_size, pipe.vae_scale_factor)
        self.layers, self.layer_names = port_locate(pipe.unet, {0} if low_memory else None, locate_middle_block)
        self.processors = [OracleProcessor(m, self, i) for i, m in enumerate(self.layers)]
        self.gen_idx = 0
        self.last_prompt = ''
        self._hooked = False

    def __enter__(self):
        if self._hooked:
            raise RuntimeError('Already hooked module')
        self._hooked = True
        for p in self.processors:
            p.saved = p.module.processor
            p.module.set_processor(p)
        self._check_inputs = self.pipe.check_inputs

        def check_inputs(prompt, *a, **kw):
            if not isinstance(prompt, str) and len(prompt) > 1:
                raise ValueError('Only single prompt generation is supported for heat map computation.')
            self.heat_maps.clear()
            self.last_prompt = prompt if isinstance(prompt, str) else prompt[0]
            return self._check_inputs(prompt, *a, **kw)

        self.pipe.check_inputs = check_inputs
        return self

    def __exit__(self, *exc):
        if not self._hooked:
            raise RuntimeError('Module is not hooked')
        self._hooked = False
        self.pipe.check_inputs = self._check_inputs
        for p in self.processors:
            p.module.set_processor(p.saved)

    def compute_global_heat_map(self, prompt=None, factors=None, head_idx=None, layer_idx=None, normalize=False):
        prompt = self.last_prompt if prompt is None else prompt
        n = len(self.pipe.tokenizer.tokenize(prompt))
        return port_global_heat_map(self.heat_maps, self.latent_hw, n, factors, head_idx, layer_idx, normalize)


def port_layer_step(q: torch.Tensor, k: torch.Tensor, heads: int, scale: float) -> torch.Tensor:
    """Rows a3+a4 on raw projections: ``q [B, hw, H*d]``, ``k [B, T, H*d]`` (what ``to_q``/``to_k`` emit) ->
    ``[H*(B/2), T, h, w]`` maps of the conditional half, exactly as trace.py:272-276 + 219-244 produce them."""
    b, n, c = q.shape
    d = c // heads
    split = lambda t: t.reshape(b, t.shape[1], heads, d).permute(0, 2, 1, 3).reshape(b * heads, t.shape[1], d)
    qh, kh = split(q), split(k)
    scores = torch.baddbmm(torch.empty(b * heads, n, k.shape[1], dtype=q.dtype), qh, kh.transpose(-1, -2),
                           beta=0, alpha=scale)
    return port_unravel(scores.softmax(dim=-1))


# =================================================================================================================
# math layer: independent float64 statement of the arithmetic
# =================================================================================================================
def math_layer_maps(q: np.ndarray, k: np.ndarray, scale: float) -> np.ndarray:
    """softmax_t(scale * q . k) for ``q [H, hw, d]``, ``k [H, T, d]`` -> ``[H, T, hw]`` in float64."""
    s = np.einsum('hpd,htd->hpt', q.astype(np.float64), k.astype(np.float64)) * scale
    s -= s.max(axis=-1, keepdims=True)
    e = np.exp(s)
    return np.ascontiguousarray((e / e.sum(axis=-1, keepdims=True)).transpose(0, 2, 1))


def _cubic_weights(t: np.ndarray, a: float = -0.75):
    """Keys' cubic convolution coefficients for taps at offsets -1, 0, +1, +2 (A = -0.75, torch's constant)."""
    near = lambda x: ((a + 2.0) * x - (a + 3.0)) * x * x + 1.0        # |x| <= 1
    far = lambda x: ((a * x - 5.0 * a) * x + 8.0 * a) * x - 4.0 * a    # 1 < |x| < 2
    return far(t + 1.0), near(t), near(1.0 - t), far(2.0 - t)


@functools.lru_cache(maxsize=None)
def math_bicubic_matrix(n_in: int, n_out: int) -> np.ndarray:
    """1-D bicubic interpolation as an ``[n_out, n_in]`` matrix: align_corners=False, source index
    ``(dst + 0.5) * n_in / n_out - 0.5`` (not clamped), taps clamped to the border, no antialiasing -- what
    ``F.interpolate(mode='bicubic')`` (called at daam/trace.py:116) does along each axis."""
    m = np.zeros((n_out, n_in), dtype=np.float64)
    src = (np.arange(n_out, dtype=np.float64) + 0.5) * (n_in / n_out) - 0.5
    base = np.floor(src)
    w = _cubic_weights(src - base)
    for tap in range(4):
        idx = np.clip(base.astype(np.int64) - 1 + tap, 0, n_in - 1)
        np.add.at(m, (np.arange(n_out), idx), w[tap])
    return m


def math_upsample(maps: np.ndarray, x: int) -> np.ndarray:
    """``[..., h, w]`` -> ``[..., x, x]`` separable bicubic in float64."""
    my, mx = math_bicubic_matrix(maps.shape[-2], x), math_bicubic_matrix(maps.shape[-1], x)
    return np.einsum('oh,...hw,pw->...op', my, maps.astype(np.float64), mx)


def math_global_heat_map(keys: Sequence[np.ndarray], x: int, n_rows: int, normalize: bool = False) -> np.ndarray:
    """mean over keys of clamp(bicubic(key)) -> first ``n_rows`` rows -> optional normalisation (a7) in float64."""
    acc = np.zeros((keys[0].shape[0], x, x), dtype=np.float64)
    for km in keys:
        acc += np.maximum(math_upsample(km, x), 0.0)
    out = (acc / len(keys))[:n_rows]
    if normalize:
        out = out / (out[1:-1].sum(0, keepdims=True) + 1e-6)
    return out
