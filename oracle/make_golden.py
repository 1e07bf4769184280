"""TEST INFRASTRUCTURE -- writes tests/golden/*.npz from the *verbatim* reference (run in the build container only).

    python -m oracle.make_golden

The reference (a Python package) cannot travel to the GPU box, so its outputs do: each fixture stores seeded inputs
and what ``/root/reference/daam`` itself computed from them on CPU fp32. ``tests/test_oracle_golden.py`` pins the
oracle to these on every box; the ``-m gpu`` tests compare the CUDA path with the same files.

Fixtures
  layer_*.npz        q [2, hw, H*d], k [2, 77, H*d] (fp16-representable values stored as fp16) and the maps
                     ``_unravel_attn(get_attention_scores(head_to_batch_dim(q), head_to_batch_dim(k)))`` -> [H,77,h,w]
                     exactly as daam/trace.py:272-276 + 219-244 produce them (rows a3+a4 of SURVEY.md section 8a).
  finalize.npz       hand-filled RawHeatMapCollection (peaky maps so that the clamp fires) and the outputs of
                     ``compute_global_heat_map`` for several filters / normalize (row a7), word maps (a8), expand_as (a10).
  pipeline_tiny.npz  a 2-step generation of the TINY synthetic pipeline under the reference's ``trace``: global heat
                     map, normalised map, filtered maps, per-key sums (rows a1-a9 end to end).
  pipeline_tiny96.npz the same for the 96x96-latent geometry of the 768-pixel models (latent_hw 9216, trace.py:32-33):
                     (96, 96) global maps from keys at 96^2 / 48^2 / 24^2.
  perkey.npz         the reference's --all-heads sweep (daam/run/generate.py:239-255) over finalize.npz's keys:
                     ``compute_global_heat_map(layer_idx=l, head_idx=h)`` for every key, plain and normalised.
  reference_trace.npz what tests/test_oracle_vs_reference.py compares the oracle with: the reference's per-key
                     accumulators, heat maps, saved heads and error messages of its scenarios, as exact bit fingerprints
                     (tests/util.py ``fingerprint``), single-threaded. The same generation's global maps are in
                     pipeline_tiny.npz.
  reference_experiment/ a ``GenerationExperiment.save`` dump written by the reference (experiment.py:140-167).

    python -m oracle.make_golden reference_trace     # regenerate only the named fixtures
"""
from __future__ import annotations

import os
import sys
import warnings
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from daam_b200.testing.synthetic import TINY96_SPEC, TINY_SPEC, SyntheticAttention, WhitespaceTokenizer, make_pipeline  # noqa: E402
from oracle.ref_loader import load_reference  # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')
PROMPT = 'a dog chasing a red ball on the beach'

LAYER_CASES = [
    # name, hw, heads, head_dim, logit gain (bigger = peakier softmax)
    ('layer_hw256_h2_d64', 256, 2, 64, 1.0),
    ('layer_hw1024_h1_d64_peaky', 1024, 1, 64, 4.0),
    ('layer_hw64_h2_d40', 64, 2, 40, 1.0),
    ('layer_hw576_h1_d64', 576, 1, 64, 2.0),     # 24x24: a partial 128-pixel tile (96x96-latent models)
]


def ref_layer_maps(daam, q, k, heads, dim_head):
    attn = SyntheticAttention(heads * dim_head, heads * dim_head, heads, dim_head)
    from daam.trace import UNetCrossAttentionHooker
    hk = UNetCrossAttentionHooker.__new__(UNetCrossAttentionHooker)   # _unravel_attn touches no instance state
    probs = attn.get_attention_scores(attn.head_to_batch_dim(q), attn.head_to_batch_dim(k), None)
    return hk._unravel_attn(probs)


def make_layers(daam):
    for i, (name, hw, heads, d, gain) in enumerate(LAYER_CASES):
        g = torch.Generator().manual_seed(100 + i)
        q = (torch.randn(2, hw, heads * d, generator=g) * gain).half()
        k = torch.randn(2, 77, heads * d, generator=g).half()
        maps = ref_layer_maps(daam, q.float(), k.float(), heads, d)
        np.savez_compressed(os.path.join(OUT, name + '.npz'), q=q.numpy(), k=k.numpy(), maps=maps.numpy(),
                            heads=heads, head_dim=d, scale=d ** -0.5)
        print(name, tuple(maps.shape), float(maps.sum()))


def make_finalize(daam):
    g = torch.Generator().manual_seed(7)
    tokens = 12
    coll = daam.RawHeatMapCollection()
    spec = [(1, 0, 0, 64), (2, 1, 0, 32), (2, 1, 1, 32), (4, 2, 0, 16), (4, 2, 1, 16), (4, 3, 0, 16)]
    keys = {}
    for factor, layer, head, side in spec:
        # two "steps" of peaky non-negative maps: exp of a wide gaussian makes bicubic undershoot below zero
        for _ in range(2):
            m = torch.exp(3.0 * torch.randn(tokens, side, side, generator=g))
            m = m / m.sum(0, keepdim=True)
            coll.update(factor, layer, head, m)
        keys[f'key_{factor}_{layer}_{head}'] = coll.ids_to_heatmaps[(factor, layer, head)].numpy()
    tok = WhitespaceTokenizer()
    prompt = 'one two three four five six seven eight nine'   # 9 words -> 11 rows <= 12 tokens
    fake = SimpleNamespace(all_heat_maps=coll, last_prompt=prompt, latent_hw=4096,
                           pipe=SimpleNamespace(tokenizer=tok))
    cg = daam.trace.compute_global_heat_map
    out = {
        'global': cg(fake).heat_maps,
        'global_norm': cg(fake, normalize=True).heat_maps,
        'factors_2_4': cg(fake, factors=[2, 4]).heat_maps,
        'layer_1': cg(fake, layer_idx=1).heat_maps,
        'head_1': cg(fake, head_idx=1).heat_maps,
        'layer_2_head_0': cg(fake, layer_idx=2, head_idx=0).heat_maps,
    }
    ghm = cg(fake)
    word = ghm.compute_word_heat_map('three')
    out['word_three'] = word.heatmap
    multi = daam.GlobalHeatMap(tok, 'red ball and red car', ghm.heat_maps)
    out['word_red_multi'] = multi.compute_word_heat_map('red').heatmap      # two occurrences -> rows 1 and 4
    img = SimpleNamespace(size=(96, 80))
    out['expand'] = word.expand_as(img)
    out['expand_abs'] = word.expand_as(img, absolute=True)
    out['expand_thr'] = word.expand_as(img, threshold=0.4)
    np.savez_compressed(os.path.join(OUT, 'finalize.npz'), prompt=prompt, tokens=tokens,
                        **keys, **{k: v.numpy() for k, v in out.items()})
    print('finalize', {k: tuple(v.shape) for k, v in out.items()})


def make_pipeline_fixture(daam):
    pipe = make_pipeline(TINY_SPEC, dtype=torch.float32, seed=3)
    with daam.trace(pipe) as tc:
        pipe(PROMPT, num_inference_steps=2, generator=torch.Generator().manual_seed(11))
        keys = [k for k, _ in tc.all_heat_maps]
        sums = np.array([float(v.double().sum()) for _, v in tc.all_heat_maps])
        absmax = np.array([float(v.abs().max()) for _, v in tc.all_heat_maps])
        out = {
            'global': tc.compute_global_heat_map().heat_maps.numpy(),
            'global_norm': tc.compute_global_heat_map(normalize=True).heat_maps.numpy(),
            'factors_2': tc.compute_global_heat_map(factors=[2]).heat_maps.numpy(),
            'layer9_head0': tc.compute_global_heat_map(layer_idx=9, head_idx=0).heat_maps.numpy(),
            'word_ball': tc.compute_global_heat_map().compute_word_heat_map('ball').heatmap.numpy(),
        }
        names = list(tc.layer_names)
    np.savez_compressed(os.path.join(OUT, 'pipeline_tiny.npz'), prompt=PROMPT, steps=2, unet_seed=3, gen_seed=11,
                        keys=np.array(keys), key_sums=sums, key_absmax=absmax, layer_names=np.array(names), **out)
    print('pipeline', len(keys), {k: tuple(v.shape) for k, v in out.items()})


def make_pipeline96_fixture(daam):
    pipe = make_pipeline(TINY96_SPEC, dtype=torch.float32, seed=5)
    with daam.trace(pipe) as tc:
        assert tc.latent_hw == 9216
        pipe(PROMPT, num_inference_steps=2, generator=torch.Generator().manual_seed(13))
        keys = [k for k, _ in tc.all_heat_maps]
        sums = np.array([float(v.double().sum()) for _, v in tc.all_heat_maps])
        out = {
            'global': tc.compute_global_heat_map().heat_maps.numpy(),
            'global_norm': tc.compute_global_heat_map(normalize=True).heat_maps.numpy(),
            'factors_4': tc.compute_global_heat_map(factors=[4]).heat_maps.numpy(),
            'word_ball': tc.compute_global_heat_map().compute_word_heat_map('ball').heatmap.numpy(),
        }
    np.savez_compressed(os.path.join(OUT, 'pipeline_tiny96.npz'), prompt=PROMPT, steps=2, unet_seed=5, gen_seed=13,
                        keys=np.array(keys), key_sums=sums, **out)
    print('pipeline96', len(keys), {k: tuple(v.shape) for k, v in out.items()})


def make_perkey_fixture(daam):
    """Every (layer, head) map of the all-heads sweep, from the keys stored in finalize.npz."""
    fx = np.load(os.path.join(OUT, 'finalize.npz'), allow_pickle=False)
    coll = daam.RawHeatMapCollection()
    order = []
    for name in fx.files:
        if name.startswith('key_'):
            f, l, h = (int(v) for v in name.split('_')[1:])
            coll.update(f, l, h, torch.from_numpy(fx[name]))
            order.append((f, l, h))
    fake = SimpleNamespace(all_heat_maps=coll, last_prompt=str(fx['prompt']), latent_hw=4096,
                           pipe=SimpleNamespace(tokenizer=WhitespaceTokenizer()))
    cg = daam.trace.compute_global_heat_map
    plain = np.stack([cg(fake, layer_idx=l, head_idx=h).heat_maps.numpy() for f, l, h in order])
    norm = np.stack([cg(fake, layer_idx=l, head_idx=h, normalize=True).heat_maps.numpy() for f, l, h in order])
    np.savez_compressed(os.path.join(OUT, 'perkey.npz'), keys=np.array(order), plain=plain, norm=norm)
    print('perkey', plain.shape)


def make_reference_trace_fixture(daam):
    """The scenarios of tests/test_oracle_vs_reference.py under the reference's own trace."""
    import json
    import tempfile
    from pathlib import Path
    from tests.util import fingerprint
    fp = lambda t: np.array(fingerprint(t), dtype=np.int64)
    out = {}
    # a 2-step generation of the TINY pipeline
    torch.manual_seed(0)
    pipe = make_pipeline(TINY_SPEC, dtype=torch.float32, seed=3)
    with daam.trace(pipe) as tc:
        pipe(PROMPT, num_inference_steps=2, generator=torch.Generator().manual_seed(11))
        keys = [k for k, _ in tc.all_heat_maps]
        out['keys'] = np.array(keys)
        out['key_shapes'] = np.array([tuple(v.shape) for _, v in tc.all_heat_maps])
        out['key_fp'] = np.stack([fp(v) for _, v in tc.all_heat_maps])
        maps = {
            'global': tc.compute_global_heat_map().heat_maps,
            'norm': tc.compute_global_heat_map(normalize=True).heat_maps,
            'f2': tc.compute_global_heat_map(factors=[2]).heat_maps,
            'l9h0': tc.compute_global_heat_map(layer_idx=9, head_idx=0).heat_maps,
            'word': tc.compute_global_heat_map().compute_word_heat_map('ball').heatmap,
        }
        out['names'] = np.array(list(tc.layer_names))
    for name, m in maps.items():
        out[f'{name}_shape'], out[f'{name}_fp'] = np.array(m.shape), fp(m)
    # the --all-heads sweep over every fifth key, on a second generation under the same trace settings
    with daam.trace(pipe) as tc:
        pipe(PROMPT, num_inference_steps=2, generator=torch.Generator().manual_seed(11))
        sweep = [tc.compute_global_heat_map(layer_idx=l, head_idx=h, normalize=True).heat_maps for f, l, h in keys[::5]]
    out['sweep_shape'], out['sweep_fp'] = np.array(sweep[0].shape), np.stack([fp(m) for m in sweep])
    # error messages, token merge indices, _unravel_attn
    with daam.trace(pipe) as tc:
        try:
            tc.compute_global_heat_map()
        except RuntimeError as e:
            out['err_no_maps'] = str(e)
    try:
        daam.compute_token_merge_indices(pipe.tokenizer, PROMPT, 'zebra')
    except ValueError as e:
        out['err_word'] = str(e)
    merge = {w: daam.compute_token_merge_indices(pipe.tokenizer, PROMPT, w) for w in ['dog', 'red', 'beach']}
    merge['x@3'] = daam.compute_token_merge_indices(pipe.tokenizer, PROMPT, 'x', word_idx=3)
    out['merge_indices'] = json.dumps(merge)
    probs = torch.rand(8, 256, 77, generator=torch.Generator().manual_seed(21))
    unravelled = daam.trace(pipe).module[0]._unravel_attn(probs)
    out['unravel_shape'], out['unravel_fp'] = np.array(unravelled.shape), fp(unravelled)
    # save_heads / load_heads
    gen = lambda: torch.Generator().manual_seed(2)
    pipe5, other = make_pipeline(TINY_SPEC, dtype=torch.float32, seed=5), make_pipeline(TINY_SPEC, dtype=torch.float32, seed=6)
    with tempfile.TemporaryDirectory() as tmp:
        with daam.trace(pipe5, save_heads=True, data_dir=tmp) as tc:
            pipe5(PROMPT, num_inference_steps=2, generator=gen())
            saved = tc.compute_global_heat_map().heat_maps.clone()
            out['save_layers'] = len(tc.layer_names)
        names = sorted(p.name for p in Path(tmp).iterdir())
        out['saved_names'] = np.array(names)
        out['heads_fp'] = np.stack([fp(torch.load(Path(tmp) / n)) for n in names])
        with daam.trace(other, load_heads=True, data_dir=tmp) as tc:
            latents = other(PROMPT, num_inference_steps=2, generator=gen()).latents
            loaded = tc.compute_global_heat_map().heat_maps.clone()
    for name, t in [('saved', saved), ('loaded', loaded), ('latents', latents)]:
        out[f'{name}_shape'], out[f'{name}_fp'] = np.array(t.shape), fp(t)
    # the 96x96-latent geometry
    pipe = make_pipeline(TINY96_SPEC, dtype=torch.float32, seed=5)
    with daam.trace(pipe) as tc:
        assert tc.latent_hw == 9216
        pipe(PROMPT, num_inference_steps=2, generator=torch.Generator().manual_seed(13))
        out['keys96'] = np.array([k for k, _ in tc.all_heat_maps])
        out['key96_shapes'] = np.array([tuple(v.shape) for _, v in tc.all_heat_maps])
        out['key96_fp'] = np.stack([fp(v) for _, v in tc.all_heat_maps])
        g = tc.compute_global_heat_map(normalize=True).heat_maps
    out['norm96_shape'], out['norm96_fp'] = np.array(g.shape), fp(g)
    np.savez_compressed(os.path.join(OUT, 'reference_trace.npz'), **out)
    print('reference_trace', len(keys), 'keys', len(names), 'saved heads')


def make_reference_experiment_fixture(daam):
    """A GenerationExperiment dump written by the reference, with the heat map it holds."""
    import PIL.Image
    dst = os.path.join(OUT, 'reference_experiment')
    os.makedirs(dst, exist_ok=True)
    maps = torch.rand(6, 16, 16, generator=torch.Generator().manual_seed(4))
    img = PIL.Image.new('RGB', (16, 16), (10, 20, 30))
    cwd = os.getcwd()
    os.chdir(dst)     # the dump pickles its path: keep it relative
    try:
        daam.GenerationExperiment(img, maps, 'a red ball', seed=3, id='q1', path='.').save(heat_maps=False)
    finally:
        os.chdir(cwd)
    np.save(os.path.join(dst, 'global_heat_map.npy'), maps.numpy())
    print('reference_experiment', sorted(os.listdir(os.path.join(dst, 'q1'))))


FIXTURES = {'layers': make_layers, 'finalize': make_finalize, 'pipeline_tiny': make_pipeline_fixture,
            'pipeline_tiny96': make_pipeline96_fixture, 'perkey': make_perkey_fixture,
            'reference_trace': make_reference_trace_fixture, 'reference_experiment': make_reference_experiment_fixture}


def main(names=None):
    warnings.filterwarnings('ignore', category=FutureWarning)
    os.makedirs(OUT, exist_ok=True)
    os.environ.setdefault('XDG_CACHE_HOME', '/tmp/daam_cache')
    torch.set_num_threads(1)   # fixtures must not depend on the thread count
    daam = load_reference()
    for name in names or FIXTURES:
        FIXTURES[name](daam)


if __name__ == '__main__':
    main(sys.argv[1:])
