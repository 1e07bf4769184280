"""Pins the oracle against the committed golden vectors (outputs of the verbatim reference, oracle/make_golden.py).

Bit-equality with the reference, on one CPU thread, is tests/test_oracle_vs_reference.py; here the tolerance only
absorbs summation order that depends on the CPU's instruction set and thread count."""
import numpy as np
import pytest
import torch

from daam_b200.testing.synthetic import TINY96_SPEC, TINY_SPEC, WhitespaceTokenizer, make_pipeline
from oracle import daam_oracle as O
from tests.util import LAYER_FIXTURES, golden

TOL = dict(rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize('name', LAYER_FIXTURES)
def test_layer_port_and_math(name):
    fx = golden(name)
    q, k = torch.from_numpy(fx['q']).float(), torch.from_numpy(fx['k']).float()
    heads, scale = int(fx['heads']), float(fx['scale'])
    maps = O.port_layer_step(q, k, heads, scale)
    np.testing.assert_allclose(maps.numpy(), fx['maps'], **TOL)
    # independent float64 statement of the same arithmetic (conditional sample = batch index 1)
    d = int(fx['head_dim'])
    q1 = q[1].reshape(-1, heads, d).permute(1, 0, 2).numpy()
    k1 = k[1].reshape(-1, heads, d).permute(1, 0, 2).numpy()
    m64 = O.math_layer_maps(q1, k1, scale).reshape(fx['maps'].shape)
    np.testing.assert_allclose(m64, fx['maps'], rtol=2e-5, atol=1e-7)
    # every pixel's probabilities sum to one (SURVEY.md section 4 invariant)
    np.testing.assert_allclose(fx['maps'].sum(axis=1), 1.0, rtol=1e-5)


def _finalize_keys(fx):
    keys = []
    for name in fx.files:
        if name.startswith('key_'):
            f, l, h = (int(v) for v in name.split('_')[1:])
            keys.append(((f, l, h), torch.from_numpy(fx[name])))
    return sorted(keys, key=lambda kv: (kv[0][1], kv[0][2]))


def test_finalize_fixture_exercises_the_clamp():
    fx = golden('finalize')
    under = min(O.math_upsample(v.numpy(), 64).min() for (f, _, _), v in _finalize_keys(fx) if f != 1)
    assert under < -1e-3, 'fixture should contain bicubic undershoot so that clamp(min=0) matters'


@pytest.mark.parametrize('case,kw', [
    ('global', {}), ('global_norm', {'normalize': True}), ('factors_2_4', {'factors': [2, 4]}),
    ('layer_1', {'layer_idx': 1}), ('head_1', {'head_idx': 1}), ('layer_2_head_0', {'layer_idx': 2, 'head_idx': 0}),
])
def test_finalize_port(case, kw):
    fx = golden('finalize')
    keys = _finalize_keys(fx)
    n_tok = len(WhitespaceTokenizer().tokenize(str(fx['prompt'])))
    out = O.port_global_heat_map(keys, 4096, n_tok, **kw)
    np.testing.assert_allclose(out.numpy(), fx[case], **TOL)


def test_finalize_math_layer():
    fx = golden('finalize')
    keys = [v.numpy() for _, v in _finalize_keys(fx)]
    out = O.math_global_heat_map(keys, 64, fx['global'].shape[0])
    np.testing.assert_allclose(out, fx['global'], rtol=2e-5, atol=2e-6)
    outn = O.math_global_heat_map(keys, 64, fx['global'].shape[0], normalize=True)
    np.testing.assert_allclose(outn, fx['global_norm'], rtol=2e-5, atol=2e-6)


def test_word_maps_and_expand():
    fx = golden('finalize')
    tok = WhitespaceTokenizer()
    g = torch.from_numpy(fx['global'])
    np.testing.assert_allclose(O.port_word_heat_map(g, tok, str(fx['prompt']), 'three').numpy(), fx['word_three'], **TOL)
    np.testing.assert_allclose(O.port_word_heat_map(g, tok, 'red ball and red car', 'red').numpy(),
                               fx['word_red_multi'], **TOL)
    w = torch.from_numpy(fx['word_three'])
    np.testing.assert_allclose(O.port_expand_as(w, (96, 80)).numpy(), fx['expand'], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(O.port_expand_as(w, (96, 80), absolute=True).numpy(), fx['expand_abs'], **TOL)
    np.testing.assert_array_equal(O.port_expand_as(w, (96, 80), threshold=0.4).numpy(), fx['expand_thr'])


def test_pipeline_fixture():
    fx = golden('pipeline_tiny')
    pipe = make_pipeline(TINY_SPEC, dtype=torch.float32, seed=int(fx['unet_seed']))
    with O.OracleTrace(pipe) as ot:
        pipe(str(fx['prompt']), num_inference_steps=int(fx['steps']),
             generator=torch.Generator().manual_seed(int(fx['gen_seed'])))
        assert [list(k) for k, _ in ot.heat_maps] == fx['keys'].tolist()
        assert ot.layer_names == fx['layer_names'].tolist()
        sums = np.array([float(v.double().sum()) for _, v in ot.heat_maps])
        np.testing.assert_allclose(sums, fx['key_sums'], rtol=1e-6)
        loose = dict(rtol=1e-4, atol=1e-6)   # two UNet steps of fp32 matmuls may differ across CPU ISAs
        np.testing.assert_allclose(ot.compute_global_heat_map().numpy(), fx['global'], **loose)
        np.testing.assert_allclose(ot.compute_global_heat_map(normalize=True).numpy(), fx['global_norm'], **loose)
        np.testing.assert_allclose(ot.compute_global_heat_map(factors=[2]).numpy(), fx['factors_2'], **loose)
        np.testing.assert_allclose(ot.compute_global_heat_map(layer_idx=9, head_idx=0).numpy(), fx['layer9_head0'],
                                   **loose)
    # per-key sums: every head sums to steps * hw (softmax rows sum to one)
    hw = {1: 4096, 2: 1024, 4: 256}
    for (f, _, _), s in zip(fx['keys'].tolist(), fx['key_sums']):
        assert abs(s - 2 * hw[f]) < 1e-2 * hw[f]


def test_pipeline96_fixture():
    """96x96-latent geometry (768-pixel models, daam/trace.py:32-33): keys at 96^2 / 48^2 / 24^2, x = 96."""
    fx = golden('pipeline_tiny96')
    pipe = make_pipeline(TINY96_SPEC, dtype=torch.float32, seed=int(fx['unet_seed']))
    with O.OracleTrace(pipe) as ot:
        assert ot.latent_hw == 9216
        pipe(str(fx['prompt']), num_inference_steps=int(fx['steps']),
             generator=torch.Generator().manual_seed(int(fx['gen_seed'])))
        assert [list(k) for k, _ in ot.heat_maps] == fx['keys'].tolist()
        sums = np.array([float(v.double().sum()) for _, v in ot.heat_maps])
        np.testing.assert_allclose(sums, fx['key_sums'], rtol=1e-6)
        loose = dict(rtol=1e-4, atol=1e-6)
        g = ot.compute_global_heat_map()
        assert tuple(g.shape) == (11, 96, 96)
        np.testing.assert_allclose(g.numpy(), fx['global'], **loose)
        np.testing.assert_allclose(ot.compute_global_heat_map(normalize=True).numpy(), fx['global_norm'], **loose)
        np.testing.assert_allclose(ot.compute_global_heat_map(factors=[4]).numpy(), fx['factors_4'], **loose)
        np.testing.assert_allclose(O.port_word_heat_map(g, pipe.tokenizer, str(fx['prompt']), 'ball').numpy(),
                                   fx['word_ball'], **loose)
    hw = {1: 9216, 2: 2304, 4: 576}
    for (f, _, _), s in zip(fx['keys'].tolist(), fx['key_sums']):
        assert abs(s - 2 * hw[f]) < 1e-2 * hw[f]


def test_per_key_sweep_port():
    """The reference's --all-heads sweep (daam/run/generate.py:239-255): one compute_global_heat_map per (layer, head)."""
    fx, pk = golden('finalize'), golden('perkey')
    keys = _finalize_keys(fx)
    n_tok = len(WhitespaceTokenizer().tokenize(str(fx['prompt'])))
    assert [list(k) for k, _ in keys] == pk['keys'].tolist()
    for i, (f, l, h) in enumerate(pk['keys'].tolist()):
        np.testing.assert_allclose(O.port_global_heat_map(keys, 4096, n_tok, layer_idx=l, head_idx=h).numpy(),
                                   pk['plain'][i], **TOL)
        np.testing.assert_allclose(O.port_global_heat_map(keys, 4096, n_tok, layer_idx=l, head_idx=h,
                                                          normalize=True).numpy(), pk['norm'][i], **TOL)
