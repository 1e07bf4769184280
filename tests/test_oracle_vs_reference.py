"""Pins oracle/daam_oracle.py bit for bit against the verbatim reference (castorini/daam).

What the reference computed in each scenario below is stored in tests/golden/reference_trace.npz (exact fingerprints of
its tensors, tests/util.py ``fingerprint``), tests/golden/pipeline_tiny.npz and tests/golden/reference_experiment/,
written by ``python -m oracle.make_golden reference_trace reference_experiment``. The oracle runs the same scenarios here
on one CPU thread, as the reference did, so that its fp32 sums are taken in the same order."""
import json
import shutil
import warnings

import numpy as np
import pytest
import torch

from daam_b200.testing.synthetic import TINY_SPEC, make_pipeline
from oracle import daam_oracle as O
from tests.util import GOLDEN, fingerprint, golden

warnings.filterwarnings('ignore', category=FutureWarning)

PROMPT = 'a dog chasing a red ball on the beach'


@pytest.fixture(scope='module', autouse=True)
def one_thread():
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(threads)


@pytest.fixture(scope='module')
def ref():
    return golden('reference_trace')


def assert_bit_equal(got, ref, name):
    assert tuple(got.shape) == tuple(ref[f'{name}_shape'].tolist()), name
    assert fingerprint(got) == ref[f'{name}_fp'].tolist(), name


@pytest.fixture(scope='module')
def runs(one_thread):
    """The 2-step generation the reference traced, under the oracle's trace."""
    torch.manual_seed(0)
    pipe = make_pipeline(TINY_SPEC, dtype=torch.float32, seed=3)
    with O.OracleTrace(pipe) as ot:
        pipe(PROMPT, num_inference_steps=2, generator=torch.Generator().manual_seed(11))
        ora_keys = {k: v.clone() for k, v in ot.heat_maps}
        g = ot.compute_global_heat_map()
        ora_out = {
            'global': g,
            'norm': ot.compute_global_heat_map(normalize=True),
            'f2': ot.compute_global_heat_map(factors=[2]),
            'l9h0': ot.compute_global_heat_map(layer_idx=9, head_idx=0),
            'word': O.port_word_heat_map(g, pipe.tokenizer, PROMPT, 'ball'),
            'names': list(ot.layer_names),
        }
    return pipe, ora_keys, ora_out


def test_layer_order_and_names(ref, runs):
    _, ora_keys, ora_out = runs
    assert ref['names'].tolist() == ora_out['names']
    assert len(ora_out['names']) == 15
    assert ref['keys'].tolist() == [list(k) for k in ora_keys]
    assert sorted({k[0] for k in ora_keys}) == [1, 2, 4]


def test_per_key_accumulators_bit_equal(ref, runs):
    _, ora_keys, _ = runs
    for i, (k, v) in enumerate(ora_keys.items()):
        assert tuple(v.shape) == tuple(ref['key_shapes'][i].tolist()), k
        assert fingerprint(v) == ref['key_fp'][i].tolist(), k


@pytest.mark.parametrize('name', ['global', 'norm', 'f2', 'l9h0', 'word'])
def test_finalize_bit_equal(ref, runs, name):
    _, _, ora_out = runs
    assert_bit_equal(ora_out[name], ref, name)


def test_error_messages_match(ref, runs):
    pipe = runs[0]
    with O.OracleTrace(pipe) as ot:
        with pytest.raises(RuntimeError) as e_ora:
            ot.compute_global_heat_map()
    assert str(e_ora.value) == str(ref['err_no_maps'])
    with pytest.raises(ValueError) as w_ora:
        O.port_token_merge_indices(pipe.tokenizer, PROMPT, 'zebra')
    assert str(w_ora.value) == str(ref['err_word'])


def test_unravel_and_merge_indices_match_reference(ref, runs):
    pipe = runs[0]
    probs = torch.rand(8, 256, 77, generator=torch.Generator().manual_seed(21))
    assert_bit_equal(O.port_unravel(probs), ref, 'unravel')
    want = json.loads(str(ref['merge_indices']))
    as_json = lambda v: json.loads(json.dumps(v))
    for word in ['dog', 'red', 'beach']:
        assert as_json(O.port_token_merge_indices(pipe.tokenizer, PROMPT, word)) == want[word]
    assert as_json(O.port_token_merge_indices(pipe.tokenizer, PROMPT, 'x', word_idx=3)) == want['x@3']


def test_math_layer_agrees_with_port(runs):
    """The float64 restatement agrees to fp32 rounding with the reference's maps, on key tensors bit-equal to its own."""
    _, ora_keys, _ = runs
    fx = golden('pipeline_tiny')
    keys = [v.numpy() for v in ora_keys.values()]
    n_rows = fx['global'].shape[0]
    g = O.math_global_heat_map(keys, 64, n_rows)
    np.testing.assert_allclose(fx['global'], g, rtol=2e-5, atol=2e-6)
    gn = O.math_global_heat_map(keys, 64, n_rows, normalize=True)
    np.testing.assert_allclose(fx['global_norm'], gn, rtol=2e-5, atol=2e-6)


def test_save_and_load_heads_match_reference(ref, tmp_path):
    """save_heads writes the same `{gen_idx}.pt` tensors; load_heads replays them into the same maps (trace.py:246-282)."""
    pipe = make_pipeline(TINY_SPEC, dtype=torch.float32, seed=5)
    d_ora = tmp_path / 'ora'
    gen = lambda: torch.Generator().manual_seed(2)
    d_ora.mkdir()
    with O.OracleTrace(pipe, save_heads=True, data_dir=d_ora) as ot:
        pipe(PROMPT, num_inference_steps=2, generator=gen())
        saved_ora = ot.compute_global_heat_map()
        assert len(ot.layer_names) == int(ref['save_layers']) == 16     # save/load also locate the mid block
    names = sorted(p.name for p in d_ora.iterdir())
    assert names == ref['saved_names'].tolist() and len(names) == 32
    for i, nme in enumerate(names):
        assert fingerprint(torch.load(d_ora / nme)) == ref['heads_fp'][i].tolist(), nme
    assert_bit_equal(saved_ora, ref, 'saved')
    other = make_pipeline(TINY_SPEC, dtype=torch.float32, seed=6)     # different weights: P comes from the files
    with O.OracleTrace(other, load_heads=True, data_dir=d_ora) as ot:
        out_ora = other(PROMPT, num_inference_steps=2, generator=gen()).latents
        loaded_ora = ot.compute_global_heat_map()
    assert_bit_equal(loaded_ora, ref, 'loaded')
    assert_bit_equal(out_ora, ref, 'latents')
    assert torch.equal(loaded_ora, saved_ora)     # the maps depend on the loaded probabilities only


def test_reference_experiment_dump_loads_in_daam_b200(tmp_path):
    """generation.pt written by the reference's GenerationExperiment.save (experiment.py:140-167) loads in ours, and back."""
    from daam_b200 import GenerationExperiment
    src = tmp_path / 'q1'
    shutil.copytree(f'{GOLDEN}/reference_experiment/q1', src)
    maps = torch.from_numpy(np.load(f'{GOLDEN}/reference_experiment/global_heat_map.npy'))
    ours = GenerationExperiment.load(src)
    assert ours.prompt == 'a red ball' and ours.seed == 3 and torch.equal(ours.global_heat_map, maps)
    assert ours.image.size == (16, 16)
    ours.id = '.'
    ours.save(str(tmp_path / 'again'))
    # same folder layout both ways (the reference's own `load` calls torch.load without weights_only=False and therefore
    # cannot read ANY pickled experiment under torch >= 2.6, its own included, so the reverse direction is checked by name)
    listing = lambda root: sorted(str(p.relative_to(root)) for p in root.rglob('*') if p.is_file())
    assert listing(tmp_path / 'again') == listing(src)


def test_latent96_geometry_bit_equal(ref):
    """768-pixel models (latent_hw 9216, daam/trace.py:32-33): reference and oracle bit-equal on the 96-latent tree,
    including the full-size 96 x 96 = 9216-position layer."""
    from daam_b200.testing.synthetic import TINY96_SPEC
    pipe = make_pipeline(TINY96_SPEC, dtype=torch.float32, seed=5)
    with O.OracleTrace(pipe) as ot:
        pipe(PROMPT, num_inference_steps=2, generator=torch.Generator().manual_seed(13))
        ora_keys = {k: v.clone() for k, v in ot.heat_maps}
        ora_g = ot.compute_global_heat_map(normalize=True)
    assert ref['keys96'].tolist() == [list(k) for k in ora_keys]
    assert {v.shape[-1] for v in ora_keys.values()} == {96, 48, 24}
    for i, (k, v) in enumerate(ora_keys.items()):
        assert tuple(v.shape) == tuple(ref['key96_shapes'][i].tolist()), k
        assert fingerprint(v) == ref['key96_fp'][i].tolist(), k
    assert tuple(ora_g.shape) == (11, 96, 96)
    assert_bit_equal(ora_g, ref, 'norm96')


def test_per_key_sweep_bit_equal(ref, runs):
    """The --all-heads sweep (daam/run/generate.py:239-255): compute_global_heat_map(layer_idx, head_idx) per key."""
    _, ora_keys, ora_out = runs
    n_rows = ora_out['global'].shape[0]
    for i, (f, l, h) in enumerate(list(ora_keys)[::5]):
        got = O.port_global_heat_map(list(ora_keys.items()), 4096, n_rows - 2, layer_idx=l, head_idx=h, normalize=True)
        assert tuple(got.shape) == tuple(ref['sweep_shape'].tolist())
        assert fingerprint(got) == ref['sweep_fp'][i].tolist(), (f, l, h)
