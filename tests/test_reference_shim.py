"""Pins the oracle to the reference's OWN code: numbers the unmodified reference sources produced on tests/tf_shim (a
torch-backed stand-in for the TensorFlow/Keras primitives), stored in tests/golden/ref_pins.{npz,json} and
tests/golden/ref_train_c1.npz, compared with oracle/*.py and with the host-side mirrors in transformertts_b200/.

tests/golden/make_reference_pins.py writes the pins, running the reference half of each test below with the same seeds.
"""
import hashlib
import importlib.util
import json
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

GOLD = Path(__file__).resolve().parent / 'golden'
sys.path.insert(0, str(GOLD))
from make_golden_ref import grad_sample_index  # noqa: E402
from make_reference_pins import FORWARD_CASES, PREDICT_SETTINGS, UPDATE_SAMPLE, sample_index  # noqa: E402
from oracle import aligner_oracle as alo  # noqa: E402
from oracle import forward_oracle as fo  # noqa: E402

META = json.loads((GOLD / 'ref_pins.json').read_text(encoding='utf-8'))
_NPZ = np.load(GOLD / 'ref_pins.npz')
VALUES, INDEX = _NPZ['values'], json.loads(str(_NPZ['index']))


@pytest.fixture(scope='module', autouse=True)
def _threads():
    torch.set_num_threads(4)
    yield


def pin(key):
    """(stored elements as a flat tensor of the reference's dtype, shape of the reference tensor)."""
    off, n, shape, dtype = INDEX[key]
    return torch.from_numpy(VALUES[off:off + n].astype(dtype)), tuple(shape)


def whole(key):
    v, shape = pin(key)
    assert v.numel() == int(np.prod(shape)), key
    return v.reshape(shape)


def _close(a, key, tol):
    """max |a - reference| over the stored elements of `key` (all of them, or its seeded sample) <= tol."""
    want, shape = pin(key)
    a = torch.as_tensor(a).double()
    assert tuple(a.shape) == shape, (tuple(a.shape), shape)
    got = a.reshape(-1)[torch.from_numpy(sample_index(key, a.numel(), want.numel()))]
    err = float((got - want.double()).abs().max()) if got.numel() else 0.0
    assert err <= tol, err
    return err


def _digest(t):
    a = np.ascontiguousarray(torch.as_tensor(t).numpy())
    return {'shape': list(a.shape), 'dtype': str(a.dtype), 'sha256': hashlib.sha256(a.tobytes()).hexdigest()}


def _json(x):
    return json.loads(json.dumps(x))


def _tf_shim():
    """tests/tf_shim/tensorflow, loaded under a private name so that `import tensorflow` elsewhere is unaffected."""
    spec = importlib.util.spec_from_file_location('tf_shim_tensorflow', Path(__file__).resolve().parent / 'tf_shim' / 'tensorflow' / '__init__.py')
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# ----------------------------------------------------------------------------------------------------------------------
# the shim itself is pinned by the reference's known answers (tests/test_loss.py of the reference, which passes on the shim)
# ----------------------------------------------------------------------------------------------------------------------
def test_reference_own_loss_test_passes_on_the_shim():
    """The reference's stop-token losses weight the Keras cross entropy by 0 on padding, 1 elsewhere and `scaling` on the stop
    index; the shim's SparseCategoricalCrossentropy with those weights and the oracle both give the known answers."""
    k = META['loss_known_answers']
    targets, logits = np.array(k['targets']), np.array(k['logits'])
    ce = _tf_shim().keras.losses.SparseCategoricalCrossentropy(from_logits=True)
    assert k['masked'] == k['scaled']['1']
    for s, want in k['scaled'].items():
        weights = (targets != 0) + (targets == k['stop_index']) * (float(s) - 1.0)
        assert abs(float(ce(targets, logits, sample_weight=weights)) - want) < 1e-7, s
        got = alo.new_scaled_crossentropy(torch.from_numpy(targets), torch.from_numpy(logits).float(), index=k['stop_index'], scaling=float(s))
        assert abs(float(got) - want) < 1e-6, s


def test_expand_docstring_example_through_reference_code():
    """model/layers.py:532-542: the reference's Expand layer (ragged-tensor construction) on its own docstring example."""
    x = torch.tensor([[[0.54710746, 0.8943467], [0.7140938, 0.97968304], [0.5347662, 0.15213418]]])
    want = x[0][[0, 1, 1, 1, 2, 2]][None]
    assert torch.equal(whole('expand_docstring'), want)
    assert torch.equal(fo.expand(x, torch.tensor([[[1.], [3.], [2.]]])), want)


# ----------------------------------------------------------------------------------------------------------------------
# ForwardTransformer: reference model code vs the oracle
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cfg_name,B,Tp,Tm,seed', FORWARD_CASES)
def test_forward_transformer_call_matches_oracle(cfg_name, B, Tp, Tm, seed):
    cfg = fo.CONFIGS[cfg_name]
    p = fo.init_params(cfg, seed=7)
    tok, dur, pit = fo.make_inputs('ragged', B, Tp, Tm, seed=seed)
    with torch.no_grad():
        got = fo.forward_transformer_call(p, cfg, tok, dur[..., None], pit[..., None])
    pre = f'forward/{cfg_name}'
    assert sorted(got['encoder_attention']) == META[pre + '/encoder_attention']
    assert sorted(got['decoder_attention']) == META[pre + '/decoder_attention']
    _close(got['mel'], pre + '/mel', 2e-5)
    _close(got['duration'], pre + '/duration', 1e-5)
    _close(got['pitch'], pre + '/pitch', 1e-5)
    assert torch.equal(got['expanded_mask'], whole(pre + '/expanded_mask'))
    for att in ('encoder_attention', 'decoder_attention'):
        for k in META[f'{pre}/{att}']:
            _close(got[att][k], f'{pre}/{att}/{k}', 1e-5)


def test_predict_with_predicted_durations_speed_and_duration_masks():
    """model/models.py:559-595: predict() with its speed regulator and per-phoneme max / min duration tables.  Durations are
    predicted (ReLU head, then * 1/speed, min/max masks, round-half-even): the integer durations must be identical."""
    cfg = fo.CONFIGS['C1']
    p = fo.init_params(cfg, seed=7)
    # a duration head that produces usable durations: positive bias on the last Dense
    p = dict(p)
    p['dur_pred.out.b'] = torch.tensor([3.2])
    tok, dur, pit = fo.make_inputs('ragged', 3, 32, 160, seed=111)
    ids = META['predict_ids']
    for i, (speed, use_max, use_min) in enumerate(PREDICT_SETTINGS):
        tok_np = tok.numpy()
        mxm = np.full(tok_np.shape, np.inf, dtype=np.float32)
        mnm = np.zeros(tok_np.shape, dtype=np.float32)
        if use_max:
            mxm[tok_np == ids['max']] = 2.0
        if use_min:
            mnm[tok_np == ids['min']] = 6.0
        with torch.no_grad():
            got = fo.forward_transformer_call(p, cfg, tok, None, None, durations_scalar=float(np.float32(1. / speed)),
                                              max_durations_mask=torch.from_numpy(mxm), min_durations_mask=torch.from_numpy(mnm))
        assert got['mel'].shape[1] > 0
        _close(got['mel'], f'predict/{i}/mel', 5e-5)
        assert torch.equal(got['expanded_mask'], whole(f'predict/{i}/expanded_mask'))


def test_train_step_of_the_reference_matches_oracle_gradients_and_adam():
    """model/models.py:464-482 run unmodified (GradientTape -> torch autograd, Keras Adam from the shim) with dropout 0:
    loss, every parameter after one optimizer step == oracle loss / gradients / Keras-form Adam update.  The reference's
    gradients (ref_train_c1.npz) and its weights after the step (ref_pins.npz) are stored at seeded element samples."""
    cfg = dict(fo.CONFIGS['C1'], dropout_rate=0.0, predictors_dropout=0.0)
    p = fo.init_params(cfg, seed=7)
    tok, dur, pit = fo.make_inputs('ragged', 3, 24, 150, seed=301)
    mel_tgt = fo.make_mel_targets(dur, 80, seed=302)
    ref = META['train_step']
    gold = np.load(GOLD / 'ref_train_c1.npz')
    assert ref['step'] == 1
    ref_out, ref_g = fo.loss_and_grads(p, cfg, tok, mel_tgt, dur, pit)
    assert abs(ref['loss'] - float(ref_out['loss'])) < 1e-5
    for k in ('mel', 'duration', 'pitch'):
        assert abs(ref['losses'][k] - float(ref_out['losses'][k])) < 1e-5
    assert sorted(k[2:] for k in gold.files if k.startswith('g:')) == sorted(ref_g)
    # gradients the reference step applied: after the first Keras-Adam step m = (1 - beta_1) * g
    gscale = max(float(g.abs().max()) for g in ref_g.values())
    for name, g in ref_g.items():
        g_ref = g.double().reshape(-1)
        idx = torch.from_numpy(grad_sample_index(name, g_ref.numel()))
        g_got = torch.from_numpy(gold['g:' + name]).double()
        assert float((g_got - g_ref[idx]).abs().max()) < 2e-5 * gscale, name
        # the applied update, where the gradient is well above fp32 noise (Adam's first step is lr * sign(g): elements
        # whose gradient is analytically zero -- the key biases -- move by +-lr on rounding noise alone, in TF as well)
        w = p[name].clone()
        m, v = torch.zeros_like(w), torch.zeros_like(w)
        fo.adam_tf_step(w, g.float(), m, v, 1, 1e-4)
        var, shape = pin('train/w:' + name)
        assert shape == tuple(w.shape), name
        sel = idx[:UPDATE_SAMPLE]
        live = g_ref[sel].abs() > 1e-4 * gscale
        if live.any():
            assert float(((w.reshape(-1)[sel] - var).double().abs() * live).max()) < 2e-7, name
            assert float(((var - p[name].reshape(-1)[sel]).abs() * live).max()) > 0.9e-4, name


# ----------------------------------------------------------------------------------------------------------------------
# Aligner (SURVEY 8f row 1): reference model code vs the oracle
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('r', [1, 2])
def test_aligner_teacher_forced_step_matches_oracle(r):
    cfg = alo.ALIGNER_CONFIGS['A-small']
    p = alo.init_aligner_params(cfg, seed=7)
    tok, mel, stop = alo.make_aligner_inputs(cfg, 3, 20, 49, seed=503)
    with torch.no_grad():
        got = alo.gta_forward(p, dict(cfg, dropout_rate=0.0, decoder_prenet_dropout=0.0), tok, mel, stop, r=r,
                              stop_scaling=cfg['stop_loss_scaling'], force_decoder_diagonal=True, force_encoder_diagonal=True)
    pre = f'aligner/r{r}'
    _close(got['mel'], pre + '/mel', 5e-5)
    _close(got['stop_prob'], pre + '/stop_prob', 5e-5)
    _close(got['linear'], pre + '/linear', 5e-5)
    for att in ('decoder_attention', 'encoder_attention'):
        for k in META[f'{pre}/{att}']:
            _close(got[att][k], f'{pre}/{att}/{k}', 1e-5)
    ref = META[pre]
    assert abs(float(got['loss']) - ref['loss']) < 2e-5
    for k in ('mel', 'stop_prob', 'diag_loss'):
        assert abs(float(got['losses'][k]) - ref['losses'][k]) < 2e-5, k


# ----------------------------------------------------------------------------------------------------------------------
# host-side mirrors vs the reference modules they mirror (bit-exact where integers / float64 host maths)
# ----------------------------------------------------------------------------------------------------------------------
def test_positional_encoding_and_masks_bitwise():
    from transformertts_b200.model import transformer_utils as our_tu
    for n, d in ((50, 128), (2000, 256), (333, 384)):
        want = META['positional_encoding'][f'{n}x{d}']
        assert _digest(our_tu.positional_encoding(n, d)) == want
        assert _digest(fo.positional_encoding(n, d)) == want
    seq = torch.tensor([[3, 7, 0, 0], [1, 0, 0, 0]], dtype=torch.int32)
    assert torch.equal(fo.create_encoder_padding_mask(seq), whole('masks/encoder_padding'))
    mel = torch.zeros(2, 5, 3)
    mel[0, :4] = 1.0
    mel[1, :2] = -2.0
    assert torch.equal(fo.create_mel_padding_mask(mel), whole('masks/mel_padding'))
    assert torch.equal(alo.create_look_ahead_mask(7), whole('masks/look_ahead_7'))


def test_scheduling_bitwise():
    from transformertts_b200.utils import scheduling as our_s
    ref = META['scheduling']
    for step, want in ref['lr']:
        assert our_s.piecewise_linear_schedule(step, ref['lr_schedule']) == want, step
    for step, want in ref['reduction']:
        assert our_s.reduction_schedule(step, ref['reduction_schedule']) == want
    # the reference's quirk: below the first breakpoint it returns the first STEP entry, not the first value
    assert our_s.reduction_schedule(5, [[10, 7], [20, 3]]) == ref['reduction_before_first_breakpoint'] == 10


def test_spectrogram_ops_and_losses():
    ref = META['ops']
    tgt, pred = whole('ops/target'), whole('ops/pred')
    assert ref['mel_lengths'] == [6, 2, 9]
    assert ref['phoneme_lengths'] == [3, 1, 5]
    assert abs(ref['masked_mae'] - float(fo.masked_mean_absolute_error(tgt, pred))) < 1e-6
    tot, vals = ref['weighted_sum']
    assert abs(vals[0] - float(fo.masked_mean_absolute_error(tgt, pred))) < 1e-6
    assert abs(vals[1] - float(fo.masked_mean_absolute_error(tgt, pred * 2))) < 1e-6
    assert abs(tot - (vals[0] * ref['coeffs'][0] + vals[1] * ref['coeffs'][1])) < 1e-6
    got = alo.new_scaled_crossentropy(whole('ops/stop_targets'), whole('ops/logits'), index=2, scaling=8.0)
    assert abs(float(got) - ref['scaled_ce']) < 1e-6


def test_tokenizer_and_metadata_readers(tmp_path):
    from transformertts_b200.data import datasets as ds
    from transformertts_b200.model.models import DEFAULT_VOCAB
    modes = {(m['add_start_end'], m['model_breathing']): m['vocab_size'] for m in META['tokenizer']['modes']}
    assert modes[(False, False)] == DEFAULT_VOCAB
    assert modes[(True, False)] == alo.ALIGNER_VOCAB
    ref = META['metadata']
    meta = tmp_path / 'metadata.csv'
    meta.write_text(ref['csv'], encoding='utf-8')
    assert _json(ds.ljspeech(meta)) == ref['ljspeech']
    got_text, got_up = ds.post_processed_reader(meta)
    assert _json([got_text, got_up]) == ref['post_processed_reader'] and len(got_up) == 20


def test_keras_weight_order_follows_the_reference_constructors():
    """model_weights.hdf5 is matched BY ORDER (transformertts_b200/model/hdf5_weights.py): the order must be the one in
    which the reference's constructors assign layers and variables (Keras: own variables first, then tracked sub-layers in
    assignment order) -- walked on the reference classes themselves through the shim's Layer tracking."""
    from transformertts_b200.model import hdf5_weights as hw
    from transformertts_b200.model.models import ForwardTransformer
    for cfg_name in ('C1', 'LJ256'):
        cfg = fo.CONFIGS[cfg_name]
        ours = ForwardTransformer(**cfg, device='cpu')
        want = [(lname, [flat for _, flat in ws]) for lname, ws in hw.keras_layer_order(ours)]
        got = META['keras_order'][cfg_name]
        assert [g[1] for g in got] == [w[1] for w in want]
        # the explicitly named layers keep their names; the two unnamed Dense layers get counter-based names in TF
        assert [g[0] for g in got if g[0][0].isupper() or '_pred' in g[0] or g[0] == 'expand'] == \
            ['Embedding', 'Encoder', 'dur_pred', 'expand', 'pitch_pred', 'Decoder']


def test_tokenizer_mirror_equals_reference_tokenizer():
    from transformertts_b200.data.text import ALL_PHONEMES, Tokenizer
    ref = META['tokenizer']
    assert list(ALL_PHONEMES) == ref['all_phonemes']
    assert len(ref['modes']) == 4
    for mode in ref['modes']:
        a = Tokenizer(add_start_end=mode['add_start_end'], model_breathing=mode['model_breathing'])
        assert a.vocab_size == mode['vocab_size']
        assert len(mode['encoded']) == 20
        for s, ids, decoded in mode['encoded']:
            assert list(a(s)) == ids
            assert a.decode(a(s)) == decoded
    alpha = ref['alphabet']
    assert list(Tokenizer(alphabet=alpha['alphabet'])(alpha['text'])) == alpha['encoded']


def test_keras_weight_order_of_the_aligner():
    from transformertts_b200.model import hdf5_weights as hw
    from transformertts_b200.model.aligner import Aligner
    cfg = alo.ALIGNER_CONFIGS['A-small']
    ours = Aligner.from_config(dict(cfg, device='cpu'), max_r=cfg['max_r'])
    want = [[flat for _, flat in ws] for _, ws in hw.keras_layer_order(ours)]
    got = META['keras_order']['aligner']
    assert [g[1] for g in got] == want      # includes DecoderPrenet's non-trainable rate variable (None) in last position
    assert [g[0] for g in got] == ['Embedding', 'Encoder', 'DecoderPrenet', 'Decoder', 'FinalProj', 'Postnet']


@pytest.mark.parametrize('r,force_long', [(4, False), (1, False), (2, True)])
def test_aligner_autoregressive_predict_matches_oracle(r, force_long):
    """Aligner.predict (models.py:271-292, encode=False) of the UNMODIFIED reference against oracle.aligner_predict: same number
    of iterations (stop decision) and the same frames.  force_long biases the stop head so the loop runs to max_length."""
    cfg = alo.ALIGNER_CONFIGS['A-small']
    p = alo.init_aligner_params(cfg, seed=7)
    if force_long:
        p = dict(p)
        p['postnet.stop.b'] = torch.tensor([6.0, 0.0, -6.0])
    tok, mel, _ = alo.make_aligner_inputs(cfg, 2, 12, 21, seed=3)
    c0 = dict(cfg, dropout_rate=0.0, decoder_prenet_dropout=0.0)
    pre = f'aligner_predict/r{r}_{int(force_long)}'
    ref = META[pre]
    o = alo.aligner_predict(p, c0, tok[0], ref['start_vec'], max_length=10, r=r, stop_prob_index=ref['stop_prob_index'])
    a, b = whole(pre + '/mel'), o['mel']
    assert a.shape == b.shape
    if force_long:
        assert a.shape[0] == (10 // r + 1) * r
    assert float((a - b).abs().max()) < 1e-5
    k = 'Decoder_LastBlock_CrossAttention'
    assert float((whole(pre + '/cross_attention') - o['decoder_attention'][k]).abs().max()) < 1e-5
