"""What tests/test_reference_shim.py compares the oracle and the host-side mirrors against, produced by the REFERENCE'S OWN
CODE (the unmodified as-ideas/TransformerTTS sources executed on tests/tf_shim):

    TTS_REFERENCE=<checkout of as-ideas/TransformerTTS> python tests/golden/make_reference_pins.py

Each section below is the reference half of one test, with the test's seeds and inputs.  Files written:

  ref_pins.npz   the arrays, end to end in one float32 vector 'values' (exact for everything stored), located by 'index'
                 (JSON: key -> [offset, count, shape, dtype]); a tensor of more than PIN_SAMPLE elements is stored as the
                 PIN_SAMPLE elements at sample_index(key) of its flattened form
  ref_pins.json  everything else: known answers, losses, schedules, attention-map names, tokenizations, metadata readers,
                 the Keras layer / weight order, and SHA-256 digests of tensors the tests compare bit for bit

The training-step gradients of the same test live in ref_train_c1.npz (make_golden_ref.py, identical step).
"""
import hashlib
import importlib.util
import json
import sys
import tempfile
import unittest
import zlib
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / 'tests'))
sys.path.insert(0, str(ROOT / 'tests' / 'golden'))
from make_golden_ref import grad_sample_index  # noqa: E402
from oracle import aligner_oracle as alo  # noqa: E402
from oracle import forward_oracle as fo  # noqa: E402

OUT = Path(__file__).resolve().parent
PIN_SAMPLE = 512
ATT_SAMPLE = 128
UPDATE_SAMPLE = 128
FORWARD_CASES = [('C1', 3, 40, 200, 101), ('LJ256', 2, 48, 300, 201), ('LJ256-dense', 2, 32, 180, 202), ('REF384', 2, 24, 150, 203)]
PREDICT_SETTINGS = [(1.0, False, False), (0.8, True, False), (1.25, False, True)]
METADATA_CSV = ('LJ001-0001.wav|Printing, in the only sense|printing in the only sense\nLJ001-0002|really?|really?\n'
                'LJ001-0003|stop!|stop!\n')


def sample_index(key: str, numel: int, k: int = PIN_SAMPLE) -> np.ndarray:
    """Seeded element sample of a flattened tensor (shared with the tests); all elements when there are at most k."""
    if numel <= k:
        return np.arange(numel)
    return np.sort(np.random.default_rng(zlib.crc32(key.encode())).choice(numel, k, replace=False))


def digest(t) -> dict:
    a = np.ascontiguousarray(torch.as_tensor(t).numpy())
    return {'shape': list(a.shape), 'dtype': str(a.dtype), 'sha256': hashlib.sha256(a.tobytes()).hexdigest()}


class Pins:
    def __init__(self):
        self.values, self.index, self.meta, self.n = [], {}, {}, 0

    def put(self, key, t, k=1 << 30, shape=None):
        a = np.asarray(torch.as_tensor(t).detach().numpy())
        v = a.reshape(-1)[sample_index(key, a.size, k)]
        assert np.array_equal(v.astype(np.float32).astype(v.dtype), v), key
        self.index[key] = [self.n, int(v.size), list(a.shape if shape is None else shape), str(a.dtype)]
        self.values.append(v.astype(np.float32))
        self.n += v.size

    def put_dict(self, key, d, k):
        self.meta[key] = sorted(d)
        for name, t in d.items():
            self.put(f'{key}/{name}', t, k)


def main():
    import ref_shim
    ref_shim.activate()
    import tensorflow as tf  # the shim
    torch.set_num_threads(4)
    pins = Pins()

    # the known answers of the reference's tests/test_loss.py, after running that file unmodified on the shim
    spec = importlib.util.spec_from_file_location('ref_test_loss', ref_shim.REFERENCE / 'tests' / 'test_loss.py')
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    res = unittest.TextTestRunner(verbosity=0).run(unittest.defaultTestLoader.loadTestsFromModule(mod))
    assert res.testsRun >= 1 and res.wasSuccessful(), res.failures + res.errors
    from utils.losses import masked_crossentropy, new_scaled_crossentropy
    targets = np.array([[0, 1, 2]])
    logits = np.array([[[.3, .2, .1], [.3, .2, .1], [.3, .2, .1]]])
    pins.meta['loss_known_answers'] = {
        'targets': targets.tolist(), 'logits': logits.tolist(), 'stop_index': 2,
        'scaled': {str(s): float(new_scaled_crossentropy(index=2, scaling=s)(targets, logits)) for s in (5, 1)},
        'masked': float(masked_crossentropy(targets, logits))}

    # Expand on its docstring example
    from model.layers import Expand
    x = torch.tensor([[[0.54710746, 0.8943467], [0.7140938, 0.97968304], [0.5347662, 0.15213418]]])
    pins.put('expand_docstring', Expand(model_dim=2)(x, torch.tensor([[[1.], [3.], [2.]]])))

    # ForwardTransformer.call
    for cfg_name, B, Tp, Tm, seed in FORWARD_CASES:
        cfg = fo.CONFIGS[cfg_name]
        p = fo.init_params(cfg, seed=7)
        tok, dur, pit = fo.make_inputs('ragged', B, Tp, Tm, seed=seed)
        durf, pitf = dur[..., None].float(), pit[..., None]
        model = ref_shim.reference_forward_transformer(cfg, p, (tok, durf, pitf))
        with torch.no_grad():
            ref = model.call(tok, target_durations=durf, target_pitch=pitf, training=False)
        pre = f'forward/{cfg_name}'
        pins.put(pre + '/mel', ref['mel'], PIN_SAMPLE)
        pins.put(pre + '/duration', ref['duration'])
        pins.put(pre + '/pitch', ref['pitch'])
        pins.put(pre + '/expanded_mask', ref['expanded_mask'])
        pins.put_dict(pre + '/encoder_attention', ref['encoder_attention'], ATT_SAMPLE)
        pins.put_dict(pre + '/decoder_attention', ref['decoder_attention'], ATT_SAMPLE)

    # ForwardTransformer.predict with the speed regulator and per-phoneme max / min durations
    cfg = fo.CONFIGS['C1']
    p = dict(fo.init_params(cfg, seed=7))
    p['dur_pred.out.b'] = torch.tensor([3.2])
    tok, dur, pit = fo.make_inputs('ragged', 3, 32, 160, seed=111)
    model = ref_shim.reference_forward_transformer(cfg, p, (tok, dur[..., None].float(), pit[..., None]))
    tokenizer = model.text_pipeline.tokenizer
    sym_a, sym_b = tokenizer.idx_to_token[int(tok[0, 0])], tokenizer.idx_to_token[int(tok[0, 1])]
    pins.meta['predict_ids'] = {'max': int(tokenizer(sym_a)[0]), 'min': int(tokenizer(sym_b)[0])}
    for i, (speed, use_max, use_min) in enumerate(PREDICT_SETTINGS):
        with torch.no_grad():
            ref = model.predict(tok, encode=False, speed_regulator=speed, phoneme_max_duration={sym_a: 2.0} if use_max else None,
                                phoneme_min_duration={sym_b: 6.0} if use_min else None)
        pins.put(f'predict/{i}/mel', ref['mel'], PIN_SAMPLE)
        pins.put(f'predict/{i}/expanded_mask', ref['expanded_mask'])

    # one training step (dropout 0): losses here, gradients in ref_train_c1.npz, weights after the Adam step at a sample
    cfg = dict(fo.CONFIGS['C1'], dropout_rate=0.0, predictors_dropout=0.0)
    p = fo.init_params(cfg, seed=7)
    tok, dur, pit = fo.make_inputs('ragged', 3, 24, 150, seed=301)
    mel_tgt = fo.make_mel_targets(dur, 80, seed=302)
    model = ref_shim.reference_forward_transformer(cfg, p, (tok, dur[..., None].float(), pit[..., None]))
    model._compile(optimizer=tf.keras.optimizers.Adam(1e-4, beta_1=0.9, beta_2=0.98, epsilon=1e-9))
    out = model.train_step(tok, mel_tgt, dur, pit)
    pins.meta['train_step'] = {'step': int(model.step), 'loss': float(out['loss']),
                               'losses': {k: float(out['losses'][k]) for k in ('mel', 'duration', 'pitch')}}
    for name, var in ref_shim.ft_named_parameters(model, cfg).items():
        w = var.detach().reshape(-1).numpy()
        pins.put('train/w:' + name, w[grad_sample_index(name, w.size)[:UPDATE_SAMPLE]], shape=var.shape)

    # Aligner teacher-forced validation step
    acfg = alo.ALIGNER_CONFIGS['A-small']
    ap = alo.init_aligner_params(acfg, seed=7)
    c0 = dict(acfg, dropout_rate=0.0, decoder_prenet_dropout=0.0)
    tok, mel, stop = alo.make_aligner_inputs(acfg, 3, 20, 49, seed=503)
    for r in (1, 2):
        model = ref_shim.reference_aligner(c0, ap, (tok, mel[:, :-1]))
        model._compile(stop_scaling=acfg['stop_loss_scaling'], optimizer=tf.keras.optimizers.Adam(1e-4, beta_1=0.9, beta_2=0.98, epsilon=1e-9))
        model.set_constants(reduction_factor=r, force_decoder_diagonal=True, force_encoder_diagonal=True)
        with torch.no_grad():
            ref = model.val_step(tok, mel, stop)
        pre = f'aligner/r{r}'
        for k in ('mel', 'stop_prob', 'linear'):
            pins.put(f'{pre}/{k}', ref[k], PIN_SAMPLE)
        pins.put_dict(pre + '/decoder_attention', ref['decoder_attention'], ATT_SAMPLE)
        pins.put_dict(pre + '/encoder_attention', ref['encoder_attention'], ATT_SAMPLE)
        pins.meta[pre] = {'loss': float(ref['loss']), 'losses': {k: float(ref['losses'][k]) for k in ('mel', 'stop_prob', 'diag_loss')}}

    # positional encoding and masks
    from model import transformer_utils as ref_tu
    pins.meta['positional_encoding'] = {f'{n}x{d}': digest(ref_tu.positional_encoding(n, d)) for n, d in ((50, 128), (2000, 256), (333, 384))}
    seq = torch.tensor([[3, 7, 0, 0], [1, 0, 0, 0]], dtype=torch.int32)
    mel = torch.zeros(2, 5, 3)
    mel[0, :4] = 1.0
    mel[1, :2] = -2.0
    pins.put('masks/encoder_padding', ref_tu.create_encoder_padding_mask(seq))
    pins.put('masks/mel_padding', ref_tu.create_mel_padding_mask(mel))
    pins.put('masks/look_ahead_7', ref_tu.create_look_ahead_mask(7))

    # schedules
    from utils import scheduling as ref_s
    lr_sched = [[0, 1.0e-4], [40000, 1.0e-4], [41000, 5.0e-5], [100000, 1.0e-5]]
    red = [[0, 10], [80000, 5], [150000, 3], [250000, 1]]
    pins.meta['scheduling'] = {
        'lr_schedule': lr_sched, 'reduction_schedule': red,
        'lr': [[s, float(ref_s.piecewise_linear_schedule(s, lr_sched))] for s in (0, 1, 39999, 40000, 40500, 40999, 41000, 77777, 100000, 250000)],
        'reduction': [[s, int(ref_s.reduction_schedule(s, red))] for s in (0, 79999, 80000, 200000, 999999)],
        'reduction_before_first_breakpoint': int(ref_s.reduction_schedule(5, [[10, 7], [20, 3]]))}

    # spectrogram ops and losses on seeded inputs
    from utils import losses as ref_l
    from utils import spectrogram_ops as ref_ops
    g = torch.Generator().manual_seed(11)
    mel = torch.randn(3, 9, 4, generator=g)
    mel[0, 6:] = 0
    mel[1, 2:] = 0
    ph = torch.tensor([[4, 5, 6, 0, 0], [9, 0, 0, 0, 0], [1, 2, 3, 4, 5]], dtype=torch.int32)
    tgt, pred = torch.randn(2, 7, 5, generator=g), torch.randn(2, 7, 5, generator=g)
    logits = torch.randn(2, 6, 3, generator=g)
    targets = torch.tensor([[1, 1, 1, 2, 0, 0], [1, 2, 0, 0, 0, 0]])
    tot, vals = ref_l.weighted_sum_losses((tgt, tgt), (pred, pred * 2), [ref_l.masked_mean_absolute_error] * 2, [1., 3.])
    for k, v in (('mel', mel), ('phonemes', ph), ('target', tgt), ('pred', pred), ('logits', logits), ('stop_targets', targets)):
        pins.put('ops/' + k, v)
    pins.meta['ops'] = {'mel_lengths': ref_ops.mel_lengths(mel).tolist(), 'phoneme_lengths': ref_ops.phoneme_lengths(ph).tolist(),
                        'masked_mae': float(ref_l.masked_mean_absolute_error(tgt, pred)),
                        'weighted_sum': [float(tot), [float(v) for v in vals]], 'coeffs': [1., 3.],
                        'scaled_ce': float(ref_l.new_scaled_crossentropy(index=2, scaling=8.0)(targets, logits))}

    # tokenizer vocabularies and metadata readers
    from data import metadata_readers as ref_mr
    from data.text.symbols import all_phonemes
    from data.text.tokenizer import Tokenizer
    with tempfile.TemporaryDirectory() as d:
        meta = Path(d) / 'metadata.csv'
        meta.write_text(METADATA_CSV, encoding='utf-8')
        pins.meta['metadata'] = {'csv': METADATA_CSV, 'ljspeech': ref_mr.ljspeech(str(meta)),
                                 'post_processed_reader': list(ref_mr.post_processed_reader(str(meta)))}
    rng = np.random.default_rng(0)
    tok_pins = {'all_phonemes': list(all_phonemes), 'modes': []}
    for se, br in ((False, False), (True, False), (False, True), (True, True)):
        t = Tokenizer(add_start_end=se, model_breathing=br)
        strings = [''.join(rng.choice(all_phonemes, size=int(rng.integers(1, 40)))) for _ in range(20)]
        tok_pins['modes'].append({'add_start_end': se, 'model_breathing': br, 'vocab_size': t.vocab_size,
                                  'encoded': [[s, list(map(int, t(s))), t.decode(t(s))] for s in strings]})
    tok_pins['alphabet'] = {'alphabet': 'abc xyz', 'text': 'a cab', 'encoded': list(map(int, Tokenizer(alphabet='abc xyz')('a cab')))}
    pins.meta['tokenizer'] = tok_pins

    # Keras layer / weight order (what model_weights.hdf5 is matched by)
    order = {}
    for cfg_name in ('C1', 'LJ256'):
        cfg = fo.CONFIGS[cfg_name]
        p = fo.init_params(cfg, seed=7)
        tok, dur, pit = fo.make_inputs('ragged', 2, 16, 60, seed=5)
        ref = ref_shim.reference_forward_transformer(cfg, p, (tok, dur[..., None].float(), pit[..., None]))
        ident = {id(v): k for k, v in ref_shim.ft_named_parameters(ref, cfg).items()}
        order[cfg_name] = [[layer.name, [ident[id(v)] for v in layer.variables if id(v) in ident]] for layer in ref.layers]
    tok, mel, _ = alo.make_aligner_inputs(acfg, 2, 12, 21, seed=3)
    ref = ref_shim.reference_aligner(acfg, ap, (tok, mel[:, :-1]))
    ident = {id(v): k for k, v in ref_shim.aligner_named_parameters(ref, acfg).items()}
    order['aligner'] = [[layer.name, [ident.get(id(v)) for v in layer.variables]] for layer in ref.layers]
    pins.meta['keras_order'] = order

    # Aligner.predict (encode=False), the autoregressive loop
    for r, force_long in ((4, False), (1, False), (2, True)):
        p = dict(ap)
        if force_long:
            p['postnet.stop.b'] = torch.tensor([6.0, 0.0, -6.0])
        ref = ref_shim.reference_aligner(c0, p, (tok, mel[:, :-1]))
        ref._set_r(r)
        with torch.no_grad():
            o_ref = ref.predict(tok[0], max_length=10, encode=False, verbose=False)
        pre = f'aligner_predict/r{r}_{int(force_long)}'
        pins.put(pre + '/mel', o_ref['mel'])
        pins.put(pre + '/cross_attention', o_ref['decoder_attention']['Decoder_LastBlock_CrossAttention'])
        pins.meta[pre] = {'start_vec': float(ref.start_vec[0, 0]), 'stop_prob_index': int(ref.stop_prob_index)}

    np.savez_compressed(OUT / 'ref_pins.npz', values=np.concatenate(pins.values), index=np.array(json.dumps(pins.index)))
    body = ',\n'.join(f'{json.dumps(k)}: {json.dumps(v, ensure_ascii=False)}' for k, v in pins.meta.items())
    (OUT / 'ref_pins.json').write_text('{\n' + body + '\n}\n', encoding='utf-8')
    print('wrote ref_pins.npz, ref_pins.json')


if __name__ == '__main__':
    main()
