"""Golden vectors produced by the REFERENCE'S OWN CODE:

    TTS_REFERENCE=<checkout of as-ideas/TransformerTTS> python tests/golden/make_golden_ref.py

The unmodified model/models.py of the reference (ForwardTransformer, Aligner) is imported and executed on top of
tests/tf_shim -- a torch-backed stand-in for the TensorFlow/Keras primitives, because TensorFlow cannot be installed in
this image (see tests/tf_shim/README.md; tests/golden/make_golden_tf.py is the same script for a machine that has the real
TensorFlow).  Weights are the seed-7 set of oracle.forward_oracle.init_params mapped onto the Keras variables; inputs come
from the seeded generators of the oracle modules.  Files written:

  c1_forward.npz     BASELINE configs[0] (2+2 layers, d=128, B=1, 32 phonemes -> 250 frames), forced and predicted durations,
                     and a ragged batch of 3 (same keys as before, now reference outputs)
  ref_lj256.npz      LJ256 (6+6 conv blocks, d=256), ragged batch of 2, 48 phonemes -> 300 frames
  ref_train_c1.npz   one reference _train_step (dropout 0): losses and gradients (small tensors whole, 4096 seeded samples
                     of every large kernel), recovered from the Keras-Adam first-moment slots (m = 0.1 g after step 1)
  aligner_small.npz  Aligner teacher-forced validation step (r = 1, decoder diagonal loss on)

The audio golden (audio_mel.npz) stays oracle-generated (tests/golden/make_golden.py): librosa cannot be imported here.
"""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / 'tests'))
import ref_shim  # noqa: E402
from oracle import aligner_oracle as alo  # noqa: E402
from oracle import forward_oracle as fo  # noqa: E402

OUT = Path(__file__).resolve().parent
SAMPLE = 4096
SOURCE = 'reference code on tests/tf_shim'


def grad_sample_index(name: str, numel: int) -> np.ndarray:
    """Seeded element sample of a large gradient tensor (shared with the tests)."""
    if numel <= SAMPLE:
        return np.arange(numel)
    seed = sum(ord(c) * (i + 1) for i, c in enumerate(name)) % (2 ** 31)
    return np.sort(np.random.default_rng(seed).choice(numel, SAMPLE, replace=False))


def main(real_tf: bool = False):
    global SOURCE
    if real_tf:
        SOURCE = 'reference code on TensorFlow'
    ref_shim.activate(real_tf=real_tf)
    import tensorflow as tf  # the shim (or, from make_golden_tf.py, the real one)
    torch.set_num_threads(4)
    torch.manual_seed(0)
    cfg = fo.CONFIGS['C1']
    p = fo.init_params(cfg, seed=7)
    tok, dur, pit = fo.make_inputs('full', 1, 32, 250, seed=100)
    durf, pitf = dur[..., None].float(), pit[..., None]
    model = ref_shim.reference_forward_transformer(cfg, p, (tok, durf, pitf))
    with torch.no_grad():
        out = model.call(tok, target_durations=durf, target_pitch=pitf, training=False)
        pred = model.predict(tok, encode=False)
        pred_int = torch.round(pred['duration'][..., 0] * 1.0).to(torch.int32)
        tok3, dur3, pit3 = fo.make_inputs('ragged', 3, 40, 200, seed=101)
        out3 = model.call(tok3, target_durations=dur3[..., None].float(), target_pitch=pit3[..., None], training=False)
    np.savez_compressed(
        OUT / 'c1_forward.npz', source=SOURCE,
        tokens=tok.numpy(), durations=dur.numpy(), pitch=pit.numpy(),
        mel=out['mel'].numpy(), duration_pred=out['duration'].numpy(), pitch_pred=out['pitch'].numpy(),
        pred_mel=pred['mel'].numpy(), pred_int_durations=pred_int.numpy(), pred_duration=pred['duration'].numpy(),
        tokens3=tok3.numpy(), durations3=dur3.numpy(), pitch3=pit3.numpy(), mel3=out3['mel'].numpy(),
        duration_pred3=out3['duration'].numpy(), pitch_pred3=out3['pitch'].numpy(),
        expanded_mask3=out3['expanded_mask'].numpy())

    # ---- LJ256, ragged
    cfgL = fo.CONFIGS['LJ256']
    pL = fo.init_params(cfgL, seed=7)
    tokL, durL, pitL = fo.make_inputs('ragged', 2, 48, 300, seed=201)
    mL = ref_shim.reference_forward_transformer(cfgL, pL, (tokL, durL[..., None].float(), pitL[..., None]))
    with torch.no_grad():
        oL = mL.call(tokL, target_durations=durL[..., None].float(), target_pitch=pitL[..., None], training=False)
    np.savez_compressed(OUT / 'ref_lj256.npz', source=SOURCE, B=2, Tp=48, Tm=300, seed=201,
                        tokens=tokL.numpy(), durations=durL.numpy(), pitch=pitL.numpy(), mel=oL['mel'].numpy(),
                        duration_pred=oL['duration'].numpy(), pitch_pred=oL['pitch'].numpy())

    # ---- one training step of the reference (dropout 0)
    cfgT = dict(cfg, dropout_rate=0.0, predictors_dropout=0.0)
    tokT, durT, pitT = fo.make_inputs('ragged', 3, 24, 150, seed=301)
    melT = fo.make_mel_targets(durT, 80, seed=302)
    mT = ref_shim.reference_forward_transformer(cfgT, p, (tokT, durT[..., None].float(), pitT[..., None]))
    mT._compile(optimizer=tf.keras.optimizers.Adam(1e-4, beta_1=0.9, beta_2=0.98, epsilon=1e-9))
    named = ref_shim.ft_named_parameters(mT, cfgT)
    oT = mT.train_step(tokT, melT, durT, pitT)
    grads = {}
    for name, var in named.items():
        g = (ref_shim.adam_first_moment(mT.optimizer, var) / (1.0 - 0.9)).reshape(-1).numpy()
        grads['g:' + name] = g[grad_sample_index(name, g.size)].astype(np.float32)
        grads['n:' + name] = np.float32(np.linalg.norm(g.astype(np.float64)))
    np.savez_compressed(OUT / 'ref_train_c1.npz', source=SOURCE, B=3, Tp=24, Tm=150, seed=301,
                        mel_seed=302, loss=float(oT['loss']), mel_loss=float(oT['losses']['mel']),
                        duration_loss=float(oT['losses']['duration']), pitch_loss=float(oT['losses']['pitch']), **grads)

    # ---- Aligner
    acfg = alo.ALIGNER_CONFIGS['A-small']
    ap = alo.init_aligner_params(acfg, seed=7)
    tokens, amel, stop = alo.make_aligner_inputs(acfg, 3, 24, 61, seed=503)
    am = ref_shim.reference_aligner(acfg, ap, (tokens, amel[:, :-1]))
    am._compile(stop_scaling=acfg['stop_loss_scaling'], optimizer=tf.keras.optimizers.Adam(1e-4))
    am.set_constants(reduction_factor=1, force_decoder_diagonal=True)
    with torch.no_grad():
        aout = am.val_step(tokens, amel, stop)
    np.savez_compressed(OUT / 'aligner_small.npz', source=SOURCE, B=3, Tp=24, Tm=61, seed=503,
                        mel=aout['mel'].numpy(), stop_prob=aout['stop_prob'].numpy(),
                        last_attention=aout['decoder_attention']['Decoder_LastBlock_CrossAttention'].numpy(),
                        loss=float(aout['loss']), mel_loss=float(aout['losses']['mel']),
                        stop_loss=float(aout['losses']['stop_prob']), diag_loss=float(aout['losses']['diag_loss']))
    print('wrote', sorted(f.name for f in OUT.glob('*.npz')))


if __name__ == '__main__':
    main()
