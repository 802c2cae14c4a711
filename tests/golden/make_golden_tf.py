"""Golden vectors from the UNMODIFIED reference on REAL TensorFlow (SURVEY.md 8c: "prefer the real reference if it appears").

    python tests/golden/make_golden_tf.py        # needs `import tensorflow` (>= 2.2) and $TTS_REFERENCE

This image has no TensorFlow wheel and no network, so this script cannot run here; it is committed so that anyone with a
TensorFlow box can regenerate tests/golden/*.npz from the real thing and re-run the suite.  It is the same program as
make_golden_ref.py (same seeds, same files, same keys) with the tests/tf_shim packages left OFF sys.path: the Keras layers
of the reference expose the same attribute names the shim mirrors (kernel / bias / gamma / beta / embeddings, Variable.assign,
optimizer.get_slot), which is all ref_shim.py relies on.  Note: under real TF the tensors are tf.Tensors, so torch inputs
are converted with .numpy() by TF itself; the np.savez calls only use .numpy().
"""
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT / 'tests'))
sys.path.insert(0, str(ROOT / 'tests' / 'golden'))

import ref_shim  # noqa: E402

if __name__ == '__main__':
    if not ref_shim.real_tensorflow_available():
        raise SystemExit('TensorFlow is not importable on this machine: use make_golden_ref.py (reference code on tests/tf_shim)')
    import make_golden_ref
    make_golden_ref.main(real_tf=True)
