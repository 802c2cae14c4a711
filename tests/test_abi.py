"""CPU tests of the C-ABI boundary: the library loads without a GPU, exports every symbol include/ttsb.h declares,
validates arguments and reports errors through ttsb_last_error (no compute calls here)."""
import ctypes as C
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope='module')
def cdll():
    from transformertts_b200 import build, lib
    build.build(verbose=False)
    return lib.load()


def test_header_symbols_are_all_exported(cdll):
    header = (ROOT / 'include' / 'ttsb.h').read_text()
    names = set(re.findall(r'\b(ttsb_[a-z0-9_]+)\s*\(', header))
    names -= {'ttsb_gemm_args', 'ttsb_mha_args'}
    assert len(names) >= 18
    for n in sorted(names):
        assert hasattr(cdll, n), f'{n} declared in include/ttsb.h but not exported by libttsb.so'
    from transformertts_b200 import lib
    assert set(lib.EXPORTS) == names


def test_abi_version_and_error_text(cdll):
    assert cdll.ttsb_abi_version() == 3
    rc = cdll.ttsb_linear_fwd(None, None)
    assert rc == -1
    assert b'NULL' in cdll.ttsb_last_error()


def test_struct_layout_matches_header():
    """ctypes mirrors of ttsb_gemm_args / ttsb_mha_args: field order and names follow the header."""
    from transformertts_b200 import lib
    header = (ROOT / 'include' / 'ttsb.h').read_text()
    for struct, cls in (('ttsb_gemm_args', lib.GemmArgs), ('ttsb_mha_args', lib.MhaArgs)):
        body = re.search(r'typedef struct %s \{(.*?)\} %s;' % (struct, struct), header, re.S).group(1)
        body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
        fields = []
        for decl in body.split(';'):
            decl = decl.strip()
            if not decl:
                continue
            for part in decl.split(','):
                name = re.findall(r'([A-Za-z_][A-Za-z0-9_]*)\s*(?:\[\d+\])?\s*$', part.strip())[0]
                fields.append(name)
        assert fields == [f[0] for f in cls._fields_], struct


def test_argument_validation_without_gpu(cdll):
    from transformertts_b200 import lib
    a = lib.GemmArgs()
    a.B, a.T, a.N, a.block_n, a.num_segments = 1, 8, 64, 48 + 1, 1
    assert cdll.ttsb_linear_fwd(C.byref(a), None) == -1
    assert b'block_n' in cdll.ttsb_last_error()
    m = lib.MhaArgs()
    assert cdll.ttsb_mha_fwd(C.byref(m), None) == -1
    assert cdll.ttsb_stft_mel_log(None, 1, 1000, None, 80, 0, None, None) == -1
    assert cdll.ttsb_durations_to_int(None, C.c_float(1.0), None, None, 1, 1, None, None, None) == -1
    # the training attention kernels: the support query is pure host logic; bad arguments are refused before any CUDA call
    assert cdll.ttsb_attn_probs_supported(128, 1008) == 1 and cdll.ttsb_attn_probs_supported(64, 48) == 1
    assert cdll.ttsb_attn_probs_supported(192, 208) == 1
    assert cdll.ttsb_attn_probs_supported(256, 1008) == 0      # Q tile + K ring + staging boxes exceed 227 KB
    assert cdll.ttsb_attn_probs_supported(96, 1008) == 0 and cdll.ttsb_attn_probs_supported(128, 1001) == 0
    assert cdll.ttsb_attn_probs_fwd(None, 768, 0, 256, 1, 2, 100, 128, None, C.c_float(0.1), C.c_float(0.1), 0, 0, None, None, 112, None) == -1
    assert b'ttsb_attn_probs_fwd' in cdll.ttsb_last_error()
    assert cdll.ttsb_attn_ds_bwd(None, 256, 0, None, 768, 512, 1, 2, 100, 128, None, None, None, C.c_float(0.1), C.c_float(0.1), 0, 0, None, 112, None) == -1
    assert b'ttsb_attn_ds_bwd' in cdll.ttsb_last_error()
    # Expand backward walks rows as float4: d % 4 != 0 and unaligned rows are refused (the pointers are never dereferenced)
    dur = C.c_void_p(0x1000)
    assert cdll.ttsb_expand_bwd(C.c_void_p(0x2000), dur, 1, 4, 8, 6, C.c_void_p(0x3000), None) == -1
    assert b'ttsb_expand_bwd' in cdll.ttsb_last_error()
    assert cdll.ttsb_expand_bwd(C.c_void_p(0x2004), dur, 1, 4, 8, 128, C.c_void_p(0x3000), None) == -1
    assert cdll.ttsb_expand_bwd(C.c_void_p(0x2000), dur, 1, 4, 8, 128, C.c_void_p(0x3008), None) == -1


def test_product_package_never_imports_the_oracle():
    """The oracle is test infrastructure: the product path must not route through it."""
    for f in (ROOT / 'transformertts_b200').rglob('*.py'):
        src = f.read_text()
        assert 'import oracle' not in src and 'from oracle' not in src, f
