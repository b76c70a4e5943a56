"""CPU-side checks of the C ABI: the library builds, loads, and exports every symbol include/sipmask_b200.h declares."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from sipmask_b200 import _lib, build
    path = build.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, 'include', 'sipmask_b200.h')).read()
    declared = sorted(set(re.findall(r'\b(smb_[a-z0-9_]+)\s*\(', header)))
    assert declared, 'no declarations parsed'
    for name in declared:
        assert hasattr(lib, name), 'missing export %s' % name
    assert sorted(declared) == sorted(_lib.SYMBOLS)
    assert lib.smb_version() >= 100


def test_ops_fail_loudly_without_cuda():
    import torch
    from sipmask_b200 import ops, _lib
    if torch.cuda.is_available():
        pytest.skip('CUDA present')
    with pytest.raises(_lib.SmbError):
        ops.crop_split(torch.zeros(4, 4, 4, 1), torch.zeros(1, 4))
    with pytest.raises(_lib.SmbError):
        ops.nms(torch.zeros(3, 5), 0.5)
    with pytest.raises(_lib.SmbError):
        ops.mask_assemble(torch.zeros(32, 4, 4), torch.zeros(1, 128), torch.zeros(1, 4), 0.5)


def test_upsample_rejects_an_output_the_input_cannot_fill():
    """smb_upsample_bilinear writes out_h x out_w <= (H*factor) x (W*factor); a larger output (or a factor-1 copy into
    another size) is refused before any memory is touched."""
    from sipmask_b200 import _lib
    lib = _lib.lib()
    p = ctypes.c_void_p(256)                       # never dereferenced: the arguments are rejected first
    assert lib.smb_upsample_bilinear(p, 8, p, 8, 0, 1, 7, 10, 8, 2, 15, 20, 0, None) != 0
    assert lib.smb_upsample_bilinear(p, 8, p, 8, 0, 1, 7, 10, 8, 2, 14, 21, 0, None) != 0
    assert lib.smb_upsample_bilinear(p, 8, p, 8, 0, 1, 7, 10, 8, 1, 6, 10, 0, None) != 0


def test_conv_plan_info_rejects_a_null_plan():
    from sipmask_b200 import _lib, conv
    vals = (ctypes.c_int * len(conv.PLAN_INFO_FIELDS))()
    assert _lib.lib().smb_conv_plan_info(None, vals, len(vals)) < 0
    assert len(conv.PLAN_INFO_FIELDS) == 11


def test_sass_contains_blackwell_instructions():
    """The conv kernel must be real tcgen05/TMA code (B200_PROFILING.md 'What proves a Blackwell-native kernel')."""
    import shutil
    import subprocess
    from sipmask_b200 import build
    if shutil.which('cuobjdump') is None:
        pytest.skip('cuobjdump not available')
    sass = subprocess.run(['cuobjdump', '-sass', build.LIB], capture_output=True, text=True).stdout
    for mnemonic in ('UTCHMMA', 'UTMALDG', 'LDTM'):
        assert mnemonic in sass, mnemonic
