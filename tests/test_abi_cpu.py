"""CPU: the C-ABI shared library loads and exports every symbol include/yolo2_b200.h declares
(no compute calls without a GPU)."""
import os
import re

from tensorflow_yolo2_b200 import _lib

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))


def header_symbols():
    src = open(os.path.join(ROOT, 'include', 'yolo2_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(y2_[a-z0-9_]+)\s*\(', src)))


def test_library_builds_and_exports_every_declared_symbol():
    from tensorflow_yolo2_b200 import build
    build.build()
    lib = _lib.load()
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), 'missing export: ' + s
    assert sorted(_lib.exported_symbols()) == syms, 'ctypes binding table out of sync with the header'
    assert lib.y2_version() == 101
    # pure host helpers (no GPU needed)
    assert lib.y2_conv_cin_padded(3) == 8 and lib.y2_conv_cin_padded(64) == 64
    assert lib.y2_conv_packed_weight_elems(3, 3, 32) == 32 * 80
    assert lib.y2_conv_packed_weight_elems(1, 1024, 125) == 128 * 1024


def test_conv_fwd_bf16_checks_the_call_before_any_kernel_path():
    """y2_conv_fwd_bf16 refuses a malformed output layout or channel count before it loads the driver or plans a kernel,
    whichever path (stream-K, input-stationary, generic) the shape would take.  Every call here is invalid, so the dummy
    pointers are never dereferenced."""
    import ctypes as C
    lib = _lib.load()
    dummy = C.c_void_p(0x1000)

    def call(Cin, Cout, flags, ldy=0, lo_off=0):
        p = _lib.ConvParams(x=dummy, w_packed=dummy, y=dummy, N=64, H=13, W=13, Cin=Cin, Cout=Cout, ksize=3, flags=flags,
                            alpha=0.1, ldy=ldy, lo_off=lo_off)
        return lib.y2_conv_fwd_bf16(C.byref(p), None), lib.y2_last_error().decode()

    split = _lib.Y2_CONV_OUT_SPLIT
    cases = [
        # stream-K shape, float32 rows of stride 256 < Cout: the rows would overlap
        (dict(Cin=1024, Cout=1024, flags=_lib.Y2_CONV_OUT_F32, ldy=256), -1, 'ldy >= c.Cout'),
        # hi | lo rows whose lo half starts inside the hi half
        (dict(Cin=1024, Cout=1024, flags=split, ldy=2048, lo_off=8), -1, 'c.lo_off >= c.Cout'),
        # lo half past the end of the row
        (dict(Cin=1024, Cout=1024, flags=split, ldy=2000, lo_off=1024), -1, 'c.ldy >= c.lo_off + c.Cout'),
        (dict(Cin=40, Cout=64, flags=0), -2, 'Cin=40 unsupported'),
    ]
    for kw, rc, msg in cases:
        got, err = call(**kw)
        assert got == rc, (kw, got, err)
        assert err.endswith(msg) if rc == -1 else msg in err, (kw, err)
    assert lib.y2_conv_fwd_bf16(None, None) == -1


def test_ops_refuse_cpu_tensors():
    import pytest
    import torch
    from tensorflow_yolo2_b200 import ops
    with pytest.raises(_lib.Y2Error):
        ops._p(torch.zeros(4))


def test_conv1_fused_byte_conversion_identity():
    """conv1_fused.cu converts a byte with ONE fma, bf16_rn(fma(v, 2/255, -1)); the preprocessing kernels (and the
    reference, pascal_voc.py:62-64) compute (v/255)*2-1 in float32.  The two agree after the bf16 rounding for every
    byte value -- that identity is what makes the fused first layer's input bit-identical."""
    import numpy as np
    import torch
    v = np.arange(256, dtype=np.float32)
    ref = ((v / np.float32(255.0)) * np.float32(2.0) - np.float32(1.0)).astype(np.float32)
    k = np.float32(2.0 / 255.0)
    fma = (v.astype(np.float64) * np.float64(k) - 1.0).astype(np.float32)      # exact product, one rounding
    a = torch.tensor(ref).to(torch.bfloat16).view(torch.int16)
    b = torch.tensor(fma).to(torch.bfloat16).view(torch.int16)
    assert torch.equal(a, b)
