"""GPU known-answer tests for the in-register LOP3 decode (bb_debug_decode), the analogue of the reference's
gtest DecodeTest.* suite (testing/cpp/lop3_type_conversion/lowprecision_to_float16.cu:51-101, lowprecision_to_int8.cu):
values -> compress -> interleave -> device decode -> exact equality.  When oracle/_ref is present the same packed
words are also decoded by the REFERENCE's device functions (oracle/ref_shim.cu) and compared bit for bit; without it the
tests that compare with the reference check the product against what those functions return, stated in closed form."""
import ctypes
import os

import numpy as np
import pytest
import torch

import bitblas_oracle as O
from bitblas_b200 import _lib

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "libbitblas_ref.so")


def _pack(values, bits, tgt, layout_il=True):
    packed = O.general_compress(values, bits)
    if layout_il:
        packed = O.interleave_weight(packed, bits, tgt)
    return torch.from_numpy(np.ascontiguousarray(packed)).cuda()


@pytest.mark.parametrize("bits", [4, 2])
@pytest.mark.parametrize("signed", [0, 1])
@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("il", [True, False])
def test_decode_to_16bit_exact(bits, signed, kind, il):
    lib = _lib.load()
    _lib.ensure_init(0)
    rng = np.random.RandomState(0)   # srand(0) in the reference KATs
    vals = rng.randint(0, 2**bits, size=(1, 4096)).astype(np.int8)
    dev = _pack(vals, bits, "float16", il)
    out = torch.empty(4096, dtype=torch.float16 if kind == 0 else torch.bfloat16, device="cuda")
    layout = _lib.BB_LAYOUT_INTERLEAVED_16 if il else _lib.BB_LAYOUT_COMPRESSED
    _lib.check(lib.bb_debug_decode(kind, bits, signed, layout, dev.data_ptr(), out.data_ptr(), dev.numel() // 4, 0))
    torch.cuda.synchronize()
    expect = vals.reshape(-1).astype(np.int32) - (2 ** (bits - 1) if signed else 0)
    assert np.array_equal(out.float().cpu().numpy().astype(np.int32), expect)


@pytest.mark.parametrize("bits", [4, 2])
@pytest.mark.parametrize("signed", [0, 1])
def test_decode_to_int8_exact(bits, signed):
    lib = _lib.load()
    _lib.ensure_init(0)
    rng = np.random.RandomState(0)
    vals = rng.randint(0, 2**bits, size=(1, 4096)).astype(np.int8)
    dev = _pack(vals, bits, "int8")
    out = torch.empty(4096, dtype=torch.int8, device="cuda")
    _lib.check(lib.bb_debug_decode(2, bits, signed, _lib.BB_LAYOUT_INTERLEAVED_8, dev.data_ptr(), out.data_ptr(), dev.numel() // 4, 0))
    torch.cuda.synchronize()
    expect = vals.reshape(-1).astype(np.int32) - (2 ** (bits - 1) if signed else 0)
    assert np.array_equal(out.cpu().numpy().astype(np.int32), expect)


@pytest.mark.parametrize("bits,kind_ref", [(4, 0), (2, 2)])
def test_decode_matches_reference_device_functions(bits, kind_ref):
    """unsigned decode vs decode_i4u_to_f16 / decode_i2u_to_f16 of fast_decoding.hpp run on this GPU; they return the fields."""
    lib = _lib.load()
    _lib.ensure_init(0)
    rng = np.random.RandomState(5)
    vals = rng.randint(0, 2**bits, size=(1, 8192)).astype(np.int8)
    dev = _pack(vals, bits, "float16")
    mine = torch.empty(8192, dtype=torch.float16, device="cuda")
    _lib.check(lib.bb_debug_decode(0, bits, 0, _lib.BB_LAYOUT_INTERLEAVED_16, dev.data_ptr(), mine.data_ptr(), dev.numel() // 4, 0))
    torch.cuda.synchronize()
    assert np.array_equal(mine.cpu().numpy().astype(np.int32), vals.reshape(-1))
    ref = _ref_lib()
    if ref is not None:
        theirs = torch.empty(8192, dtype=torch.float16, device="cuda")
        assert ref.ref_decode_f16(kind_ref, dev.data_ptr(), theirs.data_ptr(), 8192 // 8, None, None, None, None) == 0
        torch.cuda.synchronize()
        assert torch.equal(mine, theirs)


def test_int8_decode_matches_reference_device_functions():
    """unsigned 2-bit decode to int8 vs decode_i2u_to_i8s of fast_decoding.hpp run on this GPU; it returns the fields."""
    lib = _lib.load()
    _lib.ensure_init(0)
    rng = np.random.RandomState(6)
    vals = rng.randint(0, 4, size=(1, 4096)).astype(np.int8)
    dev = _pack(vals, 2, "int8")
    mine = torch.empty(4096, dtype=torch.int8, device="cuda")
    _lib.check(lib.bb_debug_decode(2, 2, 0, _lib.BB_LAYOUT_INTERLEAVED_8, dev.data_ptr(), mine.data_ptr(), dev.numel() // 4, 0))
    torch.cuda.synchronize()
    assert np.array_equal(mine.cpu().numpy(), vals.reshape(-1))
    ref = _ref_lib()
    if ref is not None:
        theirs = torch.empty(4096, dtype=torch.int8, device="cuda")
        assert ref.ref_decode_i8(2, dev.data_ptr(), theirs.data_ptr(), 4096 // 16, None) == 0
        torch.cuda.synchronize()
        assert torch.equal(mine, theirs)


@pytest.mark.parametrize("bits", [4, 2, 1])
@pytest.mark.parametrize("tgt", [0, 16, 8])
def test_device_weight_transform_matches_host(bits, tgt):
    from bitblas_b200.ops.general_matmul import WeightTransform
    rng = np.random.RandomState(7)
    w = torch.from_numpy(rng.randint(0, 2**bits, size=(64, 512)).astype(np.int8))
    wt = WeightTransform(bits, tgt)
    assert torch.equal(wt(w.cuda()).cpu(), wt(w))


# ---- the reference's full decode KAT matrix (testing/cpp/lop3_type_conversion/lowprecision_to_float16.cu:51-101: 20 TESTs,
# lowprecision_to_int8.cu: 6), run side by side with the product's decode / dequantise arithmetic on this GPU --------------
# kind ids of oracle/ref_shim.cu
REF_F16 = dict(I4U=0, I4S=1, I2U=2, I2S=3, I1U=4, I1S=5, I4U_SCALE=6, I4U_ZEROS_ORIGINAL=7, I4U_ZEROS_RESCALE=8,
               I4U_ZEROS_QUANTIZED=9, I2U_SCALE=10, I2U_ZEROS_ORIGINAL=11, I2U_ZEROS_RESCALE=12)
REF_I8 = dict(I4U=0, I4S=1, I2U=2, I2S=3, I1U=4, I1S=5)


def _ref_lib():
    """the reference's decode functions (oracle/build_ref.py), or None where they are not built"""
    if not os.path.exists(REF_SO):
        return None
    ref = ctypes.CDLL(REF_SO)
    ref.ref_decode_f16.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 2 + [ctypes.c_int] + [ctypes.c_void_p] * 4
    ref.ref_decode_i8.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    return ref


@pytest.mark.parametrize("bits,kind", [(4, "I4S"), (2, "I2S")])
def test_signed_decode_vs_reference_device_functions(bits, kind):
    """decode_i{4,2}s_to_f16: the reference's C++ harness subtracts 2^(b-1) - 1 (fast_decoding.hpp:17, MEDIAN 0x6407 / 0x6401)
    while its Python product -- which this library follows -- subtracts 2^(b-1) (lop3.py:23, general_matmul/__init__.py:688-690):
    the two decodes must differ by exactly one everywhere (SURVEY.md 8c)."""
    lib = _lib.load()
    _lib.ensure_init(0)
    vals = np.random.RandomState(11).randint(0, 2**bits, size=(1, 8192)).astype(np.int8)
    dev = _pack(vals, bits, "float16")
    mine = torch.empty(8192, dtype=torch.float16, device="cuda")
    _lib.check(lib.bb_debug_decode(0, bits, 1, _lib.BB_LAYOUT_INTERLEAVED_16, dev.data_ptr(), mine.data_ptr(), dev.numel() // 4, 0))
    torch.cuda.synchronize()
    assert np.array_equal(mine.cpu().numpy().astype(np.int32), vals.reshape(-1).astype(np.int32) - 2 ** (bits - 1))
    ref = _ref_lib()
    if ref is not None:
        theirs = torch.empty(8192, dtype=torch.float16, device="cuda")
        assert ref.ref_decode_f16(REF_F16[kind], dev.data_ptr(), theirs.data_ptr(), 8192 // 8, None, None, None, None) == 0
        torch.cuda.synchronize()
        assert torch.equal(mine + 1, theirs)


@pytest.mark.parametrize("kind,bits,mode", [
    ("I4U_SCALE", 4, 1), ("I4U_ZEROS_ORIGINAL", 4, 2), ("I4U_ZEROS_RESCALE", 4, 3), ("I4U_ZEROS_QUANTIZED", 4, 4),
    ("I2U_SCALE", 2, 1), ("I2U_ZEROS_ORIGINAL", 2, 2), ("I2U_ZEROS_RESCALE", 2, 3)])
def test_dequant_arithmetic_vs_reference_device_functions(kind, bits, mode):
    """DecodeTest.*WithScaling / *WithZerosOriginal / *Rescale / *Quantized: the tensor-core GEMM path's dequantise arithmetic
    (dq_finish: fp16 sub, then mul -- or one fma for rescale) must reproduce the reference's rounding order bit for bit, with
    non-trivial fp16 scales and non-integer fp16 zero points (one per group of 8 outputs, as in the reference KATs)."""
    lib = _lib.load()
    _lib.ensure_init(0)
    rng = np.random.RandomState(12)
    n = 16384
    vals = rng.randint(0, 2**bits, size=(1, n)).astype(np.int8)
    dev = _pack(vals, bits, "float16")
    g = n // 8
    scale = torch.from_numpy((rng.rand(g) * 3 + 0.013).astype(np.float16)).cuda()
    zeros_np = (rng.rand(g) * (2**bits - 1)).astype(np.float16)
    if mode == 3:
        zeros_np = (zeros_np.astype(np.float32) * scale.cpu().numpy().astype(np.float32)).astype(np.float16)
    zeros = torch.from_numpy(zeros_np).cuda()
    qz = torch.from_numpy(rng.randint(0, 2**bits, size=g).astype(np.int32)).cuda()
    mine = torch.empty(n, dtype=torch.float16, device="cuda")
    _lib.check(lib.bb_debug_dequant(0, bits, 0, _lib.BB_LAYOUT_INTERLEAVED_16, mode, dev.data_ptr(), scale.data_ptr(),
                                    zeros.data_ptr(), qz.data_ptr(), mine.data_ptr(), dev.numel() // 4, 0))
    torch.cuda.synchronize()
    ref = _ref_lib()
    if ref is not None:
        theirs = torch.empty(n, dtype=torch.float16, device="cuda")
        assert ref.ref_decode_f16(REF_F16[kind], dev.data_ptr(), theirs.data_ptr(), g, scale.data_ptr(),
                                  zeros.data_ptr() if mode in (2, 3) else None, qz.data_ptr() if mode == 4 else None, None) == 0
        torch.cuda.synchronize()
        assert torch.equal(mine, theirs), (mine[:16], theirs[:16])
    # and the oracle's A_dtype dequantise (the model every parity test is checked against) states the same numbers
    u = torch.from_numpy(vals.reshape(-1).astype(np.float32)).half()
    s8, z8, q8 = (scale.cpu().repeat_interleave(8), zeros.cpu().repeat_interleave(8), qz.cpu().repeat_interleave(8).half())
    rescale = (u * s8 - z8) if bits == 2 else torch.addcmul(-z8.float(), u.float(), s8.float()).half()   # 2-bit: two roundings (lop3.py:633-635)
    expect = {1: u * s8, 2: (u - z8) * s8, 3: rescale, 4: (u - q8) * s8}[mode]
    assert torch.equal(mine.cpu(), expect)


@pytest.mark.parametrize("kind,bits,signed", [("I4U", 4, 0), ("I4S", 4, 1), ("I2U", 2, 0), ("I2S", 2, 1)])
def test_int8_decode_matrix_vs_reference_device_functions(kind, bits, signed):
    """lowprecision_to_int8.cu DecodeTest.{U,}Int{4,2}ToINT8.  Signed: the reference harness subtracts 2^(b-1) - 1
    (decode_i4s_to_i8s: 7, lop3.py:1016 -- SURVEY.md 8c defect (iii)); the Python product and this library subtract 2^(b-1)."""
    lib = _lib.load()
    _lib.ensure_init(0)
    vals = np.random.RandomState(13).randint(0, 2**bits, size=(1, 8192)).astype(np.int8)
    dev = _pack(vals, bits, "int8")
    mine = torch.empty(8192, dtype=torch.int8, device="cuda")
    _lib.check(lib.bb_debug_decode(2, bits, signed, _lib.BB_LAYOUT_INTERLEAVED_8, dev.data_ptr(), mine.data_ptr(), dev.numel() // 4, 0))
    torch.cuda.synchronize()
    assert np.array_equal(mine.cpu().numpy().astype(np.int32), vals.reshape(-1).astype(np.int32) - (2 ** (bits - 1) if signed else 0))
    ref = _ref_lib()
    if ref is not None:
        theirs = torch.empty(8192, dtype=torch.int8, device="cuda")
        assert ref.ref_decode_i8(REF_I8[kind], dev.data_ptr(), theirs.data_ptr(), 8192 // 16, None) == 0
        torch.cuda.synchronize()
        delta = (theirs.cpu().to(torch.int32) - mine.cpu().to(torch.int32))
        assert (delta == (1 if signed else 0)).all(), delta.unique()


@pytest.mark.skipif(not os.path.exists(REF_SO), reason="oracle/_ref not built")
@pytest.mark.parametrize("kind,signed", [("I1U", 0), ("I1S", 1)])
def test_one_bit_reference_decode_pins_the_generic_path(kind, signed):
    """DecodeTest.{U,}Int1ToFloat16: 1-bit weights run through the generic kernel here (no in-register fast path), whose
    arithmetic is the oracle's; the reference's device decode on the C++-interleaved words must agree with it: uint1 -> {0, 1},
    int1 -> {-1, +1} (lop3.py:723-727; SURVEY.md 8c defect (ii): the TIR decode would give {0, -1})."""
    ref = _ref_lib()
    href = ctypes.CDLL(REF_SO)
    href.ref_general_compress.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    href.ref_general_interleave_fp16.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t]
    vals = np.random.RandomState(14).randint(0, 2, size=4096).astype(np.int8)
    comp = np.zeros(4096 // 8, dtype=np.int8)
    inter = np.zeros_like(comp)
    href.ref_general_compress(vals.ctypes.data, comp.ctypes.data, 1, 4096, 0)
    href.ref_general_interleave_fp16(comp.ctypes.data, inter.ctypes.data, 1, comp.nbytes)
    dev = torch.from_numpy(inter).cuda()
    theirs = torch.empty(4096, dtype=torch.float16, device="cuda")
    assert ref.ref_decode_f16(REF_F16[kind], dev.data_ptr(), theirs.data_ptr(), 4096 // 8, None, None, None, None) == 0
    torch.cuda.synchronize()
    got = theirs.cpu().numpy().astype(np.int32)
    expect = O.decode_fields(torch.from_numpy(vals.astype(np.int32)), "int" if signed else "uint", 1, torch.float32).numpy().astype(np.int32)
    assert np.array_equal(got, expect)
