"""2/3/5/6/7-bit BesTLA weights (S2_CLIP .. S7_CLIP, bestla.h:75-81): RTN quantiser, bit-plane blob layout, unpack.

Pins: the packer's planes against the REFERENCE's own compress_{2,3,5,6,7}bit (kernel_ref.h:178-345, placed as
compressBit*Weight do, bestla_prologue_b.h:512-564) through oracle/_ref/libref_btla.so; the quantised integers against the
reference's quantize_f32_sign_int_rowblock (kernel_ref.h:1608) for every bit width; the unpacked weight against the oracle's
dequantisation.  The reference's answers for these inputs are stored in tests/golden/reference.npz (oracle/golden.py)."""
import ctypes as C

import numpy as np
import pytest

import oracle
from oracle import btla_blob, golden
import neural_speed_b200 as ns

BITS = [2, 3, 5, 6, 7]


@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("alg", ["sym", "asym"])
def test_quantize_pack_unpack(bits, alg):
    rng = np.random.default_rng(10 * bits + (alg == "asym"))
    n, k, g = 100, 256, 64
    w = rng.normal(0, 0.05, (n, k)).astype(np.float32)
    blob = ns.np_bestla_quantize(w, f"int{bits}", g, alg, "fp32", "int8")
    h = btla_blob.parse(blob)
    assert h["dtype"] == (bits | (1 << 8)) and h["prologue"] == 1
    q, sc, zp = oracle.btla_quantize(np.ascontiguousarray(w.T), g, bits, alg == "asym")
    assert q.min() >= -(1 << (bits - 1)) and q.max() <= (1 << (bits - 1)) - 1
    flat = btla_blob.interleave(q, h["ntile"], h["packrow"], h["kpad"], h["npad"])
    assert bytes(h["qbuf"]) == bytes(btla_blob.compress_planes(flat, bits))
    assert len(h["qbuf"]) == h["npad"] * h["kpad"] * bits // 8  # StorageWeightKBlockNInteger::resize, bestla_storage.h:724-745
    want = oracle.btla_dequant(q, sc, zp, g)
    assert np.array_equal(ns.unpack_blob(blob, n, k), want)
    assert np.array_equal(btla_blob.unpack(blob), want)


@pytest.mark.parametrize("bits", BITS)
def test_planes_and_integers_against_the_reference_kernels(bits):
    rng = np.random.default_rng(bits)
    full = 1 << (bits - 1)
    flat = rng.integers(-full, full, 48 * 64).astype(np.int8)

    def compress():
        dst = np.zeros(flat.size * bits // 8, np.uint8)
        assert oracle.ref_btla().ref_btla_compress_bits(bits, flat.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p),
                                                        C.c_size_t(flat.size)) == 0
        return dst

    mine = btla_blob.compress_planes(flat, bits)
    golden.check(f"planes[{bits}].compress", mine, compress)
    assert np.array_equal(btla_blob.decompress_planes(mine, bits, flat.size), flat.astype(np.int32))
    w = rng.uniform(-0.5, 0.5, (128, 40)).astype(np.float32)
    w[:, 1] = np.abs(w[:, 1])
    for asym in (False, True):
        a = oracle.btla_quantize(w, 32, bits, asym, "oracle")
        for i in range(3 if asym else 2):
            golden.check(f"planes[{bits}].rtn[{asym}].{i}", a[i], lambda: oracle.btla_quantize(w, 32, bits, asym, "ref")[i])


def test_split_and_copyattr_keep_the_bit_width():
    rng = np.random.default_rng(3)
    n, k, g = 96, 256, 64
    blob = ns.np_bestla_quantize(rng.normal(0, 0.05, (n, k)).astype(np.float32), "int3", g, "sym", "fp32", "int8")
    L = ns.lib()
    L.ns_split_weight_size.restype = C.c_size_t
    size = L.ns_split_weight_size(blob.ctypes.data_as(C.c_void_p), C.c_size_t(n // 2), C.c_size_t(k))
    assert size > 0
    raw = np.zeros(size + 64, np.uint8)
    dst = raw[(-raw.ctypes.data) % 64:][:size]
    assert L.ns_split_weight(blob.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), C.c_size_t(n), C.c_size_t(k),
                             C.c_size_t(n // 2), C.c_size_t(k), C.c_size_t(1), C.c_size_t(0), False)
    h = btla_blob.parse(dst)
    assert h["dtype"] == (3 | (1 << 8)) and h["n"] == n // 2
    # bestla_split_weight semantics (model_files.h:1538-1562): unpack, slice, re-quantise with the source blob's attributes
    part = np.ascontiguousarray(btla_blob.unpack(blob)[:, n // 2:].T)
    want = ns.np_bestla_quantize(part, "int3", g, "sym", "fp32", "int8")
    assert np.array_equal(btla_blob.unpack(dst), btla_blob.unpack(want))


@pytest.mark.parametrize("name,kind", [("nf4", 0), ("fp4_bnb", 1), ("fp4_e2m1", 2)])
def test_f4_codebooks_against_the_reference_kernels(name, kind):
    """4-bit float weights (F4_NF4 / F4_BNB / F4_E2M1, bestla.h:82-84): codes and scales of the packer == the reference's
    quantize_f32_f4_rowblock (kernel_ref.h:1802), dequantised values == f4_unpack * scale (kernel_ref.h:1416-1436)."""
    rng = np.random.default_rng(40 + kind)
    n, k, g = 96, 256, 64
    w = rng.normal(0, 0.05, (n, k)).astype(np.float32)
    w[3, :64] = 0.0          # an all-zero block: absmax = FLT_MIN
    w[5, 7] = -w[5].max() * 3  # a block whose maximum is negative
    blob = ns.np_bestla_quantize(w, name, g, "sym", "fp32", "fp32")
    h = btla_blob.parse(blob)
    assert h["prologue"] == 2 and h["dtype"] == {0: 4 | (2 << 16), 1: 4 | (1 << 16), 2: 4}[kind]
    wkn = np.ascontiguousarray(w.T)

    def quantize():
        q = np.zeros((k, n), np.int8)
        sc = np.zeros((k // g, n), np.float32)
        assert oracle.ref_btla().ref_btla_quantize_f32_f4_rowblock(kind, wkn.ctypes.data_as(C.c_void_p), q.ctypes.data_as(C.c_void_p),
                                                                   k, n, n, n, sc.ctypes.data_as(C.c_void_p), g) == 0
        return q, sc

    def unpack():
        R = oracle.ref_btla()
        R.ref_btla_f4_unpack.restype = C.c_float
        R.ref_btla_f4_unpack.argtypes = [C.c_int, C.c_int8]
        return np.array([R.ref_btla_f4_unpack(kind, c) for c in range(16)], np.float32)

    q = golden.value(f"f4[{name}].q", lambda: quantize()[0])
    sc = golden.value(f"f4[{name}].sc", lambda: quantize()[1])
    lut = golden.value(f"f4[{name}].lut", unpack)
    want = (lut[q.astype(np.int32) & 15] * np.repeat(sc, g, axis=0)).astype(np.float32)
    assert np.array_equal(ns.unpack_blob(blob, n, k), want)
    flat = btla_blob.interleave(q, h["ntile"], h["packrow"], h["kpad"], h["npad"])
    assert bytes(h["qbuf"]) == bytes(btla_blob.compress_s4(flat, bias=0))
