"""CPU-side checks (no GPU): the C-ABI library loads and exports every symbol include/ns_b200.h declares,
the host packing API reproduces the oracle / the reference's blob format, and compute entry points fail loudly
(no CPU fallback) when there is no CUDA device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import oracle
from oracle import btla_blob
import neural_speed_b200 as ns

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "ns_b200.h")).read()
    declared = set(re.findall(r"^NS_API\s+[^;(]*?\b(\w+)\s*\(", hdr, re.M))
    assert len(declared) >= 45
    L = ns.lib()
    missing = [s for s in sorted(declared) if not hasattr(L, s)]
    assert not missing, missing
    assert declared == set(ns.EXPORTS), declared ^ set(ns.EXPORTS)
    assert b"sm_100a" in L.ns_version()


@pytest.mark.skipif(_has_gpu(), reason="checks the no-device behaviour")
def test_compute_fails_loudly_without_device():
    L = ns.lib()
    w = L.ns_weight_from_q4_0(C.c_void_p(1), 4, 32, 18, 0, None)
    assert not w
    assert "no CUDA device" in ns.last_error() and "no CPU fallback" in ns.last_error()
    x = np.zeros(32, np.float32)
    rc = L.ns_mul_mat_q4_0_f32_host(x.ctypes.data_as(C.c_void_p), 18, x.ctypes.data_as(C.c_void_p),
                                    x.ctypes.data_as(C.c_void_p), 32, 1, 1)
    assert rc == -2  # NS_E_NODEVICE


def test_engine_and_comm_fail_loudly_without_device():
    """the eval step and the NVLink exchange have no CPU implementation either"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    with pytest.raises(RuntimeError, match="no CUDA device"):
        ns.Llama(32, 64, 2, 2, 1, 64, 8)
    assert not ns.lib().ns_comm_create(0, 2, 1024, None)
    assert "no CUDA device" in ns.last_error()


def test_host_q4_0_quantiser_matches_oracle():
    w = np.random.default_rng(3).normal(0, 0.02, (16, 512)).astype(np.float32)
    w[2, 32:64] = 0
    assert np.array_equal(ns.quantize_q4_0_host(w), oracle.quantize_q4_0(w))


@pytest.mark.parametrize("wdt,bits", [("int4", 4), ("int8", 8)])
@pytest.mark.parametrize("alg", ["sym", "asym"])
@pytest.mark.parametrize("g,sdt,cdt", [(32, "fp32", "int8"), (128, "fp32", "int8"), (128, "bf16", "fp32"), (-1, "fp32", "bf16"),
                                       (128, "fp16", "int8")])
def test_quantize_pack_roundtrip_vs_oracle(wdt, bits, alg, g, sdt, cdt):
    if wdt == "int8" and alg == "asym" and cdt == "int8":
        cdt = "bf16"  # the reference excludes (S8, asym) from int8 compute (bestla_gemm.cpp:256)
    n, k = 100, 384  # n not a multiple of NTile=48
    w = np.random.default_rng(5).uniform(-0.5, 0.5, (n, k)).astype(np.float32)
    blob = ns.np_bestla_quantize(w, wdt, g, alg, sdt, cdt)
    gg = k if g == -1 else g
    q, sc, zp = oracle.btla_quantize(np.ascontiguousarray(w.T), gg, bits, alg == "asym")
    # 1. dequantised content == oracle quantiser + oracle dequant (scales rounded to the stored dtype)
    if sdt == "bf16":
        sc_s = oracle.bf16_bits_to_f32(oracle.f32_to_bf16_bits(sc))
    elif sdt == "fp16":
        sc_s = sc.astype(np.float16).astype(np.float32)
    else:
        sc_s = sc
    want = oracle.btla_dequant(q, sc_s, zp, gg)
    got = ns.unpack_blob(blob, n, k)
    assert np.array_equal(got, want)
    # 2. the oracle's blob parser reads the product's blob identically
    assert np.array_equal(btla_blob.unpack(blob), want)
    h = btla_blob.parse(blob)
    assert h["size"] == blob.size and h["n"] == n and h["k"] == k and h["blocksize"] == gg
    # 3. byte-for-byte equal to the oracle's serializer for the same core
    core = {"int8": "avx512_vnni_kblock", "bf16": "amx_bf16", "fp32": "avx512f", "fp16": "amx_fp16"}[cdt]
    if cdt == "bf16" and gg % 32 != 0:
        core = "avx512f"
    st = {"fp32": btla_blob.F32, "bf16": btla_blob.BF16, "fp16": btla_blob.F16}[sdt]
    ref = btla_blob.serialize(q, sc, zp, gg, core, btla_blob.S4_CLIP if bits == 4 else btla_blob.S8, st,
                              base_addr=blob.ctypes.data)
    assert bytes(blob) == ref


@pytest.mark.parametrize("g", [32, 128])
def test_nf4_quantize_pack(g):
    n, k = 96, 256
    w = np.random.default_rng(6).normal(0, 0.05, (n, k)).astype(np.float32)
    blob = ns.np_bestla_quantize(w, "nf4", g, "sym", "fp32", "fp32")
    q, sc = oracle.btla_quantize_nf4(np.ascontiguousarray(w.T), g)
    want = oracle.btla_dequant(q, sc, None, g, nf4=True)
    assert np.array_equal(ns.unpack_blob(blob, n, k), want)
    assert np.array_equal(btla_blob.unpack(blob), want)
    assert btla_blob.parse(blob)["prologue"] == 2
    ref = btla_blob.serialize(q, sc, None, g, "avx512f", btla_blob.F4_NF4, btla_blob.F32, base_addr=blob.ctypes.data)
    assert bytes(blob) == ref


def test_qpack_with_zero_points_and_gidx():
    rng = np.random.default_rng(8)
    n, k, g = 64, 256, 64
    q = rng.integers(-8, 8, (k, n)).astype(np.int8)
    sc = rng.uniform(0.01, 0.02, (k // g, n)).astype(np.float32)
    zp = rng.integers(-8, 8, (k // g, n)).astype(np.int8)
    g_idx = rng.permutation(np.repeat(np.arange(k // g), g)).astype(np.int32)
    blob = ns.np_bestla_qpack(q, sc, zp, g_idx, "int4", g, "asym", "fp32", "int8")
    ref = btla_blob.serialize(q, sc, zp, g, "avx512_vnni_kblock", btla_blob.S4_CLIP, btla_blob.F32, g_idx=g_idx,
                              base_addr=blob.ctypes.data)
    assert bytes(blob) == ref
    want = oracle.btla_dequant(q, sc, zp, g)
    assert np.array_equal(ns.unpack_blob(blob, n, k), want)
    sh = np.frombuffer(btla_blob.parse(blob)["shuffle"], np.int32)
    # every group's slots hold exactly the columns whose g_idx names that group, in ascending order
    for b in range(k // g):
        assert np.array_equal(sh[b * g:(b + 1) * g], np.nonzero(g_idx == b)[0])


def test_oracle_blob_layout_against_reference_kernels():
    """pin oracle/btla_blob.py's interleave/compress against kernel_ref.h padding_interleave + compress_s8_s4 (their answers for
    these inputs: tests/golden/reference.npz)"""
    from oracle import golden
    rng = np.random.default_rng(12)
    for (ntile, packrow, k, n) in [(48, 4, 64, 100), (48, 1, 40, 48), (24, 2, 64, 30), (48, 2, 96, 144)]:
        q = rng.integers(-8, 8, (k, n)).astype(np.int8)
        kpad = -(-k // packrow) * packrow
        npad = -(-n // ntile) * ntile

        def interleave():
            dst = np.zeros(kpad * npad, np.int8)
            oracle.ref_btla().ref_btla_padding_interleave_s8(q.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), k, n, kpad,
                                                             npad, n, kpad, ntile, packrow)
            return dst

        def compress(dst):
            packed = np.zeros(dst.size // 2, np.uint8)
            oracle.ref_btla().ref_btla_compress_s8_s4(dst.ctypes.data_as(C.c_void_p), packed.ctypes.data_as(C.c_void_p),
                                                      C.c_size_t(dst.size))
            return packed

        key = f"blob_layout[{ntile}-{packrow}-{k}-{n}]"
        mine = btla_blob.interleave(q, ntile, packrow, kpad, npad)
        golden.check(key + ".interleave", mine, interleave)
        golden.check(key + ".compress_s4", btla_blob.compress_s4(mine), lambda: compress(interleave()))


def test_packweight_copyattr_matches_direct_quantisation():
    """bestla_packweight_copyattr (ne_bestla.cpp:79-112): re-quantising with the attributes read from a blob gives the same
    bytes as quantising with those attributes directly."""
    rng = np.random.default_rng(77)
    n, k = 96, 512
    w_kn = rng.uniform(-0.5, 0.5, (k, n)).astype(np.float32)      # copyattr passes isTrans=false: [K][N]
    for alg, sdt, cdt, g in (("sym", "fp32", "int8", 128), ("asym", "bf16", "int8", 32), ("sym", "fp32", "fp32", 64),
                             ("asym", "fp32", "bf16", 128)):
        src = ns.np_bestla_quantize(rng.uniform(-1, 1, (n, k)).astype(np.float32), "int4", g, alg, sdt, cdt)
        want = ns.np_bestla_quantize(np.ascontiguousarray(w_kn.T), "int4", g, alg, sdt, cdt)
        raw = np.zeros(src.size + 64, np.uint8)          # the blob's internal padding depends on the address: align like the packer
        dst = raw[(-raw.ctypes.data) % 64:][:src.size]
        ns.lib().bestla_packweight_copyattr(w_kn.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), n, k, n,
                                            src.ctypes.data_as(C.c_void_p))
        assert dst.size == want.size and np.array_equal(dst, want), (alg, sdt, cdt, g)


def test_public_header_is_plain_c_and_matches_the_ctypes_structs(tmp_path):
    """include/ns_b200.h is the drop-in boundary: it must compile as C99 (what cgo / JNI / ctypes-gen consume) and as C++, and
    the struct the Python binding passes by pointer must have the header's layout."""
    import shutil
    import subprocess
    if not shutil.which("gcc"):
        pytest.skip("gcc missing")
    src = tmp_path / "t.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ns_b200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu\\n", sizeof(ns_llama_hparams), offsetof(ns_llama_hparams, n_vocab),'
                   ' offsetof(ns_llama_hparams, n_ctx), offsetof(ns_llama_hparams, norm_eps), offsetof(ns_llama_hparams, rope_scale));'
                   'return 0;}\n')
    inc = os.path.join(ROOT, "include")
    exe = tmp_path / "t"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", inc, str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    H = ns.LlamaHParams
    assert got == [C.sizeof(H), H.n_vocab.offset, H.n_ctx.offset, H.norm_eps.offset, H.rope_scale.offset]
    if shutil.which("g++"):
        r = subprocess.run(["g++", "-std=c++14", "-Wall", "-Werror", "-fsyntax-only", "-I", inc, "-x", "c++", str(src)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
