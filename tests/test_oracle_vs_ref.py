"""Pin the CPU oracle (oracle/oracle_*.c) against the reference's own code (oracle/_ref/*.so, the reference's sources compiled
by oracle/Makefile).  Everything here must be BIT-exact.  The reference's answers for these exact inputs are stored in
tests/golden/reference.npz (oracle/golden.py; recorded by tests/golden/make_golden_reference.py), so the pins hold on machines
without the reference."""
import numpy as np
import pytest

import oracle
from oracle import golden


def _rng(seed):
    return np.random.default_rng(seed)


def test_fp16_roundtrip_all_bit_patterns():
    L = oracle.lib()
    hs = range(0, 1 << 16, 1)
    golden.check("fp16_to_fp32", np.array([L.orc_fp16_to_fp32(h) for h in hs], np.float32),     # every NaN alike
                 lambda: np.array([oracle.ref_ggml().ref_fp16_to_fp32(h) for h in hs], np.float32))
    r = _rng(0)
    xs = np.concatenate([r.normal(0, 1, 20000), r.normal(0, 1e-6, 5000), r.normal(0, 3e4, 5000),
                         np.array([0.0, -0.0, 65504.0, 65519.9, 65520.0, 1e-8, 5.96e-8, 2.98e-8, 6.1e-5])]).astype(np.float32)
    golden.check("fp32_to_fp16", np.array([L.orc_fp32_to_fp16(float(x)) for x in xs], np.uint16),
                 lambda: np.array([oracle.ref_ggml().ref_fp32_to_fp16(float(x)) for x in xs], np.uint16))


@pytest.mark.parametrize("seed,scale", [(1, 0.02), (2, 1.0), (3, 50.0)])
def test_q4_0_quantize_dequantize(seed, scale):
    w = (_rng(seed).normal(0, scale, (64, 256))).astype(np.float32)
    w[3, :32] = 0.0  # all-zero block: d == 0 branch
    a = oracle.quantize_q4_0(w, "oracle")
    golden.check(f"q4_0[{seed}].quantize", a, lambda: oracle.quantize_q4_0(w, "ref"))
    golden.check(f"q4_0[{seed}].dequantize", oracle.dequantize_q4_0(a, 256, "oracle"), lambda: oracle.dequantize_q4_0(a, 256, "ref"))


@pytest.mark.parametrize("variant", ["runtime", "reference"])
def test_q8_0_quantize(variant):
    r = _rng(7)
    x = r.normal(0, 1.0, (32, 512)).astype(np.float32)
    x[0, :32] = 0.0
    x[1, :64] = np.round(x[1, :64] * 4) / 4  # plenty of exact .5 ties after scaling
    x[2, :32] = np.arange(32) - 15.5
    a = oracle.quantize_q8_0(x, "oracle", variant)
    golden.check(f"q8_0[{variant}].quantize", a, lambda: oracle.quantize_q8_0(x, "ref", variant))
    golden.check(f"q8_0[{variant}].dequantize", oracle.dequantize_q8_0(a, 512, "oracle"), lambda: oracle.dequantize_q8_0(a, 512, "ref"))


def test_vec_dot_and_mul_mat_bit_exact():
    r = _rng(11)
    N, K, M = 96, 1024, 5
    w = r.normal(0, 0.02, (N, K)).astype(np.float32)
    a = r.uniform(-0.5, 0.5, (M, K)).astype(np.float32)
    wq = oracle.quantize_q4_0(w)
    aq = oracle.quantize_q8_0(a)
    rows = range(0, N, 7)
    golden.check("q4_0_q8_0.vec_dot", np.array([oracle.vec_dot_q4_0_q8_0(wq[n], aq[0], K, "oracle") for n in rows], np.float32),
                 lambda: np.array([oracle.vec_dot_q4_0_q8_0(wq[n], aq[0], K, "ref") for n in rows], np.float32))
    c0 = oracle.mul_mat_q4_0_f32(wq, a, "oracle")
    golden.check("q4_0_q8_0.mul_mat", c0, lambda: oracle.mul_mat_q4_0_f32(wq, a, "ref"))
    # the scalar body only differs in fp32 summation order
    s = np.array([oracle.vec_dot_q4_0_q8_0(wq[n], aq[0], K, "oracle", scalar=True) for n in range(N)])
    np.testing.assert_allclose(s, c0[0], rtol=2e-4, atol=1e-5)


def test_btla_scalar_casts_and_bf16():
    L = oracle.lib()
    r = _rng(5)
    xs = np.concatenate([r.normal(0, 60, 4000), np.arange(-130, 131) + 0.5, np.arange(-130, 131) - 0.5,
                         [0.0, 254.5, 255.49, 300.0, -0.4]]).astype(np.float32)
    R = oracle.ref_btla
    for name, dt, scale in (("cast_f32_s8", np.int8, 1.0), ("cast_f32_u8", np.uint8, 1.0), ("cast_f32_s32", np.int32, 1.0),
                            ("f32_to_bf16", np.uint16, 1e-3)):
        mine = getattr(L, "orc_" + name)
        golden.check(f"btla.{name}", np.array([mine(float(x) * scale) for x in xs], dt),
                     lambda: np.array([getattr(R(), "ref_btla_" + name)(float(x) * scale) for x in xs], dt))
    golden.check("btla.nf4_unpack", np.array([L.orc_nf4_unpack(c) for c in range(16)], np.float32),
                 lambda: np.array([R().ref_btla_nf4_unpack(c) for c in range(16)], np.float32))
    lin = np.linspace(-1.1, 1.1, 4001).astype(np.float32)
    golden.check("btla.nf4_quantize", np.array([L.orc_nf4_quantize(float(x)) for x in lin], np.int8),
                 lambda: np.array([R().ref_btla_nf4_quantize(float(x)) for x in lin], np.int8))
    v = r.normal(0, 1, 1000).astype(np.float32)
    assert np.array_equal(oracle.f32_to_bf16_bits(v), np.array([L.orc_f32_to_bf16(float(t)) for t in v], np.uint16))


@pytest.mark.parametrize("nbits", [4, 8])
@pytest.mark.parametrize("asym", [False, True])
@pytest.mark.parametrize("g,K", [(32, 256), (128, 256), (128, 320), (256, 256)])
def test_btla_rtn_quantize(nbits, asym, g, K):
    r = _rng(100 + nbits + g + K)
    w = r.uniform(-0.5, 0.5, (K, 48)).astype(np.float32)  # bestla_ut.h fill convention
    w[:, 1] = np.abs(w[:, 1])          # one-sided column: exercises the NVal = -FullValue branch
    w[:, 2] = -np.abs(w[:, 2])
    got = oracle.btla_quantize(w, g, nbits, asym, "oracle")
    key = f"btla_rtn[{nbits}-{asym}-{g}-{K}]"
    for i, part in enumerate(("q", "sc", "zp") if asym else ("q", "sc")):
        golden.check(f"{key}.{part}", got[i], lambda: oracle.btla_quantize(w, g, nbits, asym, "ref")[i])


@pytest.mark.parametrize("g", [32, 128])
def test_btla_nf4_quantize(g):
    w = _rng(9).normal(0, 0.05, (256, 48)).astype(np.float32)
    got = oracle.btla_quantize_nf4(w, g, "oracle")
    for i, part in enumerate(("q", "sc")):
        golden.check(f"btla_nf4[{g}].{part}", got[i], lambda: oracle.btla_quantize_nf4(w, g, "ref")[i])


@pytest.mark.parametrize("g,K", [(32, 256), (128, 384), (128, 300)])
def test_btla_activation_quant(g, K):
    a = _rng(21).normal(0, 1, (4, K)).astype(np.float32)
    a[1] = np.abs(a[1])
    o = oracle.btla_quantize_act_u8(a, g, "oracle", want_reduce=True)
    for i, x in enumerate(o):
        golden.check(f"btla_act_u8[{g}-{K}].{i}", x, lambda: oracle.btla_quantize_act_u8(a, g, "ref", want_reduce=True)[i])
    o = oracle.btla_quantize_act_s8(a, g, "oracle")
    for i, x in enumerate(o):
        golden.check(f"btla_act_s8[{g}-{K}].{i}", x, lambda: oracle.btla_quantize_act_s8(a, g, "ref")[i])


# ----------------------------------------------------------------------------------------------- ggml Q6_K x Q8_K
def test_q6_K_block_sizes():
    golden.check("q6_K.block_sizes", np.array([oracle.Q6_K_BLOCK_BYTES, oracle.Q8_K_BLOCK_BYTES], np.int64),
                 lambda: np.array([oracle.ref_ggml().ref_sizeof_block_q6_K(), oracle.ref_ggml().ref_sizeof_block_q8_K()], np.int64))


@pytest.mark.parametrize("seed,scale", [(11, 0.02), (12, 1.0), (13, 40.0)])
def test_q6_K_quantisers_dequantiser_and_dot(seed, scale):
    r = _rng(seed)
    w = (r.normal(0, scale, (48, 1024))).astype(np.float32)
    w[3, :256] = 0.0          # all-zero super-block
    w[5, 16:32] = 0.0         # all-zero 16-group inside a live super-block (make_qx_quants early return)
    w[7, 300] = 1000 * scale  # outlier: exercises the clamp to [-32, 31]
    a = r.normal(0, 1.0, (3, 1024)).astype(np.float32)
    a[1, 256:512] = 0.0       # all-zero activation block: d == 0
    a[2, 7] = -a[2, 9]        # equal magnitudes, opposite signs: the first one decides the sign of `max`
    key = f"q6_K[{seed}]"
    wq = oracle.quantize_q6_K(w, "oracle")
    golden.check(f"{key}.quantize_q6_K", wq, lambda: oracle.quantize_q6_K(w, "ref"))
    aq = oracle.quantize_q8_K(a, "oracle")
    golden.check(f"{key}.quantize_q8_K", aq, lambda: oracle.quantize_q8_K(a, "ref"))
    golden.check(f"{key}.dequantize", oracle.dequantize_q6_K(wq, 1024, "oracle"), lambda: oracle.dequantize_q6_K(wq, 1024, "ref"))
    pairs = [(n, m) for n in range(0, 48, 5) for m in range(3)]
    golden.check(f"{key}.vec_dot", np.array([oracle.vec_dot_q6_K_q8_K(wq[n], aq[m], 1024, "oracle") for n, m in pairs], np.float32),
                 lambda: np.array([oracle.vec_dot_q6_K_q8_K(wq[n], aq[m], 1024, "ref") for n, m in pairs], np.float32))
    golden.check(f"{key}.mul_mat", oracle.mul_mat_q6_K_f32(wq, a, "oracle"), lambda: oracle.mul_mat_q6_K_f32(wq, a, "ref", nth=2))


def test_q6_K_random_bytes_dot():
    """Any byte pattern is a valid block_q6_K: the dot must agree on adversarial bit patterns too (fp16 d kept finite)."""
    r = _rng(21)
    k = 512
    wq = r.integers(0, 256, (16, k // 256 * 210), dtype=np.uint8)
    for b in range(k // 256):
        wq[:, b * 210 + 208:b * 210 + 210] = np.frombuffer(np.float16(r.uniform(-0.01, 0.01, 16)).tobytes(), np.uint8).reshape(16, 2)
    a = r.normal(0, 2.0, (2, k)).astype(np.float32)
    golden.check("q6_K_random.mul_mat", oracle.mul_mat_q6_K_f32(wq, a, "oracle"), lambda: oracle.mul_mat_q6_K_f32(wq, a, "ref", nth=1))
    golden.check("q6_K_random.dequantize", oracle.dequantize_q6_K(wq, k, "oracle"), lambda: oracle.dequantize_q6_K(wq, k, "ref"))


# ------------------------------------------------------------------------- element-wise ops of the Llama eval graph
# pinned against the reference's own graph engine (core/ne_layers.c through its public ne_* API, oracle/ref_ne.c)


def _vp(a):
    import ctypes as C
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("hd,theta,scale", [pytest.param(64, 10000.0, 1.0, id="64"), pytest.param(128, 10000.0, 1.0, id="128"),
                                            pytest.param(128, 500000.0, 1.0, id="128-theta5e5"),   # Llama-3
                                            pytest.param(128, 1e6, 1.0, id="128-theta1e6"),
                                            pytest.param(128, 10000.0, 4.0, id="128-scale4"),
                                            pytest.param(128, 500000.0, 4.0, id="128-theta5e5-scale4")])
def test_llama_rope_mode0_bit_exact(hd, theta, scale):
    """freq_base and freq_scale as hparams hold them (llama.cpp:243-244), at positions up to 4095"""
    from oracle import llama_model as lm
    r = _rng(31)
    default = (theta, scale) == (10000.0, 1.0)
    key = f"rope[{hd}]" if default else f"rope[{hd}-{theta:g}-{scale:g}]"

    def rope(x, n_tok, n_past):
        y = x.copy().reshape(n_tok, 3, hd)
        oracle.ref_ne().ref_ne_rope(_vp(y), hd, 3, n_tok, n_past, theta, scale)
        return y

    for pos in (0, 1, 7, 33, 127, 2047):
        x = r.normal(0, 1, (3, hd)).astype(np.float32)
        golden.check(f"{key}.pos{pos}", lm.rope_mode0(x, pos, hd, theta, scale), lambda: rope(x, 1, pos)[0])
    # several tokens in one call: position n_past + t
    x = r.normal(0, 1, (2, 3, hd)).astype(np.float32)
    golden.check(f"{key}.two_tokens", np.stack([lm.rope_mode0(x[t], 10 + t, hd, theta, scale) for t in range(2)]),
                 lambda: rope(x, 2, 10))
    # long contexts: theta_base *= theta_scale compounds its fp32 roundings, and sin / cos take arguments in the thousands
    for pos in (3071, 3998, 3999, 4095):
        x = r.normal(0, 1, (3, hd)).astype(np.float32)
        golden.check(f"{key}.pos{pos}", lm.rope_mode0(x, pos, hd, theta, scale), lambda: rope(x, 1, pos)[0])


def test_llama_softmax_and_rms_norm_bit_exact():
    from oracle import llama_model as lm
    r = _rng(32)
    def soft_max(s):
        y = s.copy()
        oracle.ref_ne().ref_ne_soft_max(_vp(y), s.shape[1], s.shape[0])
        return y

    def rms_norm(x, eps):
        y = np.zeros_like(x)
        oracle.ref_ne().ref_ne_rms_norm(_vp(x), _vp(y), x.shape[1], x.shape[0], eps)
        return y

    for n in (1, 5, 37, 300, 2048):
        s = r.normal(0, 3, (2, n)).astype(np.float32)
        golden.check(f"soft_max[{n}]", np.stack([lm.soft_max_f16table(row) for row in s]), lambda: soft_max(s))
    for n, eps in ((256, 1e-5), (4096, 1e-6)):
        x = r.normal(0, 2, (3, n)).astype(np.float32)
        golden.check(f"rms_norm[{n}]", lm.rms_norm(x, eps), lambda: rms_norm(x, eps))


@pytest.mark.parametrize("n_head,hd,length", [(4, 64, 23), (2, 128, 40), (4, 64, 1), (3, 96, 77), (2, 128, 300)])
def test_llama_single_token_attention_bit_exact(n_head, hd, length):
    """K.Q (fp16 K, Q rounded to fp16, SIMD ne_vec_dot_f16) -> scale -> soft_max -> V.P of llama.cpp:286-302"""
    from oracle import llama_model as lm
    r = _rng(33 + length)
    q = r.normal(0, 1, (n_head, hd)).astype(np.float32)
    kc = r.normal(0, 1, (n_head, length, hd)).astype(np.float16)
    vc = r.normal(0, 1, (n_head, length, hd)).astype(np.float16)
    vt = np.ascontiguousarray(vc.transpose(0, 2, 1))      # the reference's V cache is [head][hd][n_ctx]
    scale = float(np.float32(1.0) / np.float32(np.sqrt(np.float32(hd))))

    def attn():
        want = np.zeros((n_head, hd), np.float32)
        oracle.ref_ne().ref_ne_attn_1tok(_vp(q), _vp(kc), _vp(vt), _vp(want), hd, n_head, length, scale)
        return want

    got = np.zeros((n_head, hd), np.float32)
    for h in range(n_head):
        s = lm.vec_dot_f16_rows(kc[h].astype(np.float32), lm._f16(q[h])) * np.float32(scale)
        p = lm.soft_max_f16table(s)
        got[h] = lm.vec_dot_f16_rows(np.ascontiguousarray(vc[h].astype(np.float32).T), lm._f16(p))
    golden.check(f"attn_1tok[{n_head}-{hd}-{length}]", got, attn)


def _tiny_llama(seed, n_head=4, n_layer=2, n_head_kv=None):
    r = _rng(seed)
    n_head_kv = n_head_kv or n_head
    hp = dict(n_vocab=160, n_embd=256, n_head=n_head, n_head_kv=n_head_kv, n_layer=n_layer, n_ff=384, n_ctx=40, norm_eps=1e-5,
              rope_theta=10000.0, rope_scale=1.0)
    E, FF, V = hp["n_embd"], hp["n_ff"], hp["n_vocab"]
    kvd = E // n_head * n_head_kv
    w = lambda n, k: oracle.quantize_q4_0(r.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32))
    tok = r.normal(0, 1, (V, E)).astype(np.float32)
    on = r.uniform(0.5, 1.5, E).astype(np.float32)
    layers = [dict(attn_norm=r.uniform(0.5, 1.5, E).astype(np.float32), ffn_norm=r.uniform(0.5, 1.5, E).astype(np.float32),
                   wq=w(E, E), wk=w(kvd, E), wv=w(kvd, E), wo=w(E, E), w1=w(FF, E), w2=w(E, FF), w3=w(FF, E)) for _ in range(n_layer)]
    return hp, tok, on, w(V, E), layers


@pytest.mark.parametrize("n_head,n_head_kv", [(4, 4), (2, 2), (4, 2), (8, 2)])
def test_llama_eval_graph_end_to_end_bit_exact(n_head, n_head_kv):
    """oracle/llama_model.py == the reference's own engine running the graph of models/llama/llama.cpp (Q4_0 weights, fp16 KV
    cache, GQA through ne_mul_mat's head broadcast, prompt evals with the causal mask and single-token steps): logits bit for
    bit, hence identical greedy ids"""
    from oracle.llama_model import OracleLlama, greedy
    hp, tok, on, out, layers = _tiny_llama(50 + n_head, n_head, n_head_kv=n_head_kv)
    ref = oracle.RefNeLlama(hp, tok, on, out, layers) if golden.recording() else None
    orc = OracleLlama(hp, tok, on, out, layers)
    pos = 0
    for toks in ([1], [17], [150, 5, 9, 33], [44], [2, 3]):
        a = orc.eval(toks, pos)
        b = golden.value(f"llama_eval[{n_head}-{n_head_kv}].pos{pos}", lambda: ref.eval(toks, pos))
        assert np.array_equal(a, b), (toks, pos, float(np.abs(a - b).max()))
        assert greedy(a) == int(np.flatnonzero(b == b.max())[0])
        pos += len(toks)
    if ref is not None:
        ref.close()
