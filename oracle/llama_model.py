"""oracle/llama_model.py -- TEST INFRASTRUCTURE ONLY.  CPU restatement (numpy + the pinned C oracle for the matmuls) of
the reference's Llama eval graph, models/llama/llama.cpp:190-720, ggml (non-fused-attention) path:

  get_rows -> per layer [rms_norm * w (kernel_ref.h:2199-2225) -> Q/K/V matmuls -> rope mode 0 (ne_layers.c:9380-9396,
  theta_base *= theta_scale iteratively in fp32) -> fp16 KV cache -> K.Q with Q rounded to fp16
  (ne_compute_forward_mul_mat_f16_f32) -> scale -> causal mask -> soft_max with the fp16 exp table
  (ne_layers.c:8923-8945) -> V.P with P rounded to fp16 -> wo + residual -> rms_norm * w -> silu(w1 x) * (w3 x) -> w2 +
  residual] -> rms_norm * w -> output matmul.  Greedy pick: lowest index among maxima (model_utils.cpp:2963-2985).

Parity status: PINNED.  The matmuls are the pinned C oracle (bit-exact with oracle/_ref/libref_ggml.so); rope_mode0,
soft_max_f16table, rms_norm and the fp16 dot products are bit-exact with the reference's own graph engine (oracle/ref_ne.c compiles
core/ne_layers.c in place and drives it through the public ne_* API), and OracleLlama.eval reproduces, bit for bit, the logits that
engine computes for the graph of models/llama/llama.cpp (prompt evals with the causal mask and single-token steps, MHA and GQA)
-- tests/test_oracle_vs_ref.py, fixtures tests/golden/llama_ops.npz and llama_tiny.npz.  One stub sits under the
engine: bestla_layernormalization is served by the reference's portable kernel_ref.h body (its AVX2 / AVX-512 bodies need xbyak to
build; they vectorise the same sum).  The GPU engine is held to the north-star tolerance against
this oracle (1e-2 on logits, greedy ids equal wherever the top-2 margin exceeds that tolerance).
"""
import ctypes as C
import ctypes.util

import numpy as np

import oracle

# the reference calls glibc's float routines (powf / cosf / sinf, ne_layers.c:9216-9217,9300); numpy's float32 ufuncs may differ
# in the last bit, and a 1-ulp difference in theta_scale grows with the position
_libm = C.CDLL(ctypes.util.find_library("m") or "libm.so.6")
for _n in ("powf", "cosf", "sinf", "fmaf"):
    getattr(_libm, _n).restype = C.c_float
_libm.powf.argtypes = [C.c_float, C.c_float]
_libm.fmaf.argtypes = [C.c_float, C.c_float, C.c_float]
_libm.cosf.argtypes = [C.c_float]
_libm.sinf.argtypes = [C.c_float]


def _f16(x):
    return np.asarray(x, np.float32).astype(np.float16).astype(np.float32)


def rope_mode0(x, pos, hd, freq_base=10000.0, rope_scale=1.0):
    """ne_rope_inplace(mode 0) on x [n_head, hd] at position pos (ne_layers.c:9300, 9380-9396): theta_base = p, then
    theta_base *= theta_scale per pair (fp32); dst0 = x0*cos - x1*sin, dst1 = x0*sin + x1*cos.  The reference's default build
    (-O3 -mfma) contracts these to fma(x0, cos, -(x1*sin)) and fma(x0, sin, x1*cos); pinned bit-exact against the reference's
    own engine (oracle/_ref/libref_ne.so, tests/test_oracle_vs_ref.py)."""
    theta_scale = np.float32(_libm.powf(float(np.float32(freq_base)), float(np.float32(-2.0) / np.float32(hd))))
    freq_scale = np.float32(1.0) / np.float32(rope_scale)
    x = np.asarray(x, np.float32)
    out = x.copy()
    theta = np.float32(pos)
    for i0 in range(0, hd, 2):
        th = np.float32(freq_scale * theta)
        c, s = float(np.float32(_libm.cosf(float(th)))), float(np.float32(_libm.sinf(float(th))))
        theta = np.float32(theta * theta_scale)
        for h in range(x.shape[0]):
            x0, x1 = float(x[h, i0]), float(x[h, i0 + 1])
            out[h, i0] = _libm.fmaf(x0, c, -float(np.float32(np.float32(x1) * np.float32(s))))
            out[h, i0 + 1] = _libm.fmaf(x0, s, float(np.float32(np.float32(x1) * np.float32(c))))
    return out


def vec_dot_f16_rows(x, y):
    """ne_vec_dot_f16 (core/layers/vec_dot.h:94-129, NS_SIMD_VEC_DOT_F16 = ON, AVX2 + F16C) of every row of x [R, n] with y
    [n]; both already hold fp16-representable values.  Four 8-lane fp32 accumulators over chunks of 32 (element e -> accumulator
    (e % 32) / 8, lane e % 8, true fma), reduce x0+=x1, x2+=x3, x0+=x2, lane l + lane l+4, two hadds (simd.h:58-72), then the
    scalar tail in double.  A product of two fp16 values is exact in fp32, so fma(x, y, acc) = fp32(x*y + acc) computed in
    double reproduces it."""
    x = np.asarray(x, np.float32)
    y = np.asarray(y, np.float32)
    R, n = x.shape
    npk = n & ~31
    acc = np.zeros((R, 4, 8), np.float32)
    for i in range(0, npk, 32):
        xs = x[:, i:i + 32].reshape(R, 4, 8).astype(np.float64)
        ys = y[i:i + 32].reshape(1, 4, 8).astype(np.float64)
        acc = (xs * ys + acc.astype(np.float64)).astype(np.float32)
    a0 = (acc[:, 0] + acc[:, 1]).astype(np.float32)
    a2 = (acc[:, 2] + acc[:, 3]).astype(np.float32)
    a0 = (a0 + a2).astype(np.float32)
    t0 = (a0[:, :4] + a0[:, 4:]).astype(np.float32)
    t1 = np.stack([(t0[:, 0] + t0[:, 1]).astype(np.float32), (t0[:, 2] + t0[:, 3]).astype(np.float32)], 1)
    sumf = (t1[:, 0] + t1[:, 1]).astype(np.float32).astype(np.float64)
    for i in range(npk, n):
        sumf = sumf + (x[:, i] * y[i]).astype(np.float32).astype(np.float64)
    return sumf.astype(np.float32)


def soft_max_f16table(s):
    """ne_compute_forward_soft_max_f32 (ne_layers.c:8923-8945): exp through the fp16 table (argument and result rounded to
    fp16), sum in double, scale by (float)(1/sum)"""
    s = np.asarray(s, np.float32)
    e = _f16(np.exp(_f16(s - s.max()).astype(np.float64)))
    return (e * np.float32(1.0 / np.float64(e.astype(np.float64).sum()))).astype(np.float32)


def attention(k, v, q, scale):
    """One (token, head) of the ggml attention, llama.cpp:286-302: K.Q with Q rounded to fp16 (mul_mat(K fp16, Q)), times
    scale (ne_scale), soft_max through the fp16 exp table, then V.P with P rounded to fp16 (mul_mat(V fp16, P); the reference
    keeps V transposed).  k, v [len, hd] hold the fp16 cache rows 0 .. pos (the causal window), q [hd] is rotated."""
    s = vec_dot_f16_rows(np.asarray(k, np.float32), _f16(q)) * np.float32(scale)
    p = soft_max_f16table(s)
    vt = np.ascontiguousarray(np.asarray(v, np.float32).T)
    return vec_dot_f16_rows(vt, _f16(p))


def rms_norm(x, eps):
    """kernel_ref.h:2199-2225 (simplified layernorm without scale): sequential fp32 sum of squares, sqrt, reciprocal"""
    x = np.asarray(x, np.float32)
    out = np.empty_like(x)
    eps = np.float32(eps)
    for r in range(x.shape[0]):
        ms = np.float32(0)
        for v in x[r]:
            ms = np.float32(ms + np.float32(v * v))
        rms = np.float32(np.sqrt(np.float32(ms / np.float32(x.shape[1]) + eps)))
        out[r] = x[r] * (np.float32(1.0) / rms)
    return out


class OracleLlama:
    def __init__(self, hp: dict, tok_embd, out_norm, output_rows, layers, fmt="q4_0"):
        """layers: list of dicts with attn_norm, ffn_norm (f32 [E]) and wq, wk, wv, wo, w1, w2, w3 as Q4_0 row arrays
        (uint8 [N, K/32*18]); output_rows likewise (or Q6_K rows when fmt_out == 'q6_K')."""
        self.hp = dict(hp)
        self.tok_embd = np.asarray(tok_embd, np.float32)
        self.out_norm = np.asarray(out_norm, np.float32)
        self.output_rows = output_rows
        self.layers = layers
        self.out_fmt = fmt
        E, H, HK = hp["n_embd"], hp["n_head"], hp["n_head_kv"]
        self.hd = E // H
        self.kc = np.zeros((hp["n_layer"], HK, hp["n_ctx"], self.hd), np.float16)
        self.vc = np.zeros_like(self.kc)

    @staticmethod
    def _mm(rows, a):
        return oracle.mul_mat_q4_0_f32(rows, np.ascontiguousarray(a, np.float32))

    def _rms(self, x, w):
        return rms_norm(x, self.hp.get("norm_eps", 1e-6)) * w     # ne_rms_norm then ne_mul: (x * inv) * w

    def _rope(self, x, pos):
        return rope_mode0(x, pos, self.hd, self.hp.get("rope_theta", 10000.0), self.hp.get("rope_scale", 1.0))

    def eval(self, tokens, n_past):
        hp = self.hp
        E, H, HK, hd = hp["n_embd"], hp["n_head"], hp["n_head_kv"], self.hd
        n = len(tokens)
        x = self.tok_embd[np.asarray(tokens)].astype(np.float32)
        scale = np.float32(1.0) / np.float32(np.sqrt(np.float32(hd)))
        for il, L in enumerate(self.layers):
            cur = self._rms(x, L["attn_norm"])
            q = self._mm(L["wq"], cur).reshape(n, H, hd)
            k = self._mm(L["wk"], cur).reshape(n, HK, hd)
            v = self._mm(L["wv"], cur).reshape(n, HK, hd)
            attn = np.zeros((n, H, hd), np.float32)
            for t in range(n):
                pos = n_past + t
                q[t] = self._rope(q[t], pos)
                self.kc[il, :, pos, :] = self._rope(k[t], pos).astype(np.float16)
                self.vc[il, :, pos, :] = v[t].astype(np.float16)
            for t in range(n):
                ln = n_past + t + 1
                for h in range(H):
                    hk = h // (H // HK)
                    attn[t, h] = attention(self.kc[il, hk, :ln], self.vc[il, hk, :ln], q[t, h], scale)
            inp_ff = self._mm(L["wo"], attn.reshape(n, E)) + x
            cur = self._rms(inp_ff, L["ffn_norm"])
            g = self._mm(L["w1"], cur)
            silu = np.array([[oracle.lib().orc_silu(float(z)) for z in row] for row in g], np.float32)
            mid = silu * self._mm(L["w3"], cur)
            x = self._mm(L["w2"], mid) + inp_ff
        last = self._rms(x[-1:], self.out_norm)
        if self.out_fmt == "q6_K":
            return oracle.mul_mat_q6_K_f32(self.output_rows, last)[0]
        return self._mm(self.output_rows, last)[0]


def greedy(logits):
    return int(oracle.argmax(logits))
