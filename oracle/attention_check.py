"""Float64 attention and its deliberate mutants -- TEST INFRASTRUCTURE ONLY.

tests/test_gpu_attention.py holds the engine's attention output for one (query row, head) to the reference's order of operations
(oracle.llama_model.attention) and to exact float64 softmax attention on the same fp16 operands (``exact``).  A bar is only
worth something if a plausible bug misses it, so ``mutants`` computes, in float64, what the kernels would return with one such
bug each; the tests require every mutant to miss the reference-order bar by a wide margin on their data.
tests/test_attention_numerics_cpu.py checks the bars and the margins on ``synthetic`` data before any GPU run.
"""
import numpy as np

from oracle.llama_model import rope_mode0

SPLIT_KEYS = 256  # context range of one CTA of the split decode kernel (llama.cu kSplitKeys)

# Bars on |kernel - reference| / max|V of the head's live rows|.  REF_ORDER_MAX is the kernels' stated deviation from the
# reference's soft_max order (DESIGN.md section 4): normalising after the V product instead of rounding p to fp16 first.
REF_ORDER_MAX = 1e-3
EXACT_MAX = 2e-3     # against exact float64 softmax attention on the same fp16 operands
# rms bar: 2 x the largest rms (3.0e-5) of the numpy model of that deviation (tests/test_attention_numerics_cpu.py kernel_order)
# over the data kinds of the GPU cases
REF_ORDER_RMS = 6e-5


def f16(x):
    return np.asarray(x, np.float32).astype(np.float16).astype(np.float32)


def exact(k, v, q, scale):
    """softmax(K q * scale) V in float64; k, v [len, hd] and q [hd] hold fp16 values"""
    s = np.asarray(k, np.float64) @ np.asarray(q, np.float64) * float(scale)
    p = np.exp(s - s.max())
    return (p / p.sum()) @ np.asarray(v, np.float64)


def rope_neox(x, pos, hd, theta=10000.0, rope_scale=1.0):
    """RoPE with the NeoX pairing (i, i + hd/2), float64: the wrong convention for a Llama graph"""
    x = np.asarray(x, np.float64)
    i = np.arange(hd // 2)
    ang = pos / float(rope_scale) * float(theta) ** (-2.0 * i / hd)
    c, s = np.cos(ang), np.sin(ang)
    a, b = x[..., :hd // 2], x[..., hd // 2:]
    return np.concatenate([a * c - b * s, a * s + b * c], axis=-1)


def merge_without_rescale(k, v, q, scale):
    """the split decode kernel's range merge with the exp(max_s - max) weights left out (one range per SPLIT_KEYS keys)"""
    s = np.asarray(k, np.float64) @ np.asarray(q, np.float64) * float(scale)
    v = np.asarray(v, np.float64)
    num, den = 0.0, 0.0
    for i0 in range(0, len(s), SPLIT_KEYS):
        e = np.exp(s[i0:i0 + SPLIT_KEYS] - s[i0:i0 + SPLIT_KEYS].max())
        num, den = num + e @ v[i0:i0 + SPLIT_KEYS], den + e.sum()
    return num / den


def mutants(kc, vc, q_raw, q_rot, pos, h, group, scale, theta, rope_scale, split=False, q_free=True):
    """{name: float64 output} for the query of head h at position pos with one plausible bug each.

    kc, vc [n_head_kv, n_ctx, hd]: the whole fp16 cache as the engine left it (rows past the live ones included: the past-the-edge
    mutant reads whatever lies there, as a kernel with that bug would); q_raw [hd]: this head's q before RoPE, q_rot [hd]: after.
    q_free = False leaves out the mutants that only move q or the score maxima (a zero q, with all scores equal, is immune to
    them)."""
    n_head_kv, n_ctx, hd = kc.shape
    hk = h // group
    q_rot = f16(q_rot)
    k, v = kc[hk].astype(np.float32), vc[hk].astype(np.float32)
    out = {}
    if pos >= 1:
        out["newest key dropped"] = exact(k[:pos], v[:pos], q_rot, scale)
    if pos + 1 < n_ctx:
        out["key past the causal edge"] = exact(k[:pos + 2], v[:pos + 2], q_rot, scale)
    if group > 1 and n_head_kv > 1:  # (with one kv head both mappings agree)
        hw = h % n_head_kv
        out["kv head h % n_head_kv"] = exact(kc[hw, :pos + 1].astype(np.float32), vc[hw, :pos + 1].astype(np.float32), q_rot, scale)
    if q_free:
        q_next = f16(rope_mode0(np.asarray(q_raw)[None], pos + 1, hd, theta, rope_scale)[0])
        out["q rotated at pos + 1"] = exact(k[:pos + 1], v[:pos + 1], q_next, scale)
        out["q with NeoX pairing"] = exact(k[:pos + 1], v[:pos + 1], f16(rope_neox(q_raw, pos, hd, theta, rope_scale)), scale)
    if q_free and split and pos + 1 > SPLIT_KEYS:
        out["range merge without rescale"] = merge_without_rescale(k[:pos + 1], v[:pos + 1], q_rot, scale)
    return out


def synthetic(rng, n_head, n_head_kv, hd, length, norm_scale=1.0, zero_q=False):
    """Operands with the statistics of the toy engines of tests/test_gpu_attention.py: their q, k and v are W x with x an
    RMS-normalised embedding row times attention-norm weights U(0.5, 1.5) * norm_scale and W ~ N(0, 1/n_embd), i.e. elements
    ~ N(0, 1.083 * norm_scale^2).  Returns (q_raw [length, n_head, hd] fp32, kc, vc [n_head_kv, length, hd] fp16) with K already
    rotated at its position, as the cache holds it."""
    sd = np.sqrt(1.083) * norm_scale
    q = (np.zeros if zero_q else lambda s: rng.normal(0, sd, s))((length, n_head, hd)).astype(np.float32)
    k = rng.normal(0, sd, (length, n_head_kv, hd)).astype(np.float32)
    kc = np.stack([rope_mode0(k[p], p, hd) for p in range(length)], 1).astype(np.float16)
    vc = rng.normal(0, sd, (n_head_kv, length, hd)).astype(np.float16)
    return q, kc, vc
