"""The one stated deviation of the tensor-core prompt attention and of the split-context decode attention from the reference's
soft_max (DESIGN.md section 4): the reference rounds p = e / sum to fp16 BEFORE the V product (ne_compute_forward_soft_max_f32,
core/ne_layers.c:8887-8954, then mul_mat(V, P) with P converted to fp16, :6943-7083); the kernels accumulate sum e V with the exact
fp16 e and divide once at the end -- and, with several context ranges, merge per-range {max, sum e, sum e V} with exp(max_s - max)
weights.  This numpy model bounds what that costs.

It also sets and checks the bars of tests/test_gpu_attention.py, which holds the kernels' output directly to the reference order
(oracle.llama_model.attention), before any GPU run: the model stays inside them on data with the statistics of that file's
engines (oracle.attention_check.synthetic), and every deliberate bug of oracle.attention_check.mutants misses them by >= 4x."""
import numpy as np
import pytest

from oracle import attention_check as ac
from oracle import llama_model as lm


def f16(x):
    return np.asarray(x, np.float32).astype(np.float16).astype(np.float32)


def reference_order(s, v):
    mx = s.max()
    e = f16(np.exp(f16(s - mx)))
    p = f16(e * np.float32(1.0 / e.sum(dtype=np.float32)))
    return (p[:, None] * v).sum(axis=0, dtype=np.float32)


def kernel_order(s, v, ranges=1, keys=None):
    """ranges: that many equal ranges; keys: ranges of that many keys, as the split decode kernel cuts the context"""
    parts = []
    split = np.array_split(np.arange(len(s)), ranges) if keys is None else [np.arange(i, min(i + keys, len(s))) for i in range(0, len(s), keys)]
    for idx in split:
        mx = s[idx].max()
        e = f16(np.exp(f16(s[idx] - mx)))
        parts.append((mx, e.sum(dtype=np.float32), (e[:, None] * v[idx]).sum(axis=0, dtype=np.float32)))
    gm = max(p[0] for p in parts)
    num = sum(np.exp(np.float32(p[0] - gm)) * p[2] for p in parts)
    den = sum(np.exp(np.float32(p[0] - gm)) * p[1] for p in parts)
    return (num / den).astype(np.float32)


def test_normalising_after_the_v_product_stays_within_1e3_of_the_reference_order():
    rng = np.random.default_rng(0)
    worst = 0.0
    for length, hd, ranges in ((40, 64, 1), (300, 128, 1), (300, 128, 2), (2100, 128, 9)):
        for _ in range(4):
            s = rng.normal(0, 2.0, length).astype(np.float32)
            v = f16(rng.normal(0, 1.0, (length, hd)))
            a, b = reference_order(s, v), kernel_order(s, v, ranges)
            worst = max(worst, float(np.abs(a - b).max() / np.abs(a).max()))
    assert worst <= 1e-3, worst


def test_shared_oracle_attention_is_the_graph_attention_it_replaced():
    """oracle.llama_model.attention, which OracleLlama.eval and the GPU attention tests share, against the per-(token, head) body
    OracleLlama.eval had inline before, bit for bit (MHA and GQA, short and > 256-position windows)"""
    rng = np.random.default_rng(40)
    for H, HK, hd, ln in ((4, 4, 64, 1), (4, 2, 64, 37), (8, 2, 128, 300), (3, 3, 96, 77)):
        kc = rng.normal(0, 1, (HK, ln, hd)).astype(np.float16)
        vc = rng.normal(0, 1, (HK, ln, hd)).astype(np.float16)
        q = rng.normal(0, 1, (H, hd)).astype(np.float32)
        scale = np.float32(1.0) / np.float32(np.sqrt(np.float32(hd)))
        for h in range(H):
            hk = h // (H // HK)
            kk = kc[hk, :ln].astype(np.float32)
            s = lm.vec_dot_f16_rows(kk, lm._f16(q[h])) * scale
            p = lm.soft_max_f16table(s)
            vt = np.ascontiguousarray(vc[hk, :ln].astype(np.float32).T)
            old = lm.vec_dot_f16_rows(vt, lm._f16(p))
            new = lm.attention(kc[hk, :ln], vc[hk, :ln], q[h], scale)
            assert new.dtype == old.dtype and np.array_equal(new.view(np.uint32), old.view(np.uint32)), (H, HK, hd, ln, h)


# (hd, n_head, n_head_kv, context length, norm scale, zero q): the data kinds of tests/test_gpu_attention.py -- plain, peaked
# (attention-norm weights x8), flat (q = 0), and a long split context
DATA = [(64, 8, 2, 300, 1.0, False), (128, 8, 2, 777, 1.0, False), (128, 8, 8, 130, 1.0, False), (128, 8, 2, 300, 8.0, False),
        (64, 8, 4, 300, 1.0, True)]


@pytest.mark.parametrize("hd,H,HK,ln,norm,zero_q", DATA)
def test_kernel_order_meets_the_gpu_attention_bars(hd, H, HK, ln, norm, zero_q):
    """The kernels that normalise after the V product (mma prompt attention; split decode, with ranges of 256 keys merged) are
    the ones furthest from the reference order.  Their numpy model stays inside the max bars of tests/test_gpu_attention.py
    and, by ac.REF_ORDER_RMS's construction, at or under half its rms bar on the same kind of data."""
    rng = np.random.default_rng(hd + ln)
    q_raw, kc, vc = ac.synthetic(rng, H, HK, hd, ln, norm, zero_q)
    scale = np.float32(1.0) / np.float32(np.sqrt(np.float32(hd)))
    worst_ref = worst_exact = 0.0
    sq, cnt = 0.0, 0
    for pos in sorted({0, 1, 2, ln // 3, 255, 256, ln - 2, ln - 1} & set(range(ln))):
        q = lm.rope_mode0(q_raw[pos], pos, hd)
        for h in range(H):
            hk = h // (H // HK)
            k, v = kc[hk, :pos + 1].astype(np.float32), vc[hk, :pos + 1].astype(np.float32)
            vmax = float(np.abs(v).max())
            ref = lm.attention(k, v, q[h], scale)
            s = lm.vec_dot_f16_rows(k, lm._f16(q[h])) * scale
            got = kernel_order(s, v, keys=ac.SPLIT_KEYS)
            d = (got - ref) / vmax
            worst_ref = max(worst_ref, float(np.abs(d).max()))
            worst_exact = max(worst_exact, float(np.abs(got - ac.exact(k, v, lm._f16(q[h]), scale)).max()) / vmax)
            sq, cnt = sq + float((d.astype(np.float64) ** 2).sum()), cnt + d.size
    rms = (sq / cnt) ** 0.5
    print(f"kernel order vs reference order: max {worst_ref:.2e}, rms {rms:.2e} of vmax; vs exact float64 max {worst_exact:.2e}")
    assert worst_ref <= ac.REF_ORDER_MAX and worst_exact <= ac.EXACT_MAX
    assert rms <= ac.REF_ORDER_RMS / 2, rms


@pytest.mark.parametrize("hd,H,HK,ln,norm,zero_q", DATA)
def test_every_mutant_misses_the_reference_order_bar_by_4x(hd, H, HK, ln, norm, zero_q):
    """each deliberate bug of ac.mutants moves some checked row by >= 4 x ac.REF_ORDER_MAX (of that head's max|V|) on the same
    positions the GPU cases check; with q = 0 the q-rotation bugs change nothing and are left out"""
    rng = np.random.default_rng(hd + ln + 1)
    q_raw, kc, vc = ac.synthetic(rng, H, HK, hd, ln, norm, zero_q)
    scale = np.float32(1.0) / np.float32(np.sqrt(np.float32(hd)))
    worst = {}
    for pos in sorted({0, 1, 2, ln // 3, 255, 256, 257, ln - 2, ln - 1} & set(range(ln))):
        q = lm.rope_mode0(q_raw[pos], pos, hd)
        for h in range(H):
            hk = h // (H // HK)
            k, v = kc[hk, :pos + 1].astype(np.float32), vc[hk, :pos + 1].astype(np.float32)
            ref = lm.attention(k, v, q[h], scale)
            vmax = float(np.abs(v).max())
            for name, out in ac.mutants(kc, vc, q_raw[pos][h], q[h], pos, h, H // HK, scale, 10000.0, 1.0, split=True, q_free=not zero_q).items():
                worst[name] = max(worst.get(name, 0.0), float(np.abs(out - ref).max()) / vmax)
    print({k: f"{v:.2e}" for k, v in worst.items()})
    assert len(worst) == 2 + (HK < H) + (0 if zero_q else 2 + (ln > ac.SPLIT_KEYS))
    for name, err in worst.items():
        assert err >= 4 * ac.REF_ORDER_MAX, (name, err)
