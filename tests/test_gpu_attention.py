"""The attention half of the eval step -- RoPE, the fp16 KV append and every attention kernel of llama.cu -- held directly to the
reference's arithmetic, row by row, through the engine's tap (ns_llama_set_tap: a layer's q | k | v before RoPE and its attention
output) and its KV cache (ns_llama_kv_cache).

Per checked query row and head, with vmax = max|V| over the head's live rows:
  * KV append: V rows equal fp16(v) bit for bit; K rows equal fp16(rope_mode0(k)) (the pinned oracle RoPE) within one fp16 ulp and
    bit for bit on >= 99.9 % of elements (device sincosf against glibc's); rows past the live ones are still zero.
  * attention against the reference order (oracle.llama_model.attention on the GPU's own cache rows 0 .. pos and the tapped q
    rotated by rope_mode0): max error <= ac.REF_ORDER_MAX * vmax (1e-3, the stated deviation, DESIGN.md section 4) and rms over
    the case <= ac.REF_ORDER_RMS * vmax (6e-5: 2 x the 3.0e-5 the numpy kernel_order model of tests/test_attention_numerics_cpu.py
    shows on data of these engines' statistics);
  * against exact float64 softmax attention on the same fp16 operands: max error <= ac.EXACT_MAX * vmax (2e-3);
  * every deliberate bug of oracle.attention_check.mutants misses the reference-order bar by >= 4x on the case's data, so a case
    too flat to tell them apart fails by itself.

Which case runs which kernel (llama.cu enqueue_forward):
  attn_decode_kernel<64/128> (m == 1, split context)     test_decode_attention[split-*], test_large_context_short_sequence,
                                                        test_rope_parameters, test_softmax_edges, test_tap_leaves_the_logits_alone
  attn_fast_kernel<HD, true> (m == 1, NS_ATTN_OLD_DECODE) test_decode_attention[old-*]
  attn_fast_kernel<HD, false> + rope_kv_kernel (2..7)   test_prompt_attention[*-m2 / -m7], the 7-token prompts of the decode cases,
                                                        test_softmax_edges
  attn_mma_kernel<64/128> + rope_kv_kernel (m >= 8)     test_prompt_attention[*-m8 .. -m130], the long prompts of every other case
  attn_kernel + rope_kv_kernel (other head sizes / NS_ATTN_SCALAR)  test_generic_head_sizes, test_prompt_attention[scalar-*]
"""
import numpy as np
import pytest
import torch

import neural_speed_b200 as ns
import oracle
from oracle import attention_check as ac
from oracle.llama_model import attention as ref_attention
from oracle.llama_model import rope_mode0

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    ns.lib().bestla_init()
    yield


def _build(hd, n_head, n_head_kv, n_ctx, fmt="q4_0", seed=0, n_layer=1, norm_scale=1.0, zero_wq=False, theta=10000.0, rope_scale=1.0):
    """a toy Llama with head size hd; attention-norm weights U(0.5, 1.5) * norm_scale (the data of ac.synthetic)"""
    rng = np.random.default_rng(seed)
    E, kvd, FF, V = n_head * hd, n_head_kv * hd, 512, 320
    hp = dict(n_vocab=V, n_embd=E, n_head=n_head, n_head_kv=n_head_kv, n_layer=n_layer, n_ff=FF, n_ctx=n_ctx, norm_eps=1e-5,
              rope_theta=theta, rope_scale=rope_scale)

    def weight(n, k, zero=False):
        w = np.zeros((n, k), np.float32) if zero else rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32)
        if fmt == "q4_0":
            return ns.Weight.from_q4_0_host(oracle.quantize_q4_0(w), n, k)
        return ns.Weight.from_blob(ns.np_bestla_quantize(w, "int4", 32, "sym", "fp32", "fp32"))  # fp32 compute

    eng = ns.Llama(**hp)
    eng.set_f32(ns.Llama.TOK_EMBD, 0, rng.normal(0, 1, (V, E)).astype(np.float32))
    eng.set_f32(ns.Llama.OUT_NORM, 0, rng.uniform(0.5, 1.5, E).astype(np.float32))
    eng.set_weight(ns.Llama.OUTPUT, 0, weight(V, E))
    for il in range(n_layer):
        eng.set_f32(ns.Llama.ATTN_NORM, il, (rng.uniform(0.5, 1.5, E) * norm_scale).astype(np.float32))
        eng.set_f32(ns.Llama.FFN_NORM, il, rng.uniform(0.5, 1.5, E).astype(np.float32))
        eng.set_weight(ns.Llama.WQ, il, weight(E, E, zero_wq))
        for tid, (n, k) in ((ns.Llama.WK, (kvd, E)), (ns.Llama.WV, (kvd, E)), (ns.Llama.WO, (E, E)), (ns.Llama.W1, (FF, E)),
                            (ns.Llama.W2, (E, FF)), (ns.Llama.W3, (FF, E))):
            eng.set_weight(tid, il, weight(n, k))
    return hp, eng


def _ulps(a, b):
    """distance in fp16 ulps between two fp16 arrays (+0 and -0 alike)"""
    def ordered(x):
        u = x.view(np.uint16).astype(np.int32)
        return np.where(u & 0x8000, -(u & 0x7FFF), u & 0x7FFF)
    return np.abs(ordered(a) - ordered(b))


def _sample(m, n_past):
    """query rows of an eval to check: all of a short one; else its ends, the 64-row q-tile and 64-key tile edges, the 256-key
    range edges it crosses, and a few more"""
    if m <= 16:
        return list(range(m))
    rows = {0, 1, m // 2, m - 2, m - 1} | {r for r in (15, 16, 62, 63, 64, 65, 127, 128) if r < m}
    rows |= {p - n_past + d for p in range(256, n_past + m, 256) for d in (-1, 0, 1) if 0 <= p - n_past + d < m}
    rows |= set(np.random.default_rng(m * 7919 + n_past).integers(0, m, 3).tolist())
    return sorted(rows)


class Checker:
    """follows one engine through a sequence of evals with a tap on `layer` and checks each against the references"""

    def __init__(self, hp, eng, layer=0, split=False, q_free=True, max_rows=1):
        self.hp, self.eng, self.layer, self.split, self.q_free = hp, eng, layer, split, q_free
        H, HK, n_ctx = hp["n_head"], hp["n_head_kv"], hp["n_ctx"]
        self.hd = hp["n_embd"] // H
        self.group = H // HK
        self.scale = np.float32(1.0) / np.float32(np.sqrt(np.float32(self.hd)))
        self.vexp = np.zeros((HK, n_ctx, self.hd), np.float16)
        self.vknown = np.zeros(n_ctx, bool)   # rows written by a tapped step (a generate call taps only its last)
        self.live = 0
        self.worst_ref = self.worst_exact = 0.0
        self.sq, self.cnt, self.rows = 0.0, 0, 0
        self.k_equal = self.k_total = self.k_ulps = 0
        self.mut = {}
        eng.set_tap(layer, max_rows)

    def _theta(self):
        return self.hp["rope_theta"], self.hp["rope_scale"]

    def eval(self, tokens, n_past):
        self.eng.eval(tokens, n_past)
        self.check(len(tokens), n_past, n_past + len(tokens))

    def generate(self, first, n_past, n_new):
        self.eng.generate(first, n_past, n_new)
        self.vknown[n_past:n_past + n_new - 1] = False  # written by untapped steps
        self.check(1, n_past + n_new - 1, n_past + n_new)

    def check(self, m, n_past, end):
        hp, hd, HK, H = self.hp, self.hd, self.hp["n_head_kv"], self.hp["n_head"]
        q, k, v, attn = (t.cpu().numpy() for t in self.eng.tap(m))
        kc, vc = (t.cpu().numpy() for t in self.eng.kv_cache(self.layer))
        rows = _sample(m, n_past)
        # ---- KV append
        self.vexp[:, n_past:n_past + m] = v.reshape(m, HK, hd).transpose(1, 0, 2).astype(np.float16)
        self.vknown[n_past:n_past + m] = True
        self.live = max(self.live, end)
        vk = self.vknown[:self.live]
        assert np.array_equal(vc[:, :self.live][:, vk].view(np.uint16), self.vexp[:, :self.live][:, vk].view(np.uint16)), "V cache"
        assert not vc[:, self.live:].view(np.uint16).any() and not kc[:, self.live:].view(np.uint16).any(), "stray cache writes"
        kexp = np.stack([rope_mode0(k[t].reshape(HK, hd), n_past + t, hd, *self._theta()) for t in rows], 1).astype(np.float16)
        ul = _ulps(kc[:, [n_past + t for t in rows]], kexp)
        assert ul.max() <= 1, ("K cache", int(ul.max()))
        self.k_equal += int((ul == 0).sum())
        self.k_total += ul.size
        self.k_ulps = max(self.k_ulps, int(ul.max()))
        # ---- attention, row by row
        for t in rows:
            pos = n_past + t
            q_raw = q[t].reshape(H, hd)
            q_rot = rope_mode0(q_raw, pos, hd, *self._theta())
            for h in range(H):
                hk = h // self.group
                kk, vv = kc[hk, :pos + 1].astype(np.float32), vc[hk, :pos + 1].astype(np.float32)
                vmax = max(float(np.abs(vv).max()), 1e-30)
                got = attn[t, h * hd:(h + 1) * hd]
                ref = ref_attention(kk, vv, q_rot[h], self.scale)
                d = (got - ref) / vmax
                self.worst_ref = max(self.worst_ref, float(np.abs(d).max()))
                self.sq, self.cnt = self.sq + float((d.astype(np.float64) ** 2).sum()), self.cnt + d.size
                ex = ac.exact(kk, vv, ac.f16(q_rot[h]), self.scale)
                self.worst_exact = max(self.worst_exact, float(np.abs(got - ex).max()) / vmax)
                for name, out in ac.mutants(kc, vc, q_raw[h], q_rot[h], pos, h, self.group, self.scale, *self._theta(), split=self.split,
                                            q_free=self.q_free).items():
                    self.mut[name] = max(self.mut.get(name, 0.0), float(np.abs(out - ref).max()) / vmax)
            self.rows += 1

    def finish(self, label):
        rms = (self.sq / max(self.cnt, 1)) ** 0.5
        frac = self.k_equal / max(self.k_total, 1)
        print(f"{label}: {self.rows} rows; vs reference order max {self.worst_ref:.2e} rms {rms:.2e}, vs float64 max "
              f"{self.worst_exact:.2e} (of vmax); K cache bit-identical {frac:.5f} (max {self.k_ulps} ulp); weakest mutant "
              + (f"{min(self.mut.values()):.2e} ({min(self.mut, key=self.mut.get)})" if self.mut else "none"))
        self.eng.set_tap(-1)
        self.eng.close()
        assert self.worst_ref <= ac.REF_ORDER_MAX, self.worst_ref
        assert rms <= ac.REF_ORDER_RMS, rms
        assert self.worst_exact <= ac.EXACT_MAX, self.worst_exact
        assert frac >= 0.999, frac
        expect = {"newest key dropped", "key past the causal edge"} | ({"kv head h % n_head_kv"} if 1 < self.group < self.hp["n_head"] else set())
        if self.q_free:
            expect |= {"q rotated at pos + 1", "q with NeoX pairing"} | ({"range merge without rescale"} if self.split else set())
        assert set(self.mut) == expect, sorted(self.mut)
        for name, err in self.mut.items():
            assert err >= 4 * ac.REF_ORDER_MAX, (name, err)


def _tokens(rng, n):
    return [int(t) for t in rng.integers(3, 320, n)]


@pytest.mark.parametrize("hd", [64, 128])
@pytest.mark.parametrize("n_head,n_head_kv", [(8, 8), (8, 4), (8, 2), (8, 1)])
@pytest.mark.parametrize("kernel", ["split", "old"])
def test_decode_attention(kernel, n_head, n_head_kv, hd, monkeypatch):
    """single-token evals at 0, 1, 255, 256, 257, 511, 512, 513, 767, 768 and 776 = n_ctx - 1 (n_ctx = 777: the last of the four
    256-key ranges is ragged; at 256 and 768 a range holds only the new token), the gaps filled by prompts (checked too), and two
    consecutive generate calls whose last steps sit in two and three ranges (the per-head merge ticket must be back at zero
    after each graph replay)"""
    if kernel == "old":
        monkeypatch.setenv("NS_ATTN_OLD_DECODE", "1")
    hp, eng = _build(hd, n_head, n_head_kv, 777, seed=hd + n_head_kv)
    c = Checker(hp, eng, split=kernel == "split", max_rows=253)
    rng = np.random.default_rng(n_head_kv)
    for pos in (0, 1):
        c.eval(_tokens(rng, 1), pos)
    c.eval(_tokens(rng, 253), 2)                  # 2 .. 254
    for pos in (255, 256, 257):
        c.eval(_tokens(rng, 1), pos)
    c.eval(_tokens(rng, 247), 258)                # 258 .. 504
    c.generate(_tokens(rng, 1)[0], 505, 6)        # 505 .. 510
    c.generate(_tokens(rng, 1)[0], 511, 3)        # 511 .. 513
    for pos in (511, 512, 513):                   # the same positions again, now each one tapped
        c.eval(_tokens(rng, 1), pos)
    c.eval(_tokens(rng, 253), 514)                # 514 .. 766
    for pos in (767, 768):
        c.eval(_tokens(rng, 1), pos)
    c.eval(_tokens(rng, 7), 769)                  # 769 .. 775
    c.eval(_tokens(rng, 1), 776)
    c.finish(f"decode {kernel} hd {hd} heads {n_head}/{n_head_kv}")


def test_large_context_short_sequence():
    """n_ctx 32768 (the gguf loader's default): 128 split CTAs per head, all but a few of which return at once"""
    hp, eng = _build(128, 8, 2, 32768, seed=3)
    c = Checker(hp, eng, split=True, max_rows=699)
    rng = np.random.default_rng(3)
    c.eval(_tokens(rng, 1), 0)
    c.eval(_tokens(rng, 1), 1)
    c.eval(_tokens(rng, 298), 2)                  # 2 .. 299
    c.eval(_tokens(rng, 1), 300)
    c.eval(_tokens(rng, 699), 301)                # 301 .. 999
    c.eval(_tokens(rng, 1), 1000)
    c.finish("n_ctx 32768")


PROMPTS = [pytest.param(hd, h, hk, m, False, id=f"hd{hd}-{h}x{hk}-m{m}") for hd in (64, 128) for h, hk in ((8, 8), (8, 2))
           for m in (2, 7, 8, 63, 64, 65, 130)] + [pytest.param(128, 8, 2, 65, True, id="scalar-hd128-8x2-m65"),
                                                   pytest.param(64, 8, 8, 130, True, id="scalar-hd64-8x8-m130")]


@pytest.mark.parametrize("hd,n_head,n_head_kv,m,scalar", PROMPTS)
def test_prompt_attention(hd, n_head, n_head_kv, m, scalar, monkeypatch):
    """m new tokens at n_past 0, 1, 37, 64 and 255, the last chunk ending exactly at n_ctx = 255 + m; m <= 7 runs attn_fast_kernel,
    m >= 8 attn_mma_kernel (64-row q tiles, 64-key tiles, causal mask), NS_ATTN_SCALAR the generic attn_kernel.  BesTLA weights
    with fp32 compute feed the tap"""
    if scalar:
        monkeypatch.setenv("NS_ATTN_SCALAR", "1")
    hp, eng = _build(hd, n_head, n_head_kv, 255 + m, fmt="btla", seed=m + hd)
    c = Checker(hp, eng, max_rows=255)
    rng = np.random.default_rng(m)
    for n_past in (0, 1, 37, 64, 255):
        if c.live < n_past:
            c.eval(_tokens(rng, n_past - c.live), c.live)
        c.eval(_tokens(rng, m), n_past)
    c.finish(f"prompt hd {hd} heads {n_head}/{n_head_kv} m {m}{' scalar' if scalar else ''}")


@pytest.mark.parametrize("hd", [32, 80, 96, 256])
@pytest.mark.parametrize("group", [1, 2])
def test_generic_head_sizes(hd, group):
    """head sizes without a specialised kernel run attn_kernel at every m (1, 5, 40), across the 256 boundary; a second layer
    (tapped) checks the per-layer cache offsets"""
    hp, eng = _build(hd, 8, 8 // group, 320, fmt="q4_0" if group == 1 else "btla", seed=hd, n_layer=2)
    c = Checker(hp, eng, layer=1, max_rows=210)
    rng = np.random.default_rng(hd)
    c.eval(_tokens(rng, 40), 0)                   # 0 .. 39
    c.eval(_tokens(rng, 1), 40)
    c.eval(_tokens(rng, 5), 41)                   # 41 .. 45
    c.eval(_tokens(rng, 205), 46)                 # 46 .. 250
    c.eval(_tokens(rng, 5), 251)                  # 251 .. 255
    c.eval(_tokens(rng, 1), 256)
    c.eval(_tokens(rng, 40), 257)                 # 257 .. 296
    c.eval(_tokens(rng, 1), 297)
    c.finish(f"generic hd {hd} group {group}")


@pytest.mark.parametrize("theta,rope_scale", [(500000.0, 1.0), (1e6, 1.0), (500000.0, 4.0)])
def test_rope_parameters(theta, rope_scale):
    """Llama-3's rope_theta and a linear rope_scale, positions up to n_ctx - 1 = 4095 (sin / cos of large arguments; theta_base
    *= theta_scale compounds over 64 pairs); K checked at sampled positions, always the last"""
    hp, eng = _build(128, 8, 2, 4096, seed=int(theta) % 97, theta=theta, rope_scale=rope_scale)
    c = Checker(hp, eng, split=True, max_rows=2095)
    rng = np.random.default_rng(5)
    c.eval(_tokens(rng, 2000), 0)
    c.eval(_tokens(rng, 2095), 2000)              # 2000 .. 4094
    c.eval(_tokens(rng, 1), 4095)
    c.finish(f"rope theta {theta:g} scale {rope_scale:g}")


@pytest.mark.parametrize("edge", ["peaked", "flat"])
def test_softmax_edges(edge):
    """peaked: attention-norm weights x8, scores span tens of units and most fp16 exps underflow to 0; flat: Wq = 0, so q = 0
    and p is uniform (the kernels' single division against the reference's fp16(1 / sum)); mma prompt, attn_fast prompt and
    split decode over one and two ranges"""
    hp, eng = _build(128, 8, 2, 320, seed=9, norm_scale=8.0 if edge == "peaked" else 1.0, zero_wq=edge == "flat")
    c = Checker(hp, eng, split=True, q_free=edge != "flat", max_rows=223)
    rng = np.random.default_rng(9)
    c.eval(_tokens(rng, 70), 0)
    c.eval(_tokens(rng, 1), 70)
    c.eval(_tokens(rng, 1), 71)
    c.eval(_tokens(rng, 5), 72)                   # 72 .. 76
    c.eval(_tokens(rng, 223), 77)                 # 77 .. 299
    c.eval(_tokens(rng, 1), 300)
    c.finish(f"softmax {edge}")


@pytest.mark.parametrize("hd,n_head_kv,fmt", [(64, 2, "q4_0"), (128, 8, "q4_0"), (128, 2, "btla")])
def test_tap_leaves_the_logits_alone(hd, n_head_kv, fmt):
    """logits with a tap equal those of an untapped engine with the same weights, bit for bit, through prompts, single-token
    evals (the one-token graph, recaptured with the copies) and generate; an eval longer than the tap fails clearly; removing the
    tap restores the untapped graph.  (Prompts stay at <= 16 tokens: longer ones may take the split-k tcgen05 GEMM, whose
    atomic sums are not bit-reproducible between two engines.)"""
    hp, a = _build(hd, 8, n_head_kv, 64, fmt=fmt, seed=4)
    _, b = _build(hd, 8, n_head_kv, 64, fmt=fmt, seed=4)
    a.set_tap(0, 8)
    rng = np.random.default_rng(4)
    steps = [(_tokens(rng, 7), 0), (_tokens(rng, 1), 7), (_tokens(rng, 1), 8), (_tokens(rng, 8), 9), (_tokens(rng, 1), 17)]
    for toks, n_past in steps:
        la, ta = a.eval(toks, n_past)
        lb, tb = b.eval(toks, n_past)
        assert np.array_equal(la.view(np.uint32), lb.view(np.uint32)) and ta == tb, n_past
    assert list(a.generate(5, 18, 6)) == list(b.generate(5, 18, 6))
    with pytest.raises(RuntimeError, match="tap"):
        a.eval(_tokens(rng, 9), 24)
    a.set_tap(-1)
    toks = _tokens(rng, 9)
    la, lb = a.eval(toks, 24)[0], b.eval(toks, 24)[0]
    assert np.array_equal(la.view(np.uint32), lb.view(np.uint32))
    assert list(a.generate(3, 33, 4)) == list(b.generate(3, 33, 4))
    with pytest.raises(RuntimeError):
        a.kv_cache(hp["n_layer"])
    a.close()
    b.close()
