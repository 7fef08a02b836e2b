"""Device-resident Llama eval step (SURVEY §8 f.1) against the CPU restatement of the reference graph (oracle/llama_model.py).
North-star bar: logits within 1e-2, greedy token ids equal (checked wherever the oracle's top-2 margin exceeds the tolerance)."""
import numpy as np
import pytest
import torch

import neural_speed_b200 as ns
import oracle
from oracle.llama_model import OracleLlama, greedy

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    ns.lib().bestla_init()
    yield


def _build(n_head_kv=4, out_fmt="q4_0", seed=0, n_layer=2, n_ctx=48, n_head=4, jig=0):
    rng = np.random.default_rng(seed)
    hp = dict(n_vocab=320, n_embd=256, n_head=n_head, n_head_kv=n_head_kv, n_layer=n_layer, n_ff=512, n_ctx=n_ctx, norm_eps=1e-5,
              rope_theta=10000.0, rope_scale=1.0)
    E, FF, V = hp["n_embd"], hp["n_ff"], hp["n_vocab"]
    kvd = E // hp["n_head"] * n_head_kv
    tok = rng.normal(0, 1, (V, E)).astype(np.float32)
    out_norm = rng.uniform(0.5, 1.5, E).astype(np.float32)

    def w(n, k):
        return rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32)

    shapes = dict(wq=(E, E), wk=(kvd, E), wv=(kvd, E), wo=(E, E), w1=(FF, E), w2=(E, FF), w3=(FF, E))
    layers = []
    for _ in range(n_layer):
        L = dict(attn_norm=rng.uniform(0.5, 1.5, E).astype(np.float32), ffn_norm=rng.uniform(0.5, 1.5, E).astype(np.float32))
        for name, (n, k) in shapes.items():
            L[name] = oracle.quantize_q4_0(w(n, k))
        layers.append(L)
    wout = w(V, E)
    out_rows = oracle.quantize_q6_K(wout) if out_fmt == "q6_K" else oracle.quantize_q4_0(wout)
    orc = OracleLlama(hp, tok, out_norm, out_rows, layers, fmt=out_fmt)
    if jig:  # the same CPU graph with every embedding value moved by +-jig ulp: measures the conditioning of the graph itself
        sgn = (np.random.default_rng(99).integers(0, 2, tok.shape) * 2 - 1).astype(np.int32)
        orc.jig = OracleLlama(hp, (tok.view(np.int32) + sgn * jig).view(np.float32), out_norm, out_rows, layers, fmt=out_fmt)
    eng = ns.Llama(**hp)
    eng.set_f32(ns.Llama.TOK_EMBD, 0, tok)
    eng.set_f32(ns.Llama.OUT_NORM, 0, out_norm)
    outw = ns.Weight.from_q6_K_host(out_rows, V, E) if out_fmt == "q6_K" else ns.Weight.from_q4_0_host(out_rows, V, E)
    eng.set_weight(ns.Llama.OUTPUT, 0, outw)
    ids = dict(wq=ns.Llama.WQ, wk=ns.Llama.WK, wv=ns.Llama.WV, wo=ns.Llama.WO, w1=ns.Llama.W1, w2=ns.Llama.W2, w3=ns.Llama.W3)
    for il, L in enumerate(layers):
        eng.set_f32(ns.Llama.ATTN_NORM, il, L["attn_norm"])
        eng.set_f32(ns.Llama.FFN_NORM, il, L["ffn_norm"])
        for name, (n, k) in shapes.items():
            eng.set_weight(ids[name], il, ns.Weight.from_q4_0_host(L[name], n, k))
    return hp, orc, eng


def _check_logits(got, want, tol=1e-2):
    scale = max(1.0, float(np.abs(want).max()))
    err = float(np.abs(got - want).max())
    assert err <= tol * scale, (err, scale)
    top = np.sort(want)[-2:]
    if top[1] - top[0] > 2 * tol * scale:        # unambiguous pick: ids must agree
        assert int(np.argmax(got)) == greedy(want)


@pytest.mark.parametrize("n_head,n_head_kv,out_fmt", [(4, 4, "q4_0"), (4, 2, "q4_0"), (4, 4, "q6_K"), (2, 2, "q4_0"), (2, 1, "q4_0"),
                                                       (8, 8, "q4_0")])
def test_token_by_token_decode_matches_the_cpu_graph(n_head, n_head_kv, out_fmt):
    """head sizes 64 and 128 take the fused rope + KV-append + attention kernel, 32 the generic one"""
    hp, orc, eng = _build(n_head_kv, out_fmt, seed=n_head_kv, n_head=n_head)
    toks = [1, 17, 300, 5, 123, 77, 9]
    for pos, t in enumerate(toks):
        want = orc.eval([t], pos)
        got, nxt = eng.eval([t], pos)
        _check_logits(got, want)
        assert nxt == int(np.argmax(got)) or got[nxt] == got.max()   # device argmax: lowest index among maxima
        assert nxt == int(np.flatnonzero(got == got.max())[0])
    eng.close()


def test_small_prompt_eval_then_decode():
    """a 3-token prompt in one eval (M <= 4: the exact-integer GEMV path), then two single-token steps"""
    hp, orc, eng = _build(seed=5)
    prompt = [1, 200, 31]
    _check_logits(eng.eval(prompt, 0)[0], orc.eval(prompt, 0))
    _check_logits(eng.eval([8], 3)[0], orc.eval([8], 3))
    _check_logits(eng.eval([250], 4)[0], orc.eval([250], 4))
    eng.close()


@pytest.mark.parametrize("n_head", [4, 2])
def test_long_prompt_goes_through_the_tensor_core_gemm(n_head):
    """M > 16 rows take the bf16 tcgen05 GEMM: same graph, bf16 matmul numerics (looser bar), KV cache usable afterwards"""
    hp, orc, eng = _build(n_head, seed=6, n_head=n_head)
    prompt = list(np.random.default_rng(1).integers(3, hp["n_vocab"], 24))
    _check_logits(eng.eval(prompt, 0)[0], orc.eval(prompt, 0), tol=4e-2)
    _check_logits(eng.eval([42], 24)[0], orc.eval([42], 24), tol=4e-2)
    eng.close()


def test_exact_prefill_mode_keeps_reference_numerics_for_long_prompts():
    """a 70-token prompt: default = bf16 tensor-core GEMM (looser bar); exact mode = pieces of 32 on the integer tensor cores,
    held to the north-star 1e-2, and the KV cache it leaves serves the following single-token steps"""
    hp, orc, eng = _build(seed=12, n_ctx=96, jig=64)
    prompt = [int(t) for t in np.random.default_rng(3).integers(3, hp["n_vocab"], 70)]
    want = orc.eval(prompt, 0)
    # 70 positions of Q8_0 rounding decisions: the CPU graph against itself with inputs moved by +-64 ulp differs by 1.6e-2 here
    # (+-4 ulp: 0.9e-2) -- the bar is the north star or 1.5 x that measured floor, whichever is larger (cf. the 7B-shape test)
    floor = float(np.abs(orc.jig.eval(prompt, 0) - want).max()) / max(1.0, float(np.abs(want).max()))
    tol = min(max(1e-2, 1.5 * floor), 2.5e-2)
    eng.set_exact_prefill(True)
    _check_logits(eng.eval(prompt, 0)[0], want, tol=tol)
    _check_logits(eng.eval([9], 70)[0], orc.eval([9], 70), tol=tol)
    eng.close()


def test_generate_feeds_the_argmax_on_device():
    hp, orc, eng = _build(seed=7)
    first, n_new = 11, 10
    out = eng.generate(first, 0, n_new)
    # the same steps through ns_llama_eval, one host round trip per token: identical kernels, identical picks
    hp2, _, eng2 = _build(seed=7)
    t, ref = first, []
    for pos in range(n_new):
        _, t = eng2.eval([t], pos, want_logits=False)
        ref.append(t)
    assert list(out) == ref
    # and against the CPU graph while the pick is unambiguous
    t = first
    for pos in range(n_new):
        want = orc.eval([t], pos)
        top = np.sort(want)[-2:]
        if top[1] - top[0] <= 2e-2 * max(1.0, float(np.abs(want).max())):
            break
        assert int(out[pos]) == greedy(want)
        t = int(out[pos])
    eng.close()
    eng2.close()


def test_argument_checks():
    hp, orc, eng = _build(seed=8, n_ctx=16)
    rc = ns.lib().ns_llama_eval(eng.h, np.zeros(20, np.int32).ctypes.data, 20, 0, None, None)
    assert rc != 0 and "n_ctx" in ns.last_error()
    eng2 = ns.Llama(**hp)
    with pytest.raises(RuntimeError):
        eng2.eval([1], 0)                      # no tensors set: refuses instead of reading null pointers
    eng.close()
    eng2.close()


def test_llama2_7b_shaped_greedy_decode_matches_the_reference_engine():
    """North-star parity at the model's real shapes: n_embd 4096, 32 heads of 128, n_ff 11008, vocab 32000, Q4_0 weights (two
    decoder layers + the full output head keep the CPU side to a few minutes).  A 12-token prompt evaluated token by token, then
    16 greedy steps against the REFERENCE's own graph engine (oracle.RefNeLlama = core/ne_layers.c compiled where it lies; the
    numpy restatement -- bit-identical to it -- when that library is absent).  Token ids must be identical wherever the
    reference's top-2 margin exceeds the bound; ids are fed from the reference so one near-tie cannot derail the rest.

    The logit bound.  Every matmul of the step is within 4e-7 of the oracle at these shapes (profiles/diag_7b_stages.py; the
    residue is fp32 summation order), but each Q8_0 activation quantisation is a rounding DISCONTINUITY: one code that lands
    on the other side of .5 moves that element by 1/127 of its block maximum, and the next quantisation amplifies that
    again.  The reference run against ITSELF with every embedding value moved by +-64 ulp (4e-6 relative) differs by
    1.4e-2 max / 3e-3 rms of max|logit| on this model, and does not grow further with a larger perturbation: that is the
    conditioning floor of the Q4_0 x Q8_0 path at this width, measured below in the same loop (`self_err`).  The CUDA
    step has to stay within max(1e-2, 1.5 x the largest self_err seen so far) of the reference at every step, and within 2.5e-2 outright."""
    rng = np.random.default_rng(2024)
    hp = dict(n_vocab=32000, n_embd=4096, n_head=32, n_head_kv=32, n_layer=2, n_ff=11008, n_ctx=64, norm_eps=1e-5, rope_theta=10000.0,
              rope_scale=1.0)
    E, FF, V = hp["n_embd"], hp["n_ff"], hp["n_vocab"]
    tok = rng.standard_normal((V, E), dtype=np.float32)
    out_norm = rng.uniform(0.5, 1.5, E).astype(np.float32)

    def qw(n, k):
        return oracle.quantize_q4_0((rng.standard_normal((n, k), dtype=np.float32) * np.float32(1.0 / np.sqrt(k))))

    shapes = dict(wq=(E, E), wk=(E, E), wv=(E, E), wo=(E, E), w1=(FF, E), w2=(E, FF), w3=(FF, E))
    layers = []
    for _ in range(hp["n_layer"]):
        lay = dict(attn_norm=rng.uniform(0.5, 1.5, E).astype(np.float32), ffn_norm=rng.uniform(0.5, 1.5, E).astype(np.float32))
        for name, (n, k) in shapes.items():
            lay[name] = qw(n, k)
        layers.append(lay)
    out_rows = qw(V, E)
    mk = (lambda t_: oracle.RefNeLlama(hp, t_, out_norm, out_rows, layers)) if oracle.ref_ne() is not None else (
        lambda t_: OracleLlama(hp, t_, out_norm, out_rows, layers))
    ref = mk(tok)
    jig = (rng.integers(0, 2, tok.shape, dtype=np.int8).astype(np.int32) * 2 - 1) * 64
    ref_jig = mk((tok.view(np.int32) + jig).view(np.float32))  # the same engine, inputs moved by +-64 ulp
    del jig
    eng = ns.Llama(**hp)
    eng.set_f32(ns.Llama.TOK_EMBD, 0, tok)
    eng.set_f32(ns.Llama.OUT_NORM, 0, out_norm)
    eng.set_weight(ns.Llama.OUTPUT, 0, ns.Weight.from_q4_0_host(out_rows, V, E))
    ids = dict(wq=ns.Llama.WQ, wk=ns.Llama.WK, wv=ns.Llama.WV, wo=ns.Llama.WO, w1=ns.Llama.W1, w2=ns.Llama.W2, w3=ns.Llama.W3)
    for il, lay in enumerate(layers):
        eng.set_f32(ns.Llama.ATTN_NORM, il, lay["attn_norm"])
        eng.set_f32(ns.Llama.FFN_NORM, il, lay["ffn_norm"])
        for name, (n, k) in shapes.items():
            eng.set_weight(ids[name], il, ns.Weight.from_q4_0_host(lay[name], n, k))
    prompt = [1] + [int(t) for t in rng.integers(3, V, 11)]
    pos, agree, checked, worst, worst_self = 0, 0, 0, 0.0, 0.0
    t = prompt[0]
    for step in range(len(prompt) + 16):
        want = ref.eval([t], pos)
        self_err = float(np.abs(ref_jig.eval([t], pos) - want).max())
        got, nxt = eng.eval([t], pos)
        scale = max(1.0, float(np.abs(want).max()))
        err = float(np.abs(got - want).max())
        worst_self = max(worst_self, self_err / scale)     # running maximum: the floor is a property of the model, not of one step
        bound = min(max(1e-2, 1.5 * worst_self), 2.5e-2) * scale
        assert err <= bound, (step, err / scale, worst_self)
        worst = max(worst, err / scale)
        top = np.sort(want)[-2:]
        if top[1] - top[0] > 2 * bound:
            checked += 1
            agree += int(nxt == greedy(want))
        pos += 1
        t = prompt[pos] if pos < len(prompt) else greedy(want)
    print(f"7B-shape decode: worst |dlogit|/max|logit| {worst:.2e}; the reference against itself (+-64 ulp inputs) {worst_self:.2e}; "
          f"ids {agree}/{checked}")
    assert checked >= 8 and agree == checked, (agree, checked)
    eng.close()
    for r in (ref, ref_jig):
        if hasattr(r, "close"):
            r.close()


def _build_smooth(n_head, n_head_kv, n_ctx, seed=0, n_layer=2):
    """the same toy Llama with BesTLA int4 weights evaluated in fp32 (no activation quantiser): the logits are a smooth function of
    the attention output, so two attention kernels can be compared tightly through the whole engine"""
    rng = np.random.default_rng(seed)
    hp = dict(n_vocab=320, n_embd=256, n_head=n_head, n_head_kv=n_head_kv, n_layer=n_layer, n_ff=512, n_ctx=n_ctx, norm_eps=1e-5,
              rope_theta=10000.0, rope_scale=1.0)
    E, FF, V = hp["n_embd"], hp["n_ff"], hp["n_vocab"]
    kvd = E // n_head * n_head_kv
    mk = lambda n, k: ns.Weight.from_blob(ns.np_bestla_quantize(rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32), "int4", 32, "sym",
                                                                "fp32", "fp32"))
    eng = ns.Llama(**hp)
    eng.set_f32(ns.Llama.TOK_EMBD, 0, rng.normal(0, 1, (V, E)).astype(np.float32))
    eng.set_f32(ns.Llama.OUT_NORM, 0, rng.uniform(0.5, 1.5, E).astype(np.float32))
    eng.set_weight(ns.Llama.OUTPUT, 0, mk(V, E))
    shapes = {ns.Llama.WQ: (E, E), ns.Llama.WK: (kvd, E), ns.Llama.WV: (kvd, E), ns.Llama.WO: (E, E), ns.Llama.W1: (FF, E),
              ns.Llama.W2: (E, FF), ns.Llama.W3: (FF, E)}
    for il in range(n_layer):
        eng.set_f32(ns.Llama.ATTN_NORM, il, rng.uniform(0.5, 1.5, E).astype(np.float32))
        eng.set_f32(ns.Llama.FFN_NORM, il, rng.uniform(0.5, 1.5, E).astype(np.float32))
        for tid, (n, k) in shapes.items():
            eng.set_weight(tid, il, mk(n, k))
    return hp, eng


@pytest.mark.parametrize("n_head,n_head_kv", [(4, 4), (2, 2), (4, 2)])
def test_tensor_core_prompt_attention_matches_the_scalar_kernel(n_head, n_head_kv, monkeypatch):
    """Prompts of >= 8 tokens run the causal attention on mma.sync (attn_mma_kernel: 64 query rows per CTA, K/V tiles of 64 keys):
    several q tiles, several key tiles, ragged last tiles and a non-zero n_past (chunked prompt), head sizes 64 and 128, GQA.
    Compared with the decode-shaped scalar kernel (NS_ATTN_SCALAR=1, itself held to the CPU graph by the tests above) on an engine
    whose matmuls are smooth (fp32 compute): only the fp16 rounding of the probabilities differs (5e-4 relative)."""
    hp, eng = _build_smooth(n_head, n_head_kv, n_ctx=400, seed=21)
    rng = np.random.default_rng(8)
    p1 = [int(t) for t in rng.integers(3, hp["n_vocab"], 37)]
    p2 = [int(t) for t in rng.integers(3, hp["n_vocab"], 141)]
    p3 = [int(t) for t in rng.integers(3, hp["n_vocab"], 200)]

    def run():
        return [eng.eval(p1, 0)[0], eng.eval(p2, len(p1))[0], eng.eval([11], len(p1) + len(p2))[0], eng.eval(p3, len(p1) + len(p2) + 1)[0]]

    a = run()
    monkeypatch.setenv("NS_ATTN_SCALAR", "1")
    b = run()
    monkeypatch.delenv("NS_ATTN_SCALAR")
    for x, y in zip(a, b):
        assert np.isfinite(x).all()
        # bf16 activation rounding in the tensor-core GEMMs of both runs turns 5e-4 into a few 1e-3; a layout bug would be O(1)
        assert float(np.abs(x - y).max()) <= 1e-2 * max(1.0, float(np.abs(y).max())), float(np.abs(x - y).max())
    eng.close()


def test_tensor_core_prompt_attention_against_the_cpu_graph():
    """a 37 + 90 token chunked prompt in exact-prefill mode (integer matmuls as the reference, attention on mma.sync) against the
    CPU graph, bar = north star or 1.5 x the graph's own conditioning floor (see the exact-prefill test)"""
    hp, orc, eng = _build(seed=23, n_ctx=160, jig=64)
    eng.set_exact_prefill(True)
    rng = np.random.default_rng(9)
    p1 = [int(t) for t in rng.integers(3, hp["n_vocab"], 37)]
    p2 = [int(t) for t in rng.integers(3, hp["n_vocab"], 90)]
    w1, w2 = orc.eval(p1, 0), orc.eval(p2, len(p1))
    j1, j2 = orc.jig.eval(p1, 0), orc.jig.eval(p2, len(p1))
    floor = max(float(np.abs(j1 - w1).max()) / max(1.0, float(np.abs(w1).max())), float(np.abs(j2 - w2).max()) / max(1.0, float(np.abs(w2).max())))
    tol = min(max(1e-2, 1.5 * floor), 2.5e-2)
    _check_logits(eng.eval(p1, 0)[0], w1, tol=tol)
    _check_logits(eng.eval(p2, len(p1))[0], w2, tol=tol)
    eng.close()


@pytest.mark.parametrize("n_head,n_head_kv", [(4, 4), (2, 1)])
def test_split_context_decode_attention_matches_the_single_cta_kernel(n_head, n_head_kv, monkeypatch):
    """decode attention with K / V staged by TMA and the context split into ranges of 256 positions (attn_decode_kernel) against the
    one-CTA-per-head kernel with dependent row loads (NS_ATTN_OLD_DECODE=1), token by token across the 256 and 512 boundaries
    (1, 2 and 3 active ranges; a range holding only the new token), head sizes 64 and 128, GQA; smooth fp32-compute engine.  Past
    512: three single-token evals, two consecutive generate calls, and an eval that attends to the rows those calls wrote"""
    rng = np.random.default_rng(5)
    prompt = [int(t) for t in rng.integers(3, 320, 250)]
    steps = [int(t) for t in rng.integers(3, 320, 12)]
    jump = [int(t) for t in rng.integers(3, 320, 250)]

    def run(old):
        if old:
            monkeypatch.setenv("NS_ATTN_OLD_DECODE", "1")
        hp, eng = _build_smooth(n_head, n_head_kv, n_ctx=600, seed=31)
        outs = [eng.eval(prompt, 0)[0]]
        n_past = len(prompt)
        for t in steps:  # positions 250 .. 261: crosses into the second range
            outs.append(eng.eval([t], n_past)[0])
            n_past += 1
        outs.append(eng.eval(jump, n_past)[0])  # to position 512
        n_past += len(jump)
        for t in steps[:3]:                     # positions 512 .. 514: three active ranges
            outs.append(eng.eval([t], n_past)[0])
            n_past += 1
        gen = []
        for first in (7, 8):                    # two consecutive generate calls (graph replays, merge ticket reset between)
            gen.append(eng.generate(first, n_past, 4))
            n_past += 4
        outs.append(eng.eval([9], n_past)[0])   # attends to the K / V rows the generated steps wrote
        eng.close()
        if old:
            monkeypatch.delenv("NS_ATTN_OLD_DECODE")
        return outs, gen

    a, ga = run(False)
    b, gb = run(True)
    assert len(a) == len(b) == 1 + len(steps) + 1 + 3 + 1
    same_ids = all(np.array_equal(x, y) for x, y in zip(ga, gb))  # else the last eval attends to different tokens' rows
    for i, (x, y) in enumerate(zip(a, b) if same_ids else zip(a[:-1], b[:-1])):
        assert np.isfinite(x).all()
        assert float(np.abs(x - y).max()) <= 1e-2 * max(1.0, float(np.abs(y).max())), (i, float(np.abs(x - y).max()))
    assert [len(g) for g in ga] == [len(g) for g in gb] == [4, 4]  # (greedy ids may part at a near-tie; the logits are the check)


def test_long_context_decode_against_the_cpu_graph():
    """300-token prompt (tensor-core prompt attention), then single-token steps with two active ranges, against the CPU graph"""
    hp, orc, eng = _build(seed=33, n_ctx=320, jig=64)
    eng.set_exact_prefill(True)
    rng = np.random.default_rng(11)
    prompt = [int(t) for t in rng.integers(3, hp["n_vocab"], 300)]
    want = orc.eval(prompt, 0)
    floor = float(np.abs(orc.jig.eval(prompt, 0) - want).max()) / max(1.0, float(np.abs(want).max()))
    tol = min(max(1e-2, 1.5 * floor), 2.5e-2)
    _check_logits(eng.eval(prompt, 0)[0], want, tol=tol)
    n_past = len(prompt)
    for t in (9, 200, 31):
        want = orc.eval([t], n_past)
        floor = float(np.abs(orc.jig.eval([t], n_past) - want).max()) / max(1.0, float(np.abs(want).max()))
        _check_logits(eng.eval([t], n_past)[0], want, tol=min(max(1e-2, 1.5 * floor), 2.5e-2))
        n_past += 1
    eng.close()
