"""INTEGRATION.md A exercised for real: the REFERENCE's own graph engine (neural_speed/core/ne_layers.c, compiled where it lies
into oracle/_ref/libref_ne_ns.so) linked against libns_b200.so instead of the reference's core/layers/*.cpp.  ne_graph_compute
(ne_layers.c:11915-12010) asks bestla_support for every node, sizes its work buffer from the answer, enters the BesTLA nodes once
(n_tasks = 1) through bestla_parallel_for and lands in the CUDA drop-ins (bestla_f32f32_forward, bestla_fusion_QKV / FFN_SiLu,
bestla_mul / add / layernormalization).  A tiny Llama with BesTLA int4 blobs must give the logits of the CPU oracle
(oracle/llama_model.py with the BesTLA u8 x s8 arithmetic of kernel_ref.h:1825,2372) within the north-star 1e-2 and pick the
same greedy tokens."""
import numpy as np
import pytest
import torch

import neural_speed_b200 as ns
import oracle
from oracle.llama_model import OracleLlama, greedy

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _need():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    if oracle.ref_ne_ns() is None:
        pytest.skip("oracle/_ref/libref_ne_ns.so not built (the reference's engine is not part of this repository)")
    ns.lib().bestla_init()
    yield
    ns.lib().ns_host_cache_clear()


class BtlaOracleLlama(OracleLlama):
    """OracleLlama whose matmul weights are (q [K,N] int8, scales [K/g,N], zp, g): BesTLA int8 compute = u8 activations per
    K-block (kernel_ref.h:1825) x s4 weights, exact integer block dots (kernel_ref.h:2372)."""

    @staticmethod
    def _mm(w, a):
        q, sc, zp, g = w
        a8, asc, azp = oracle.btla_quantize_act_u8(np.ascontiguousarray(a, np.float32), g)
        return oracle.btla_gemv_u8s8(a8, asc, azp, q, sc, zp, g)


def _build(g, alg, seed=0, n_layer=2):
    rng = np.random.default_rng(seed)
    hp = dict(n_vocab=320, n_embd=256, n_head=4, n_head_kv=4, n_layer=n_layer, n_ff=512, n_ctx=32, norm_eps=1e-5, rope_theta=10000.0,
              rope_scale=1.0)
    E, FF, V = hp["n_embd"], hp["n_ff"], hp["n_vocab"]
    tok = rng.normal(0, 1, (V, E)).astype(np.float32)
    out_norm = rng.uniform(0.5, 1.5, E).astype(np.float32)
    shapes = dict(wq=(E, E), wk=(E, E), wv=(E, E), wo=(E, E), w1=(FF, E), w2=(E, FF), w3=(FF, E))

    def quant(n, k):
        w = rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32)
        blob = ns.np_bestla_quantize(w, "int4", g, alg, "fp32", "int8")
        q, sc, zp = oracle.btla_quantize(np.ascontiguousarray(w.T), g, 4, alg == "asym")
        return blob, (q, sc, zp, g)

    blobs, orcs = [], []
    for _ in range(n_layer):
        lb = dict(attn_norm=rng.uniform(0.5, 1.5, E).astype(np.float32), ffn_norm=rng.uniform(0.5, 1.5, E).astype(np.float32))
        lo = dict(lb)
        for name, (n, k) in shapes.items():
            lb[name], lo[name] = quant(n, k)
        blobs.append(lb)
        orcs.append(lo)
    out_blob, out_orc = quant(V, E)
    return hp, tok, out_norm, (out_blob, blobs), (out_orc, orcs)


@pytest.mark.parametrize("g,alg,fused,threads", [(32, "sym", True, 1), (128, "asym", True, 4), (32, "sym", False, 3)])
def test_reference_engine_on_cuda_dropins(g, alg, fused, threads):
    hp, tok, out_norm, (out_blob, blobs), (out_orc, orcs) = _build(g, alg)
    orc = BtlaOracleLlama(hp, tok, out_norm, out_orc, orcs)
    eng = oracle.RefNeLlama(hp, tok, out_norm, out_blob, blobs, btla=True, fused=fused, n_threads=threads, on_ns=True)
    L = ns.lib()
    lc0 = L.ns_launch_count()
    prompt = [1, 17, 301, 5, 88]
    want = orc.eval(prompt, 0)
    got = eng.eval(prompt, 0)
    assert L.ns_launch_count() > lc0, "the reference engine did not reach the CUDA kernels"
    n_past = len(prompt)
    toks = []
    for step in range(6):
        scale = max(1.0, float(np.abs(want).max()))
        assert np.isfinite(got).all()
        assert float(np.abs(got - want).max()) <= 1e-2 * scale, (step, float(np.abs(got - want).max()), scale)
        top = np.sort(want)[-2:]
        nxt = greedy(want)
        if top[1] - top[0] > 2e-2 * scale:
            assert greedy(got) == nxt
        toks.append(nxt)
        want = orc.eval([nxt], n_past)
        got = eng.eval([nxt], n_past)
        n_past += 1
    eng.close()
    assert len(set(toks)) > 1
