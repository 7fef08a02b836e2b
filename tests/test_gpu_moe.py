"""GPU parity tests of the expert-indexed nodes (mixture of experts): ns_mul_mat_id / ns_ffn_id / ns_mul_mat_id_q4_0_f32_host.

Reference: ne_mul_mat_id, ne_mul_id_ffn_silu (core/ne_layers.c:2384-2460); compute ne_compute_forward_mul_mat_id_q_f32
(:7345-7498, ggml types), _q_f32_bestla (:7783-7916, BesTLA blobs), ne_compute_forward_ffn_id_silu (:8053-8071).
Checkers: the oracle restatement (pinned bit-for-bit to the reference engine in tests/test_moe_cpu.py), the golden fixture
generated from the reference engine, and the reference's OWN engine linked against libns_b200.so (oracle/_ref/libref_ne_ns.so).
Bars: groups of <= 32 tokens run exact-integer block sums (GEMV ring / integer tensor cores): 1e-4 (fp32 summation order only);
larger groups take the bf16 tensor-core GEMM: the north-star 1e-2.
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle
import neural_speed_b200 as ns

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    ns.lib().bestla_init()
    yield
    ns.lib().ns_host_cache_clear()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def sync():
    torch.cuda.synchronize()
    ns.lib().bestla_device_sync(None)


def close(got, want, rtol):
    scale = float(np.abs(want).max()) + 1e-30
    np.testing.assert_allclose(got, want, rtol=rtol, atol=rtol * scale)


def _q4_experts(rng, n_as, n, k):
    rows = [oracle.quantize_q4_0(rng.normal(0, 0.02, (n, k)).astype(np.float32)) for _ in range(n_as)]
    return rows, [ns.Weight.from_q4_0_host(r, n, k) for r in rows]


@pytest.mark.parametrize("m,on_device", [(1, False), (2, True), (7, False), (40, True), (300, False)])
def test_q4_0_mul_mat_id_matches_the_oracle(m, on_device):
    rng = np.random.default_rng(50 + m)
    n_as, n, k, n_used = 8, 192, 1024, 2
    rows, ws = _q4_experts(rng, n_as, n, k)
    a = rng.normal(0, 1, (m, k)).astype(np.float32)
    ids = rng.integers(0, n_as, (m, n_used)).astype(np.int32)
    if m >= 7:
        ids[:3, 1] = 6  # a contiguous run on one expert
    ad = dev(a)
    idd = dev(ids)
    for slot in range(n_used):
        out = torch.full((m, n), float("nan"), device="cuda")
        torch.cuda.synchronize()
        ns.mul_mat_id(ws, (idd.data_ptr(), n_used) if on_device else ids, slot, ad.data_ptr(), k, out.data_ptr(), n, m)
        sync()
        want = oracle.mul_mat_id_q4_0_f32(rows, ids, slot, a)
        biggest = int(np.bincount(ids[:, slot], minlength=n_as).max())
        close(out.cpu().numpy(), want, 1e-4 if biggest <= 32 else 1e-2)
    # the exact-integer path whatever the group size
    out = torch.full((m, n), float("nan"), device="cuda")
    torch.cuda.synchronize()
    ns.mul_mat_id(ws, ids, 0, ad.data_ptr(), k, out.data_ptr(), n, m, flags=ns.MM_FORCE_GEMV)
    sync()
    close(out.cpu().numpy(), oracle.mul_mat_id_q4_0_f32(rows, ids, 0, a), 1e-4)


def test_tokens_already_grouped_take_no_gather():
    """ids sorted by expert: the rows are used in place (no gather / scatter launches)."""
    rng = np.random.default_rng(3)
    n_as, n, k, m = 4, 128, 512, 8
    rows, ws = _q4_experts(rng, n_as, n, k)
    a = rng.normal(0, 1, (m, k)).astype(np.float32)
    ids = np.array([[0], [0], [1], [1], [1], [3], [3], [3]], np.int32)
    ad = dev(a)
    out = torch.full((m, n), float("nan"), device="cuda")
    torch.cuda.synchronize()
    lc0 = ns.lib().ns_launch_count()
    ns.mul_mat_id(ws, ids, 0, ad.data_ptr(), k, out.data_ptr(), n, m)
    sync()
    launches = ns.lib().ns_launch_count() - lc0
    close(out.cpu().numpy(), oracle.mul_mat_id_q4_0_f32(rows, ids, 0, a), 1e-4)
    assert launches <= 2 * 3, launches  # three experts with tokens: one matmul (+ at most an activation image) each


def test_golden_fixture_through_the_host_drop_in():
    z = np.load(os.path.join(G, "moe_q4_0.npz"))
    rows = [np.ascontiguousarray(r) for r in z["rows"]]
    a, ids = np.ascontiguousarray(z["a"]), np.ascontiguousarray(z["ids"])
    n, k = rows[0].shape[0], a.shape[1]
    ptrs = (C.c_void_p * len(rows))(*[r.ctypes.data for r in rows])
    for slot in range(ids.shape[1]):
        out = np.zeros((a.shape[0], n), np.float32)
        rc = ns.lib().ns_mul_mat_id_q4_0_f32_host(ptrs, len(rows), rows[0].shape[1], ids.ctypes.data_as(C.c_void_p), ids.shape[1], slot,
                                                  a.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), k, n, a.shape[0])
        assert rc == 0, ns.last_error()
        close(out, z["out"][slot], 1e-4)


def test_expert_id_out_of_range_fails_loudly():
    rng = np.random.default_rng(4)
    rows, ws = _q4_experts(rng, 2, 64, 256)
    a = dev(rng.normal(0, 1, (2, 256)).astype(np.float32))
    out = torch.zeros(2, 64, device="cuda")
    with pytest.raises(RuntimeError, match="expert id"):
        ns.mul_mat_id(ws, np.array([[0], [2]], np.int32), 0, a.data_ptr(), 256, out.data_ptr(), 64, 2)


def _btla_oracle_mm(w_nk, g, asym, a):
    q, sc, zp = oracle.btla_quantize(np.ascontiguousarray(w_nk.T), g, 4, asym)
    a8, asc, azp = oracle.btla_quantize_act_u8(np.ascontiguousarray(a, np.float32), g)
    return oracle.btla_gemv_u8s8(a8, asc, azp, q, sc, zp, g)


def _btla_experts(g, alg):
    rng = np.random.default_rng(60 + g)
    n_as, n, k, m, n_used = 4, 256, 512, 9, 2
    w = [rng.normal(0, 1.0 / np.sqrt(k), (n, k)).astype(np.float32) for _ in range(n_as)]
    blobs = [ns.np_bestla_quantize(x, "int4", g, alg, "fp32", "int8") for x in w]
    a = rng.normal(0, 1, (m, k)).astype(np.float32)
    ids = rng.integers(0, n_as, (m, n_used)).astype(np.int32)
    want = np.stack([_btla_oracle_mm(w[int(ids[t, 1])], g, alg == "asym", a[t:t + 1])[0] for t in range(m)])
    return blobs, a, ids, want


@pytest.mark.parametrize("g,alg,threads", [(32, "sym", 1), (128, "asym", 3)])
def test_btla_experts_through_the_reference_engine_on_the_drop_ins(g, alg, threads):
    """ne_graph_compute of the REFERENCE (linked against libns_b200.so) runs NE_OP_MUL_MAT_ID on BesTLA experts token by token
    through bestla_f32f32_forward: it must give the CPU oracle's numbers.  Runs where oracle/_ref was built with the reference."""
    Lns = oracle.ref_ne_ns()
    if Lns is None:
        pytest.skip("oracle/_ref/libref_ne_ns.so not built (the reference's engine is not part of this repository)")
    blobs, a, ids, want = _btla_experts(g, alg)
    n, k = want.shape[1], a.shape[1]
    lc0 = ns.lib().ns_launch_count()
    eng = oracle.ref_mul_mat_id(Lns, blobs, oracle.NE_TYPE_BTLA, n, k, ids, 1, a, n_threads=threads)
    assert ns.lib().ns_launch_count() > lc0, "the reference engine did not reach the CUDA kernels"
    close(eng, want, 1e-4)


@pytest.mark.parametrize("g,alg", [(32, "sym"), (128, "asym")])
def test_btla_experts_grouped_by_ns_mul_mat_id(g, alg):
    """ns_mul_mat_id groups the tokens by expert: it must give the CPU oracle's numbers for the selected expert of every token."""
    blobs, a, ids, want = _btla_experts(g, alg)
    m, n, k = a.shape[0], want.shape[1], a.shape[1]
    ws = [ns.Weight.from_blob(b) for b in blobs]
    ad = dev(a)
    out = torch.full((m, n), float("nan"), device="cuda")
    torch.cuda.synchronize()
    ns.mul_mat_id(ws, ids, 1, ad.data_ptr(), k, out.data_ptr(), n, m)
    sync()
    close(out.cpu().numpy(), want, 1e-4)


def _ffn_id_experts():
    rng = np.random.default_rng(71)
    n_as, k, fmid, g = 4, 256, 704, 128
    mk = lambda r, c: ns.np_bestla_quantize(rng.normal(0, 1.0 / np.sqrt(c), (r, c)).astype(np.float32), "int4", g, "sym", "fp32", "int8")
    gate, up, down = [mk(fmid, k) for _ in range(n_as)], [mk(fmid, k) for _ in range(n_as)], [mk(k, fmid) for _ in range(n_as)]
    wg, wu, wd = ([ns.Weight.from_blob(b) for b in bl] for bl in (gate, up, down))
    m = 6
    x = rng.normal(0, 1, (m, k)).astype(np.float32)
    ids = rng.integers(0, n_as, (m, 2)).astype(np.int32)
    return (gate, up, down), (wg, wu, wd), x, ids


def _ffn_id(wg, wu, wd, x, ids):
    m, k, fmid = x.shape[0], x.shape[1], wg[0].n
    xd = dev(x)
    tmp = torch.zeros(2 * m * fmid, device="cuda")
    out = torch.full((m, k), float("nan"), device="cuda")
    torch.cuda.synchronize()
    ns.ffn_id(wg, wd, wu, ids, 1, xd.data_ptr(), k, tmp.data_ptr(), out.data_ptr(), k, m)
    sync()
    got = out.cpu().numpy()
    for t in range(m):  # per-token fused FFN of the selected expert (same kernels, m = 1)
        e = int(ids[t, 1])
        one = torch.full((1, k), float("nan"), device="cuda")
        t1 = torch.zeros(2 * fmid, device="cuda")
        torch.cuda.synchronize()
        ns.ffn_silu(wg[e], wd[e], wu[e], xd[t:t + 1].data_ptr(), k, t1.data_ptr(), one.data_ptr(), k, 1)
        sync()
        close(got[t:t + 1], one.cpu().numpy(), 1e-4)
    return got


def test_ffn_id_against_per_token_fused_ffns():
    """ne_mul_id_ffn_silu: a 6-token batch with per-token experts through ns_ffn_id against per-token fused FFNs."""
    _, (wg, wu, wd), x, ids = _ffn_id_experts()
    _ffn_id(wg, wu, wd, x, ids)


def test_ffn_id_against_the_reference_engine_and_the_oracle():
    """ne_mul_id_ffn_silu: one decode token through the reference engine on the drop-ins (it reads ONE id for the whole node,
    ne_layers.c:8062) against ns_ffn_id.  Runs where oracle/_ref was built with the reference."""
    Lns = oracle.ref_ne_ns()
    if Lns is None:
        pytest.skip("oracle/_ref/libref_ne_ns.so not built (the reference's engine is not part of this repository)")
    (gate, up, down), (wg, wu, wd), x, ids = _ffn_id_experts()
    got = _ffn_id(wg, wu, wd, x, ids)
    k, fmid = x.shape[1], wg[0].n
    eng = oracle.ref_ffn_id_silu(Lns, gate, down, up, k, fmid, k, ids[:1], 1, x[:1], n_threads=2)
    close(eng, got[:1], 1e-4)
