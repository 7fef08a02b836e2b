"""CPU side of the expert-indexed matmul (ne_mul_mat_id): the oracle restatement against the REFERENCE's own engine
(ne_compute_forward_mul_mat_id_q_f32, core/ne_layers.c:7345-7498, run through ne_graph_compute; its answers for these inputs
are stored in tests/golden/reference.npz) and against the committed golden fixture generated from it
(tests/golden/make_golden_moe.py)."""
import os

import numpy as np
import pytest

import oracle
from oracle import golden

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_restatement_matches_the_golden_fixture_bit_for_bit():
    z = np.load(os.path.join(G, "moe_q4_0.npz"))
    rows = [np.ascontiguousarray(r) for r in z["rows"]]
    for slot in range(z["ids"].shape[1]):
        got = oracle.mul_mat_id_q4_0_f32(rows, z["ids"], slot, z["a"])
        assert np.array_equal(got, z["out"][slot])


@pytest.mark.parametrize("n_threads", [1, 3])
def test_restatement_matches_the_reference_engine(n_threads):
    rng = np.random.default_rng(7 + n_threads)
    n_as, n, k, n_tok, n_used = 8, 64, 512, 11, 2
    rows = [oracle.quantize_q4_0(rng.normal(0, 0.02, (n, k)).astype(np.float32)) for _ in range(n_as)]
    a = rng.normal(0, 1.0, (n_tok, k)).astype(np.float32)
    ids = rng.integers(0, n_as, (n_tok, n_used)).astype(np.int32)
    ids[:3, 0] = 5  # a run of tokens on one expert and experts nobody picked
    for slot in range(n_used):
        got = oracle.mul_mat_id_q4_0_f32(rows, ids, slot, a)
        golden.check(f"mul_mat_id[{n_threads}].slot{slot}", got,
                     lambda: oracle.ref_mul_mat_id(oracle.ref_ne(), rows, oracle.NE_TYPE_Q4_0, n, k, ids, slot, a, n_threads=n_threads))


def test_host_side_grouping_of_tokens_by_expert():
    """ns_moe_plan: the grouping ns_mul_mat_id performs before it launches anything (matrix_rows / matrix_row_counts of
    ne_layers.c:7440-7449): stable sort by expert, spans, the already-grouped shortcut, the reference's id range assertion."""
    import ctypes as C

    import neural_speed_b200 as ns
    L = ns.lib()
    rng = np.random.default_rng(2)
    m, n_as, n_used = 37, 6, 2
    ids = rng.integers(0, n_as, (m, n_used)).astype(np.int32)
    ids[:, 1][ids[:, 1] == 4] = 0  # an expert nobody picks
    order = np.zeros(m, np.int32)
    span = np.zeros(2 * n_as, np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for slot in range(n_used):
        rc = L.ns_moe_plan(p(ids), n_used, slot, m, n_as, p(order), p(span))
        assert rc == 0
        want = np.argsort(ids[:, slot], kind="stable")
        assert np.array_equal(order, want)
        counts = np.bincount(ids[:, slot], minlength=n_as)
        assert np.array_equal(span[1::2] - span[0::2], counts)
        assert span[0] == 0 and np.array_equal(span[2::2], span[1:-1:2])  # contiguous spans
    grouped = np.sort(ids[:, :1], axis=0)
    assert L.ns_moe_plan(p(np.ascontiguousarray(grouped)), 1, 0, m, n_as, p(order), p(span)) == 1
    assert np.array_equal(order, np.arange(m))
    bad = ids.copy()
    bad[5, 0] = n_as
    assert L.ns_moe_plan(p(bad), n_used, 0, m, n_as, p(order), p(span)) < 0 and "expert id" in ns.last_error()
    assert L.ns_moe_plan(p(ids), n_used, 2, m, n_as, p(order), p(span)) < 0  # slot outside the selection
