"""GPU parity tests of scoring / top-k / metrics.  Indices must be BIT-EXACT against the oracle's
canonical score + stable descending order (ties -> lower item id), as north_star requires."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import mf_oracle as o

pytestmark = pytest.mark.gpu
G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))


def cpu(t):
    return t.detach().cpu().numpy()


def model_with(U, V):
    from teamoflow_b200.mf.matrix_factorization import MatrixFactorization
    from teamoflow_b200.mf._engine import new_storage
    m = MatrixFactorization(U.shape[1])
    r = U.shape[1]
    m.user_embedding = new_storage(U.shape[0], r, torch.as_tensor(U, device="cuda"))[:, :r]
    m.item_embedding = new_storage(V.shape[0], r, torch.as_tensor(V, device="cuda"))[:, :r]
    return m


def fused_topk(U, V, k, clamp, item_offset=0):
    from teamoflow_b200.mf._engine import new_storage
    from teamoflow_b200.mf.matrix_factorization import score_topk
    r = U.shape[1]
    Us = new_storage(U.shape[0], r, torch.as_tensor(U, device="cuda"))
    Vs = new_storage(V.shape[0], r, torch.as_tensor(V, device="cuda"))
    idx, sc = score_topk(Us, Vs, r, k, clamp, item_offset)
    torch.cuda.synchronize()
    return cpu(idx), cpu(sc)


def oracle_topk(U, V, k, clamp):
    P = o.canonical_scores(U, V)
    if clamp:
        P = np.where(P > 0, P, np.float32(0))
    idx = o.topk_stable(P, k)
    return idx, np.take_along_axis(P, idx.astype(np.int64), 1)


def test_predict_dense_is_canonical_bit_exact():
    rng = np.random.default_rng(0)
    U = rng.standard_normal((70, 37)).astype(np.float32)
    V = rng.standard_normal((90, 37)).astype(np.float32)
    m = model_with(U, V)
    P = cpu(m.predict())
    assert np.array_equal(P, o.canonical_scores(U, V))
    from teamoflow_b200.mf.predict_graphs import DotProductPrediction
    assert np.array_equal(cpu(DotProductPrediction().get_prediction(m.user_embedding, m.item_embedding)), P)
    A = (rng.random((70, 90)) < 0.1).astype(np.float32)
    allp, unobs = m.predict(torch.as_tensor(A))
    assert np.array_equal(cpu(unobs), P[A == 0])
    ranks = cpu(m.predict_ranks(torch.as_tensor(A)))
    assert np.array_equal(ranks, o.topk_stable(P[A == 0], int((A == 0).sum())))


@pytest.mark.parametrize("n_u,n_i,r,k", [(300, 5000, 32, 10), (129, 257, 128, 100), (64, 1000, 10, 1), (500, 3000, 64, 128),
                                         (130, 700, 200, 17), (10, 40, 5, 40)])
@pytest.mark.parametrize("clamp", [False, True])
def test_fused_topk_random_bit_exact(n_u, n_i, r, k, clamp):
    rng = np.random.default_rng(n_u + n_i + r)
    U = (rng.standard_normal((n_u, r)) / np.sqrt(r)).astype(np.float32)
    V = (rng.standard_normal((n_i, r)) / np.sqrt(r)).astype(np.float32)
    if clamp:
        U[3] = -np.abs(U[3]); V[:] = np.where(rng.random((n_i, 1)) < 0.5, np.abs(V), V)  # rows with few positive scores
        U[5] = 0.0
    idx, sc = fused_topk(U, V, k, clamp)
    widx, wsc = oracle_topk(U, V, k, clamp)
    assert np.array_equal(idx, widx)
    assert np.array_equal(sc, wsc)


def test_fused_topk_grid_golden_ties():
    c = G["grid_topk"]
    U = np.array(c["U_int"], np.float32) / c["scale"]
    V = np.array(c["V_int"], np.float32) / c["scale"]
    idx, _ = fused_topk(U, V, c["k"], False)
    assert idx.tolist() == c["raw"]
    idx, _ = fused_topk(U, V, c["k"], True)
    assert idx.tolist() == c["clamped"]


def test_fused_topk_massive_ties_take_exact_path():
    rng = np.random.default_rng(1)
    U = rng.standard_normal((40, 16)).astype(np.float32)
    V = np.tile(rng.standard_normal((1, 16)).astype(np.float32), (3000, 1))  # every item identical
    V[1234] *= 2.0
    for clamp in (False, True):
        idx, sc = fused_topk(U, V, 20, clamp)
        widx, wsc = oracle_topk(U, V, 20, clamp)
        assert np.array_equal(idx, widx) and np.array_equal(sc, wsc)


def test_fused_topk_adversarial_increasing_scores():
    # scores increase with the item id: every item beats the running threshold (worst case for the filter)
    n_i, r = 6000, 8
    U = np.ones((33, r), np.float32)
    V = np.tile(np.linspace(-1, 1, n_i, dtype=np.float32)[:, None], (1, r))
    idx, _ = fused_topk(U, V, 50, False)
    widx, _ = oracle_topk(U, V, 50, False)
    assert np.array_equal(idx, widx)


def test_item_sharded_topk_merge_equals_single_shot():
    from teamoflow_b200 import _abi
    rng = np.random.default_rng(2)
    n_u, n_i, r, k = 200, 4000, 48, 25
    U = (rng.standard_normal((n_u, r)) / 7).astype(np.float32)
    V = (rng.standard_normal((n_i, r)) / 7).astype(np.float32)
    V[100] = V[3900]  # a tie across shards
    bounds = [0, 1300, 2600, 4000]
    idxs, scs = [], []
    for a, b in zip(bounds[:-1], bounds[1:]):
        i, s = fused_topk(U, V[a:b], k, True, item_offset=a)
        idxs.append(i); scs.append(s)
    idx_in = torch.as_tensor(np.stack(idxs), device="cuda").contiguous()
    sc_in = torch.as_tensor(np.stack(scs), device="cuda").contiguous()
    out_i = torch.empty(n_u, k, dtype=torch.int32, device="cuda")
    out_s = torch.empty(n_u, k, dtype=torch.float32, device="cuda")
    _abi.call("tmf_topk_merge", _abi.ptr(idx_in), _abi.ptr(sc_in), 3, n_u, k, _abi.ptr(out_i), _abi.ptr(out_s))
    widx, wsc = oracle_topk(U, V, k, True)
    assert np.array_equal(cpu(out_i), widx) and np.array_equal(cpu(out_s), wsc)


def test_metrics_golden_and_quirks():
    c = G["metrics_4x5"]
    P, A, k = np.array(c["P"], np.float32), np.array(c["A"], np.float32), c["k"]
    m = model_with(P, np.eye(5, dtype=np.float32))  # U = P, V = I  =>  scores == P exactly
    At = torch.as_tensor(A)
    assert cpu(m._topk(k, clamp=True)).tolist() == c["topk_clamped"]
    np.testing.assert_array_equal(cpu(m.recall_at_k(At, k)), np.array(c["recall_drop"], np.float32))
    keep = [np.inf if x == "inf" else x for x in c["recall_keep"]]
    np.testing.assert_array_equal(cpu(m.recall_at_k(At, k, preserve_rows=True)), np.array(keep, np.float32))
    np.testing.assert_array_equal(cpu(m.precision_at_k(At, k)), np.array(c["precision_drop"], np.float32))
    np.testing.assert_array_equal(cpu(m.precision_at_k(At, k, preserve_rows=True)), np.array(c["precision_keep"], np.float32))
    assert float(m.f1_at_k(At, k)) == float(o.f1_at_k(P, A, k))


@pytest.mark.parametrize("k", [1, 10, 30])
def test_metrics_random_vs_oracle(k):
    rng = np.random.default_rng(k)
    n_u, n_i, r = 150, 400, 16
    U = (rng.standard_normal((n_u, r)) / 4).astype(np.float32)
    V = (rng.standard_normal((n_i, r)) / 4).astype(np.float32)
    A = np.where(rng.random((n_u, n_i)) < 0.05, rng.choice([-2.0, 1.0, 3.0, 5.0], (n_u, n_i)), 0.0).astype(np.float32)
    A[7] = 0.0
    m = model_with(U, V)
    P = o.canonical_scores(U, V)
    At = torch.as_tensor(A)
    from scipy import sparse
    for Ain in (At, sparse.csr_matrix(A)):  # dense like the reference, or sparse (extension)
        np.testing.assert_array_equal(cpu(m.recall_at_k(Ain, k)), o.recall_at_k(P, A, k))
        np.testing.assert_array_equal(cpu(m.recall_at_k(Ain, k, True)), o.recall_at_k(P, A, k, True))
        np.testing.assert_array_equal(cpu(m.precision_at_k(Ain, k)), o.precision_at_k(P, A, k))
    np.testing.assert_allclose(float(m.f1_at_k(At, k)), float(o.f1_at_k(P, A, k)), rtol=1e-6)
    np.testing.assert_allclose(cpu(m.dcg_at_k(At, k)), o.dcg_at_k(P, A, k), rtol=2e-6, atol=1e-6)
    np.testing.assert_allclose(cpu(m.idcg_at_k(At, k)), o.idcg_at_k(P, A, k), rtol=2e-6, atol=1e-6)
    np.testing.assert_allclose(cpu(m.ndcg_at_k(At, k)), o.ndcg_at_k(P, A, k), rtol=5e-6, atol=1e-6)
    np.testing.assert_allclose(cpu(m.ndcg_at_k(At, k, True)), o.ndcg_at_k(P, A, k, True), rtol=5e-6, atol=1e-6)


def test_idcg_uses_negative_gains_when_k_exceeds_nonnegative_count():
    U = np.ones((2, 2), np.float32); V = np.array([[1, 0], [0.5, 0], [0.2, 0], [0.1, 0]], np.float32)
    A = np.array([[2.0, -1.0, -3.0, 1.0], [-1.0, -1.0, -2.0, -4.0]], np.float32)
    m = model_with(U, V)
    P = o.canonical_scores(U, V)
    np.testing.assert_allclose(cpu(m.idcg_at_k(torch.as_tensor(A), 4)), o.idcg_at_k(P, A, 4), rtol=2e-6)
    np.testing.assert_allclose(cpu(m.dcg_at_k(torch.as_tensor(A), 4)), o.dcg_at_k(P, A, 4), rtol=2e-6)


def test_retrieve_user_recs_all_modes():
    rng = np.random.default_rng(4)
    U = rng.standard_normal((30, 6)).astype(np.float32)
    V = rng.standard_normal((200, 6)).astype(np.float32)
    V[50] = V[10]
    m = model_with(U, V)
    P = o.canonical_scores(U, V)
    for user, k in ((None, 5), (3, None), (3, 7), (None, None)):
        got = m.retrieve_user_recs(user=user, k=k)
        assert got.dtype == np.int32
        assert np.array_equal(got, o.retrieve_user_recs(P, user=user, k=k))


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("n_u,n_i,r", [(128, 256, 64), (200, 700, 128), (130, 300, 10), (64, 513, 200)])
def test_tensor_core_scores_within_stated_error_bound(n_u, n_i, r, fmt):
    """The raw tcgen05 GEMM scores obey |s~ - s| <= |du||v| + |u~||dv| + accumulation slack, with u~ = the 16-bit rounding
    of u in the operand format (0 = bf16, 1 = fp16), du = u - u~ (the premise of the exact top-k; the kernel uses the same
    bound with the slab maxima of |v|, |dv|)."""
    from teamoflow_b200 import _abi
    from teamoflow_b200.mf._engine import new_storage
    rng = np.random.default_rng(r)
    U = (rng.standard_normal((n_u, r)) * rng.uniform(0.1, 3.0, (n_u, 1))).astype(np.float32)
    V = (rng.standard_normal((n_i, r)) * rng.uniform(0.1, 3.0, (n_i, 1))).astype(np.float32)
    half_ulp = 2.0 ** -8 if fmt == 0 else 2.0 ** -11
    if n_u >= 200:  # adversarial rows: every component just below a rounding boundary of the format, all products positive
        U[:8] = np.float32(1.0 + half_ulp - 2.0 ** -20) * (2.0 ** rng.integers(-1, 2, (8, 1))).astype(np.float32)
        V[:8] = np.float32(1.0 + half_ulp - 2.0 ** -20)
    Us = new_storage(n_u, r, torch.as_tensor(U, device="cuda")); Vs = new_storage(n_i, r, torch.as_tensor(V, device="cuda"))
    P = torch.full((n_u, n_i), float("nan"), device="cuda")
    ws_bytes = _abi.query("tmf_score_topk_ws_bytes", n_u, n_i, r, 1)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    _abi.call("tmf_score_dense_tc", _abi.ptr(Us), n_u, _abi.ptr(Vs), n_i, r, Us.shape[1], fmt, _abi.ptr(P), _abi.ptr(ws), ws_bytes)
    torch.cuda.synchronize()
    got = cpu(P).astype(np.float64)
    exact = U.astype(np.float64) @ V.astype(np.float64).T
    rnd = (lambda X: torch.as_tensor(X).bfloat16().float().numpy()) if fmt == 0 else (lambda X: torch.as_tensor(X).half().float().numpy())
    Ub, Vb = rnd(U).astype(np.float64), rnd(V).astype(np.float64)
    nrm = lambda X: np.linalg.norm(X, axis=1)  # noqa: E731
    k_pad = (r + 63) // 64 * 64
    bound = (nrm(U - Ub)[:, None] * nrm(V.astype(np.float64))[None, :] + nrm(Ub)[:, None] * nrm(V - Vb)[None, :]
             + 2.4e-7 * k_pad * nrm(Ub)[:, None] * nrm(V.astype(np.float64))[None, :])
    assert np.isfinite(got).all()
    err = np.abs(got - exact)
    assert (err <= bound + 1e-30).all(), f"max err/bound = {(err / bound).max():.3f}"
    # and it really is a product of operands rounded to that format, not something sloppier
    assert np.median(err / bound) < 0.3
    if n_u >= 200:  # the adversarial block really exceeds the naive one-half-ulp figure: the bound must come from the data
        naive = 1.05 * half_ulp * nrm(U.astype(np.float64))[:8, None] * nrm(V.astype(np.float64))[None, :8]
        assert (err[:8, :8] > naive).all()


def test_operand_format_follows_the_data():
    """fp16 operands where they round the embeddings better, bf16 where a component would overflow fp16 or sits in its
    subnormal range -- and the top-k is exact either way."""
    from teamoflow_b200 import _abi
    from teamoflow_b200.mf._engine import new_storage
    rng = np.random.default_rng(8)
    n_u, n_i, r = 128, 256, 64
    base_u = rng.standard_normal((n_u, r)).astype(np.float32)
    base_v = rng.standard_normal((n_i, r)).astype(np.float32)
    for scale, want in ((0.1, "f16"), (1e5, "bf16"), (1e-7, "bf16")):
        U, V = base_u * np.float32(scale), base_v * np.float32(scale if scale < 1 else 1.0)
        Us = new_storage(n_u, r, torch.as_tensor(U, device="cuda")); Vs = new_storage(n_i, r, torch.as_tensor(V, device="cuda"))
        ws_bytes = _abi.query("tmf_score_topk_ws_bytes", n_u, n_i, r, 1)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        P = {}
        for fmt in (-1, 0, 1):
            P[fmt] = torch.full((n_u, n_i), float("nan"), device="cuda")
            _abi.call("tmf_score_dense_tc", _abi.ptr(Us), n_u, _abi.ptr(Vs), n_i, r, Us.shape[1], fmt, _abi.ptr(P[fmt]), _abi.ptr(ws), ws_bytes)
        torch.cuda.synchronize()
        assert torch.equal(P[-1], P[1] if want == "f16" else P[0]), (scale, want)
        idx, sc = fused_topk(U, V, 10, False)
        widx, wsc = oracle_topk(U, V, 10, False)
        assert np.array_equal(idx, widx) and np.array_equal(sc, wsc)


def test_topk_exact_with_adversarial_bf16_rounding():
    """Operands that sit next to bf16 rounding boundaries: class A items (all components just BELOW a boundary, rounded
    down) and class D items (just ABOVE it, rounded up) have interleaved true scores but tensor-core scores that differ
    by 2^-7 |u||v| -- the whole width the rigorous bound allows."""
    rng = np.random.default_rng(77)
    n_u, n_i, r, k = 130, 3000, 64, 20
    lo_ = 1.0 + 2.0 ** -8 - 2.0 ** -20   # -> bf16 1.0
    hi_ = 1.0 + 2.0 ** -8 + 2.0 ** -20   # -> bf16 1 + 2^-7
    U = np.full((n_u, r), lo_, np.float32) * (2.0 ** rng.integers(-1, 2, (n_u, 1))).astype(np.float32)
    V = np.empty((n_i, r), np.float32)
    V[0::2] = (lo_ - 2.0 ** -21 * rng.integers(0, 8, (n_i // 2, 1))).astype(np.float32)
    V[1::2] = (hi_ + 2.0 ** -21 * rng.integers(0, 8, (n_i // 2, 1))).astype(np.float32)
    for clamp in (False, True):
        idx, sc = fused_topk(U, V, k, clamp)
        widx, wsc = oracle_topk(U, V, k, clamp)
        assert np.array_equal(idx, widx) and np.array_equal(sc, wsc)


def test_topk_degenerate_shapes():
    rng = np.random.default_rng(11)
    for n_u, n_i, r, k in ((1, 1, 1, 1), (1, 130, 3, 128), (257, 129, 7, 5), (3, 385, 2, 100), (5, 2049, 4, 9)):
        U = rng.standard_normal((n_u, r)).astype(np.float32)
        V = rng.standard_normal((n_i, r)).astype(np.float32)
        for clamp in (False, True):
            idx, sc = fused_topk(U, V, k, clamp)
            widx, wsc = oracle_topk(U, V, k, clamp)
            assert np.array_equal(idx, widx) and np.array_equal(sc, wsc), (n_u, n_i, r, k, clamp)


def test_topk_larger_sweep_with_rebuilds_bit_exact():
    """enough items per row (60k) that lists are rebuilt/compacted several times, k=100, r=128"""
    rng = np.random.default_rng(12)
    n_u, n_i, r, k = 300, 60_000, 128, 100
    U = (rng.standard_normal((n_u, r)) / np.sqrt(r)).astype(np.float32)
    V = (rng.standard_normal((n_i, r)) / np.sqrt(r)).astype(np.float32) * rng.uniform(0.5, 2.0, (n_i, 1)).astype(np.float32)
    idx, sc = fused_topk(U, V, k, False)
    # oracle on the few thousand best approximate candidates per row only (full 300 x 60k canonical is slow on CPU)
    P = U.astype(np.float64) @ V.astype(np.float64).T
    cand = np.argpartition(-P, 400, axis=1)[:, :400]
    for u in range(n_u):
        c = np.sort(cand[u])
        s = o.canonical_pair_scores(U, V, np.full(c.size, u), c)
        order = np.lexsort((c, -s.astype(np.float64)))[:k]
        assert np.array_equal(idx[u], c[order].astype(np.int32)), u
        assert np.array_equal(sc[u], s[order])


# ------------------------------------------------------------------ item-sharded scoring with exchanged bounds


def _bounded_slabs(U, V, k, clamp, bounds, n_virtual, sample_frac=1.0):
    """The protocol of dist.sharded_topk with the ranks played one after the other on this GPU: bound pass per
    (user slice, slab sample), bounded main pass per slab, merge."""
    from teamoflow_b200 import _abi
    from teamoflow_b200.mf import dist as tdist
    from teamoflow_b200.mf._engine import new_storage
    from teamoflow_b200.mf.matrix_factorization import score_topk
    r = U.shape[1]
    n_u = U.shape[0]
    Us = new_storage(n_u, r, torch.as_tensor(U, device="cuda"))
    slabs = [new_storage(b - a, r, torch.as_tensor(V[a:b], device="cuda")) for a, b in zip(bounds[:-1], bounds[1:])]
    ub = tdist.shard_bounds(n_u, n_virtual)
    rb = torch.cat([tdist.topk_row_bounds(Us, slabs[g], r, k, clamp, bounds[g], ub[g], ub[g + 1],
                                          max(int(slabs[g].shape[0] * sample_frac), 1)) for g in range(n_virtual)]).contiguous()
    idxs, scs = [], []
    for g in range(n_virtual):
        i, s = score_topk(Us, slabs[g], r, k, clamp, bounds[g], row_bound=rb)
        idxs.append(i); scs.append(s)
    idx_in, sc_in = torch.stack(idxs).contiguous(), torch.stack(scs).contiguous()
    out_i = torch.empty(n_u, k, dtype=torch.int32, device="cuda")
    out_s = torch.empty(n_u, k, dtype=torch.float32, device="cuda")
    _abi.call("tmf_topk_merge", _abi.ptr(idx_in), _abi.ptr(sc_in), n_virtual, n_u, k, _abi.ptr(out_i), _abi.ptr(out_s))
    torch.cuda.synchronize()
    n_pad = int((idx_in == 2 ** 31 - 1).sum())
    return cpu(out_i), cpu(out_s), n_pad, cpu(rb)


@pytest.mark.parametrize("clamp", [False, True])
# sample_frac 0.0125: each bound is the k-th best of only k items, so loose that bounded rows fill their lists
@pytest.mark.parametrize("sample_frac", [1.0, 0.3, 0.0125])
def test_bounded_item_slabs_merge_equals_single_shot(clamp, sample_frac):
    rng = np.random.default_rng(12)
    n_u, n_i, r, k = 700, 6000, 48, 25
    U = (rng.standard_normal((n_u, r)) / 7).astype(np.float32)
    V = (rng.standard_normal((n_i, r)) / 7).astype(np.float32)
    V[100] = V[5900]  # a tie across slabs
    idx, sc, n_pad, rb = _bounded_slabs(U, V, k, clamp, [0, 2000, 4000, 6000], 3, sample_frac)
    widx, wsc = oracle_topk(U, V, k, clamp)
    assert np.array_equal(idx, widx) and np.array_equal(sc, wsc)
    # a bound is a lower bound of the global k-th best score
    assert np.all(rb <= wsc[:, k - 1])


def test_bounded_item_slabs_exact_ties_and_nonpositive_rows():
    # grid-valued embeddings: every score exact in fp32, massive ties; rows whose scores are all <= 0 get no usable
    # bound in clamp mode (B <= 0) and must fall back to the filler rule (k lowest ids of each slab)
    rng = np.random.default_rng(3)
    n_u, n_i, r, k = 300, 3000, 16, 20
    U = rng.integers(-4, 5, (n_u, r)).astype(np.float32) / 8
    V = rng.integers(-4, 5, (n_i, r)).astype(np.float32) / 8
    U[:40] = -np.abs(U[:40]); V[:, :] = np.abs(V)  # rows 0..39: every score <= 0
    for clamp in (False, True):
        idx, sc, _, _ = _bounded_slabs(U, V, k, clamp, [0, 1000, 2100, 3000], 3)
        widx, wsc = oracle_topk(U, V, k, clamp)
        assert np.array_equal(idx, widx) and np.array_equal(sc, wsc)


def test_bounded_scoring_at_scale_matches_unbounded():
    # more tiles per slab than the warm-up, a user count that is not a multiple of the 128-row block
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    from teamoflow_b200 import _abi
    from teamoflow_b200.mf import dist as tdist
    from teamoflow_b200.mf._engine import new_storage
    from teamoflow_b200.mf.matrix_factorization import score_topk
    n_u, n_i, r, k, G_ = 3001, 60_000, 128, 100, 4
    U = new_storage(n_u, r); U[:, :r] = torch.randn(n_u, r, generator=g, device="cuda") / r ** 0.5
    V = new_storage(n_i, r); V[:, :r] = torch.randn(n_i, r, generator=g, device="cuda") / r ** 0.5
    ib, ub = tdist.shard_bounds(n_i, G_), tdist.shard_bounds(n_u, G_)
    want_i, want_s = score_topk(U, V, r, k, False)
    rb = torch.cat([tdist.topk_row_bounds(U, V[ib[q]:ib[q + 1]], r, k, False, ib[q], ub[q], ub[q + 1],
                                          tdist.bound_sample_size(ib[q + 1] - ib[q], n_i, k)) for q in range(G_)]).contiguous()
    lists = [score_topk(U, V[ib[q]:ib[q + 1]], r, k, False, ib[q], row_bound=rb) for q in range(G_)]
    idx_in = torch.stack([l[0] for l in lists]).contiguous()
    sc_in = torch.stack([l[1] for l in lists]).contiguous()
    out_i, out_s = torch.empty_like(want_i), torch.empty_like(want_s)
    _abi.call("tmf_topk_merge", _abi.ptr(idx_in), _abi.ptr(sc_in), G_, n_u, k, _abi.ptr(out_i), _abi.ptr(out_s))
    assert torch.equal(out_i, want_i) and torch.equal(out_s, want_s)


# ------------------------------------------------------------------ peer-memory kernels with local "peers"


def _ptr_array(tensors):
    import ctypes as C
    return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def test_peer_merge_kernel_with_local_peers():
    from teamoflow_b200 import _abi
    rng = np.random.default_rng(8)
    n_u, n_i, r, k, G_ = 257, 5000, 32, 17, 4
    U = (rng.standard_normal((n_u, r)) / 5).astype(np.float32)
    V = (rng.integers(-3, 4, (n_i, r)) / 4).astype(np.float32)
    b = [0, 1250, 2500, 3750, 5000]
    lists = [fused_topk(U, V[a:c], k, False, item_offset=a) for a, c in zip(b[:-1], b[1:])]
    li = [torch.as_tensor(l[0], device="cuda").contiguous() for l in lists]
    ls = [torch.as_tensor(l[1], device="cuda").contiguous() for l in lists]
    outs_i = [torch.full((n_u, k), -7, dtype=torch.int32, device="cuda") for _ in range(2)]
    outs_s = [torch.full((n_u, k), -7.0, dtype=torch.float32, device="cuda") for _ in range(2)]
    lo, n = 31, 150  # a user slice: rows outside it stay untouched
    _abi.call("tmf_topk_merge_peer", _ptr_array(li), _ptr_array(ls), G_, lo, n, k, _ptr_array(outs_i), _ptr_array(outs_s), 2)
    torch.cuda.synchronize()
    widx, wsc = oracle_topk(U, V, k, False)
    for oi, os_ in zip(outs_i, outs_s):
        assert np.array_equal(cpu(oi)[lo:lo + n], widx[lo:lo + n]) and np.array_equal(cpu(os_)[lo:lo + n], wsc[lo:lo + n])
        assert (cpu(oi)[:lo] == -7).all() and (cpu(oi)[lo + n:] == -7).all()


def test_peer_reduce_push_sum_order_and_fused_adam():
    from teamoflow_b200 import _abi
    rng = np.random.default_rng(4)
    G_, n = 3, 4096 + 8
    parts = [torch.as_tensor(rng.standard_normal(n).astype(np.float32), device="cuda") for _ in range(G_)]
    want = cpu(parts[0]).copy()
    for p_ in parts[1:]:
        want = want + cpu(p_)  # rank order, fp32
    dsts = [torch.zeros(n, dtype=torch.float32, device="cuda") for _ in range(G_)]
    off, cnt = 8, 4000
    _abi.call("tmf_peer_reduce_push", _ptr_array(parts), _ptr_array(dsts), G_, 1, off, cnt, -1.0)
    torch.cuda.synchronize()
    for d in dsts:
        assert np.array_equal(cpu(d)[off:off + cnt], want[off:off + cnt]) and not cpu(d)[:off].any() and not cpu(d)[off + cnt:].any()
    # fused Adam step 1: identical bits to tmf_adam1 applied to the summed gradient
    w0 = torch.as_tensor(rng.standard_normal(n).astype(np.float32), device="cuda")
    ws = [w0.clone() for _ in range(G_)]
    _abi.call("tmf_peer_reduce_push", _ptr_array(parts), _ptr_array(ws), G_, 2, 0, n, 0.1)
    ref = w0.clone()
    gsum = torch.as_tensor(want, device="cuda")
    _abi.call("tmf_adam1", _abi.ptr(ref), _abi.ptr(gsum), n, 0.1)
    torch.cuda.synchronize()
    for w in ws:
        assert torch.equal(w, ref)


def test_peer_alloc_export_and_barrier_single_rank():
    import ctypes as C
    from teamoflow_b200 import _abi
    base = C.c_void_p()
    _abi.call_nostream("tmf_peer_alloc", 4096, C.byref(base))
    handle = C.create_string_buffer(64)
    _abi.call_nostream("tmf_ipc_export", base, handle)
    assert any(handle.raw)
    pads = (C.c_void_p * 1)(base.value)
    for epoch in (1, 2, 3):
        _abi.call("tmf_peer_barrier", pads, 1, 0, epoch, 0)
    torch.cuda.synchronize()
    # a rank that never arrives: the barrier gives up after timeout_ms, flags the pad (byte 132 = 1 + missing rank) and
    # returns -- no trap, the CUDA context stays usable (ADVICE r1)
    pads2 = (C.c_void_p * 2)(base.value, base.value + 2048)  # "rank 1" is a second pad nobody signals from
    _abi.call("tmf_peer_barrier", pads2, 2, 0, 7, 50)
    torch.cuda.synchronize()
    from teamoflow_b200.mf.dist import _DevMem
    pad = torch.as_tensor(_DevMem(base.value, 256), device="cuda").view(torch.int32)
    assert int(pad[33]) == 2
    _abi.call("tmf_fill_uniform", _abi.ptr(torch.empty(4, 4, device="cuda")), 4, 4, 4, 1)  # the context is alive
    torch.cuda.synchronize()
    del pad
    _abi.call_nostream("tmf_peer_free", base)


@pytest.mark.gpu
@pytest.mark.parametrize("ld", [64, 128])
def test_gather_rate_aid_reads_every_row(ld):
    """tmf_gather_rate (bench.py's roofline denominator of the user pass) folds exactly the rows it was given."""
    import torch
    from teamoflow_b200 import _abi
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    table = torch.randint(-8, 9, (1000, ld), generator=g, device="cuda").float() / 8     # grid values: any summation order is exact
    idx = torch.randint(0, 1000, (50_003,), generator=g, device="cuda", dtype=torch.int32)
    out = torch.empty(148 * 8 * 256, dtype=torch.float32, device="cuda")
    _abi.call("tmf_gather_rate", _abi.ptr(table), 1000, ld, _abi.ptr(idx), idx.numel(), _abi.ptr(out), out.numel())
    torch.cuda.synchronize()
    assert float(out.double().sum()) == float(table[idx.long()].double().sum())


@pytest.mark.gpu
def test_topk_long_item_sweep_does_not_trip_the_wait_guard():
    """30M items: one user-block sweep lasts > 0.1 s, longer than the poll-count guard of the first mbarrier waits allowed
    (the producer waits a whole sweep for the A tile to be released).  Checked against a chunked fp64 top-k + canonical rerank."""
    from teamoflow_b200.mf._engine import new_storage
    from teamoflow_b200.mf.matrix_factorization import score_topk
    n_u, n_i, r, k = 64, 30_000_000, 8, 10
    g = torch.Generator(device="cuda"); g.manual_seed(77)
    U = new_storage(n_u, r); U[:, :r] = torch.randn(n_u, r, generator=g, device="cuda")
    V = new_storage(n_i, r)
    for a in range(0, n_i, 5_000_000):
        V[a:a + 5_000_000, :r] = torch.randn(5_000_000, r, generator=g, device="cuda")
    idx, sc = score_topk(U, V, r, k, False, 0)
    torch.cuda.synchronize()
    # candidates: top-40 per row by fp64 score over item chunks, then the oracle's canonical score and tie order
    best_s = torch.full((n_u, 40), float("-inf"), dtype=torch.float64, device="cuda")
    best_i = torch.zeros((n_u, 40), dtype=torch.int64, device="cuda")
    Ud = U[:, :r].double()
    for a in range(0, n_i, 2_000_000):
        P = Ud @ V[a:a + 2_000_000, :r].double().T
        s, i = torch.topk(P, 40, dim=1)
        cs, ci = torch.cat([best_s, s], 1), torch.cat([best_i, i + a], 1)
        best_s, sel = torch.topk(cs, 40, dim=1)
        best_i = torch.gather(ci, 1, sel)
        del P
    Uh, cand = cpu(U[:, :r]), best_i.cpu().numpy()
    Vc = cpu(V[best_i.reshape(-1), :r]).reshape(n_u, 40, r)
    got_i, got_s = cpu(idx), cpu(sc)
    for u in range(n_u):
        c = cand[u]
        order0 = np.argsort(c)
        c, Vu = c[order0], Vc[u][order0]
        s = o.canonical_pair_scores(Uh[u:u + 1], Vu, np.zeros(c.size, np.int64), np.arange(c.size))
        order = np.lexsort((c, -s.astype(np.float64)))[:k]
        assert np.array_equal(got_i[u], c[order].astype(np.int32)), u
        assert np.array_equal(got_s[u], s[order]), u
