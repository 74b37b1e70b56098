"""GPU tests of the fused top-k for 128 < k <= 1024 (the kernel's wide configuration) and of the public methods that
now use it.  Indices and scores must be BIT-EXACT against the oracle's canonical scores in stable descending order
(ties -> lower item id)."""
import numpy as np
import pytest
import torch

from oracle import mf_oracle as o
from test_gpu_score import _bounded_slabs, cpu, fused_topk, model_with, oracle_topk

pytestmark = pytest.mark.gpu


def _random(rng, n_u, n_i, r):
    U = (rng.standard_normal((n_u, r)) / np.sqrt(r)).astype(np.float32)
    V = (rng.standard_normal((n_i, r)) / np.sqrt(r)).astype(np.float32)
    return U, V


def _check_rows(U, V, idx, sc, rows, k, clamp=False):
    """oracle on a subset of the rows (the full canonical matrix of a large shape is slow on the CPU)"""
    widx, wsc = oracle_topk(U[rows], V, k, clamp)
    assert np.array_equal(idx[rows], widx) and np.array_equal(sc[rows], wsc)


# every k and r of interest appears with both score modes; 200 users = one full and one partial 128-row block
@pytest.mark.parametrize("k,r,n_i", [(129, 10, 3000), (200, 64, 6000), (256, 128, 9000), (500, 200, 5000), (1000, 64, 20000),
                                     (1024, 128, 12000), (1024, 10, 9000)])
@pytest.mark.parametrize("clamp", [False, True])
def test_wide_topk_random_bit_exact(k, r, n_i, clamp):
    rng = np.random.default_rng(k + r + n_i)
    U, V = _random(rng, 200, n_i, r)
    if clamp:
        U[3] = -np.abs(U[3]); V[:] = np.where(rng.random((n_i, 1)) < 0.5, np.abs(V), V)  # rows with few positive scores
        U[5] = 0.0
    idx, sc = fused_topk(U, V, k, clamp)
    widx, wsc = oracle_topk(U, V, k, clamp)
    assert np.array_equal(idx, widx)
    assert np.array_equal(sc, wsc)
    if clamp:  # an all-zero row: the k lowest ids, score +0
        assert np.array_equal(idx[5], np.arange(k)) and not np.signbit(sc[5]).any() and not sc[5].any()


@pytest.mark.parametrize("n_i", [300, 1024])
def test_wide_topk_k_equals_n_items(n_i):
    rng = np.random.default_rng(n_i)
    U, V = _random(rng, 131, n_i, 32)
    V[17] = V[250]  # an exact tie
    for clamp in (False, True):
        idx, sc = fused_topk(U, V, n_i, clamp)
        widx, wsc = oracle_topk(U, V, n_i, clamp)
        assert np.array_equal(idx, widx) and np.array_equal(sc, wsc)


def test_wide_topk_clamp_nonpositive_rows_get_the_lowest_ids():
    # every score of every row <= 0: the clamped answer is ids 0..k-1 with score 0, whatever the raw order
    rng = np.random.default_rng(7)
    n_i, r, k = 15000, 16, 700
    U = -np.abs(rng.standard_normal((140, r))).astype(np.float32)
    V = np.abs(rng.standard_normal((n_i, r))).astype(np.float32)
    V[:2000] *= 1e-3  # the lowest ids have the best raw scores: the filter would drop every other item early
    idx, sc = fused_topk(U, V, k, True)
    assert np.array_equal(idx, np.tile(np.arange(k, dtype=np.int32), (140, 1)))
    assert not sc.any() and not np.signbit(sc).any()


def test_wide_topk_massive_ties_take_exact_path():
    rng = np.random.default_rng(9)
    U = rng.standard_normal((150, 12)).astype(np.float32)
    V = np.tile(rng.standard_normal((1, 12)).astype(np.float32), (12000, 1))  # every item identical
    for clamp in (False, True):
        idx, sc = fused_topk(U, V, 300, clamp)
        widx, wsc = oracle_topk(U, V, 300, clamp)
        assert np.array_equal(idx, widx) and np.array_equal(sc, wsc)


def test_wide_topk_increasing_scores_force_saturation_rebuilds():
    # every item beats the running threshold: the lists saturate and are rebuilt over and over
    n_i, r = 30000, 8
    U = np.ones((33, r), np.float32)
    U[1] = -1.0
    V = np.tile(np.linspace(-1, 1, n_i, dtype=np.float32)[:, None], (1, r))
    idx, sc = fused_topk(U, V, 1000, False)
    widx, wsc = oracle_topk(U, V, 1000, False)
    assert np.array_equal(idx, widx) and np.array_equal(sc, wsc)


def test_wide_topk_long_sweep():
    rng = np.random.default_rng(13)
    n_u, n_i, r, k = 260, 200_000, 64, 1024
    U, V = _random(rng, n_u, n_i, r)
    V *= rng.uniform(0.5, 2.0, (n_i, 1)).astype(np.float32)
    idx, sc = fused_topk(U, V, k, False)
    _check_rows(U, V, idx, sc, np.r_[0:8, rng.choice(np.arange(8, n_u), 24, replace=False)], k)


@pytest.mark.parametrize("clamp", [False, True])
def test_wide_bounded_item_slabs_merge_equals_single_shot(clamp):
    rng = np.random.default_rng(21)
    n_u, n_i, r, k = 300, 9000, 48, 300
    U = (rng.standard_normal((n_u, r)) / 7).astype(np.float32)
    V = (rng.standard_normal((n_i, r)) / 7).astype(np.float32)
    V[100] = V[8900]  # a tie across slabs
    idx, sc, _, rb = _bounded_slabs(U, V, k, clamp, [0, 3000, 6100, 9000], 3, 0.5)
    widx, wsc = oracle_topk(U, V, k, clamp)
    assert np.array_equal(idx, widx) and np.array_equal(sc, wsc)
    assert np.all(rb <= wsc[:, k - 1])


@pytest.mark.parametrize("k", [200, 500])
def test_wide_k_public_metrics_and_recs(k):
    from scipy import sparse
    rng = np.random.default_rng(k)
    n_u, n_i, r = 150, 2000, 16
    U = (rng.standard_normal((n_u, r)) / 4).astype(np.float32)
    V = (rng.standard_normal((n_i, r)) / 4).astype(np.float32)
    A = np.where(rng.random((n_u, n_i)) < 0.05, rng.choice([-2.0, 1.0, 3.0, 5.0], (n_u, n_i)), 0.0).astype(np.float32)
    A[7] = 0.0
    m = model_with(U, V)
    P = o.canonical_scores(U, V)
    At = torch.as_tensor(A)
    assert np.array_equal(m.retrieve_user_recs(k=k), o.retrieve_user_recs(P, k=k))
    assert np.array_equal(m.retrieve_user_recs(user=9, k=k), o.retrieve_user_recs(P, user=9, k=k))
    for Ain in (At, sparse.csr_matrix(A)):
        np.testing.assert_array_equal(cpu(m.recall_at_k(Ain, k)), o.recall_at_k(P, A, k))
        np.testing.assert_array_equal(cpu(m.precision_at_k(Ain, k)), o.precision_at_k(P, A, k))
    np.testing.assert_allclose(cpu(m.dcg_at_k(At, k)), o.dcg_at_k(P, A, k), rtol=2e-6, atol=1e-6)
    np.testing.assert_allclose(cpu(m.ndcg_at_k(At, k)), o.ndcg_at_k(P, A, k), rtol=5e-6, atol=1e-6)


def test_wide_k_recommend_exact_fallback_and_padding():
    from scipy import sparse
    rng = np.random.default_rng(30)
    n_u, n_i, r, k = 70, 2000, 16, 300
    U = rng.integers(-4, 5, (n_u, r)).astype(np.float32) / 8  # grid values: exact ties, the id tie-break matters
    V = rng.integers(-4, 5, (n_i, r)).astype(np.float32) / 8
    A = np.where(rng.random((n_u, n_i)) < 0.05, 1.0, 0.0).astype(np.float32)
    A[0, :1500] = 1.0               # more seen items among its top-1024 than the list can absorb -> exact fallback
    A[1, :] = 1.0; A[1, 5:105] = 0  # 100 unseen items < k -> padded with -1
    A[2] = 0.0
    m = model_with(U, V)
    P = o.canonical_scores(U, V).astype(np.float64)
    P[A != 0] = -np.inf
    want = o.topk_stable(P, k)
    n_unseen = (A == 0).sum(1)
    want = np.where(np.arange(k)[None, :] < n_unseen[:, None], want, -1)
    for seen in (sparse.csr_matrix(A), torch.as_tensor(A)):
        np.testing.assert_array_equal(cpu(m.recommend(seen, k=k)), want)
    np.testing.assert_array_equal(cpu(m.recommend(sparse.csr_matrix(A), k=k, users=[1, 0, 9])), want[[1, 0, 9]])


def test_wide_k_beyond_the_dense_path():
    # n_users * n_items >= 2^31: the dense score matrix + sort refuse this shape; the fused kernel ranks it
    rng = np.random.default_rng(3)
    n_u, n_i, r, k = 40_000, 60_000, 32, 200
    assert n_u * n_i >= 2 ** 31
    U, V = _random(rng, n_u, n_i, r)
    m = model_with(U, V)
    got = m.retrieve_user_recs(k=k)
    again = m.retrieve_user_recs(k=k)
    assert got.shape == (n_u, k) and np.array_equal(got, again)
    rows = rng.choice(n_u, 64, replace=False)
    assert np.array_equal(got[rows], o.retrieve_user_recs(o.canonical_scores(U[rows], V), k=k))
