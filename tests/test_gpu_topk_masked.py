"""GPU tests of the masked fused top-k (``tmf_score_topk_masked``: the best k UNSEEN items per user) and of what is built on it:
``evaluation.recall_at_k / precision_at_k / ndcg_at_k(exclude=...)`` and ``MatrixFactorization.recommend``.

The oracle is ``oracle.canonical_scores``, clamped first in clamp mode, with the excluded cells at -inf, ranked by
``topk_stable``; slots beyond a row's unseen items are (INT32_MAX, -inf).  Indices and scores must match BIT FOR BIT."""
import numpy as np
import pytest
import torch
from scipy import sparse

from oracle import mf_oracle as o
from test_gpu_score import cpu, fused_topk, model_with

pytestmark = pytest.mark.gpu

PAD = 2 ** 31 - 1


def _random(rng, n_u, n_i, r):
    U = (rng.standard_normal((n_u, r)) / np.sqrt(r)).astype(np.float32)
    V = (rng.standard_normal((n_i, r)) / np.sqrt(r)).astype(np.float32)
    return U, V


def _csr(mask, item_offset=0):
    ptr = np.zeros(mask.shape[0] + 1, np.int32)
    ptr[1:] = np.cumsum(mask.sum(1))
    return ptr, (np.nonzero(mask)[1] + item_offset).astype(np.int32)


def _csr_from_lists(lists):
    ptr = np.zeros(len(lists) + 1, np.int32)
    ptr[1:] = np.cumsum([len(x) for x in lists])
    idx = np.concatenate([np.sort(np.asarray(x, np.int64)) for x in lists]).astype(np.int32) if ptr[-1] else np.zeros(0, np.int32)
    return ptr, idx


def masked_topk(U, V, k, clamp, ptr, idx, item_offset=0):
    from teamoflow_b200.mf._engine import new_storage
    from teamoflow_b200.mf.evaluation import score_topk_masked
    r = U.shape[1]
    Us = new_storage(U.shape[0], r, torch.as_tensor(U, device="cuda"))
    Vs = new_storage(V.shape[0], r, torch.as_tensor(V, device="cuda"))
    i, s = score_topk_masked(Us, Vs, r, k, clamp, torch.as_tensor(ptr, device="cuda"), torch.as_tensor(idx, device="cuda"),
                             item_offset)
    torch.cuda.synchronize()
    return cpu(i), cpu(s)


def oracle_masked(U, V, k, clamp, ptr, idx, rows=None, item_offset=0):
    rows = np.arange(U.shape[0]) if rows is None else np.asarray(rows)
    n_i = V.shape[0]
    P = o.canonical_scores(U[rows], V)
    if clamp:
        P = np.where(P > 0, P, np.float32(0))
    P = P.astype(np.float32)
    n_unseen = np.empty(len(rows), np.int64)
    for j, u in enumerate(rows):
        c = idx[ptr[u]:ptr[u + 1]].astype(np.int64) - item_offset
        c = c[(c >= 0) & (c < n_i)]
        P[j, c] = -np.inf
        n_unseen[j] = n_i - c.size
    widx = o.topk_stable(P, k)
    wsc = np.take_along_axis(P, widx.astype(np.int64), 1)
    pad = np.arange(k)[None, :] >= n_unseen[:, None]
    widx = np.where(pad, PAD, widx + item_offset).astype(np.int32)
    wsc = np.where(pad, np.float32(-np.inf), wsc).astype(np.float32)
    return widx, wsc


def _check(U, V, k, clamp, ptr, idx, rows=None):
    got_i, got_s = masked_topk(U, V, k, clamp, ptr, idx)
    widx, wsc = oracle_masked(U, V, k, clamp, ptr, idx, rows)
    if rows is not None:
        got_i, got_s = got_i[rows], got_s[rows]
    assert np.array_equal(got_i, widx)
    assert np.array_equal(got_s, wsc)
    if clamp:
        assert not np.signbit(got_s[got_s == 0]).any()
    return got_i, got_s


def _top_n_by_score(U, V, n):
    """each row's own best n items by canonical score (what training makes a user's seen set look like)"""
    P = o.canonical_scores(U, V).astype(np.float64)
    return [o.topk_stable(P[u], n) for u in range(U.shape[0])]


@pytest.mark.parametrize("k", [1, 10, 128, 129, 500, 1024])
@pytest.mark.parametrize("r", [10, 64, 128])
@pytest.mark.parametrize("clamp", [False, True])
def test_masked_topk_random_bit_exact(k, r, clamp):
    rng = np.random.default_rng(k * 7 + r)
    U, V = _random(rng, 200, 3000, r)
    if clamp:
        U[3] = -np.abs(U[3]); V[:] = np.where(rng.random((3000, 1)) < 0.5, np.abs(V), V)  # rows with few positive scores
        U[5] = 0.0
    mask = rng.random((200, 3000)) < 0.05
    _check(U, V, k, clamp, *_csr(mask))


@pytest.mark.parametrize("n_seen", [50, 300, 3000])
@pytest.mark.parametrize("k", [10, 129])
@pytest.mark.parametrize("clamp", [False, True])
def test_masked_topk_trained_like_rows(n_seen, k, clamp):
    # the seen set is each row's own top-n_seen: every item above the unseen top-k is excluded, so a threshold built from
    # listed seen items would drop the answer
    rng = np.random.default_rng(n_seen + k)
    U, V = _random(rng, 150, 8000, 32)
    _check(U, V, k, clamp, *_csr_from_lists(_top_n_by_score(U, V, n_seen)))


@pytest.mark.parametrize("k", [100, 300])
@pytest.mark.parametrize("clamp", [False, True])
def test_masked_topk_special_rows(k, clamp):
    rng = np.random.default_rng(k)
    n_u, n_i = 140, 9000
    U, V = _random(rng, n_u, n_i, 24)
    mask = rng.random((n_u, n_i)) < 0.02
    mask[0] = False; mask[0, :5001] = True    # fewer than k entries listed at the first rebuild
    mask[1] = True; mask[1, [7, 900, 4000, 8000, 8999]] = False  # 5 unseen items: padded
    mask[2] = True                             # nothing unseen: all padding
    mask[3] = False                            # nothing seen
    mask[130, 1::2] = True                     # a partial user block
    got_i, got_s = _check(U, V, k, clamp, *_csr(mask))
    assert (got_i[2] == PAD).all() and np.isneginf(got_s[2]).all()
    assert (got_i[1, 5:] == PAD).all() and np.array_equal(np.sort(got_i[1, :5]), [7, 900, 4000, 8000, 8999])


@pytest.mark.parametrize("k", [50, 700])
def test_masked_topk_clamp_fillers_are_the_lowest_unseen_ids(k):
    rng = np.random.default_rng(k)
    n_u, n_i, r = 130, 15000, 16
    U = -np.abs(rng.standard_normal((n_u, r))).astype(np.float32)
    V = np.abs(rng.standard_normal((n_i, r))).astype(np.float32)  # every score <= 0
    U[7] = -U[7]                                                   # one row with every score > 0
    mask = rng.random((n_u, n_i)) < 0.05
    mask[:, 0:200:2] = True                                        # the lowest ids are seen
    got_i, got_s = _check(U, V, k, True, *_csr(mask))
    for u in range(n_u):
        if u != 7:
            assert np.array_equal(got_i[u], np.nonzero(~mask[u])[0][:k])
            assert not got_s[u].any() and not np.signbit(got_s[u]).any()


@pytest.mark.parametrize("k", [50, 300])
@pytest.mark.parametrize("clamp", [False, True])
def test_masked_topk_identical_items_take_exact_path(k, clamp):
    rng = np.random.default_rng(9 + k)
    U = rng.standard_normal((150, 12)).astype(np.float32)
    V = np.tile(rng.standard_normal((1, 12)).astype(np.float32), (12000, 1))  # every item identical
    mask = rng.random((150, 12000)) < 0.05
    mask[0, :2000] = True
    mask[1] = True; mask[1, 11990:] = False  # 10 unseen items
    mask[2] = True
    _check(U, V, k, clamp, *_csr(mask))


@pytest.mark.parametrize("k", [50, 300])
def test_masked_topk_repeated_excluded_ids(k):
    # the fused path and the exact path (identical items) must not count a repeated id twice
    rng = np.random.default_rng(k)
    for same in (False, True):
        U, V = _random(rng, 140, 6000, 12)
        if same:
            V[:] = V[0]
        mask = rng.random((140, 6000)) < 0.05
        mask[1] = True; mask[1, 5990:] = False  # 10 unseen items
        ptr, idx = _csr(mask)
        rep = np.repeat(np.arange(idx.size), 1 + (np.arange(idx.size) % 3 == 0))  # every third id twice
        rows = np.repeat(np.arange(140), np.diff(ptr))[rep]
        ptr2 = np.zeros(141, np.int32); ptr2[1:] = np.cumsum(np.bincount(rows, minlength=140))
        got = masked_topk(U, V, k, False, ptr2, idx[rep])
        want = oracle_masked(U, V, k, False, ptr, idx)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


@pytest.mark.parametrize("k", [100, 1000])
def test_masked_topk_long_sweep_with_top_seen(k):
    rng = np.random.default_rng(k)
    U, V = _random(rng, 130, 200_000, 32)
    _check(U, V, k, False, *_csr_from_lists(_top_n_by_score(U, V, 2000)))


@pytest.mark.parametrize("k", [100, 300])
@pytest.mark.parametrize("clamp", [False, True])
def test_masked_item_slabs_merge_equals_single_shot(k, clamp):
    from teamoflow_b200 import _abi
    rng = np.random.default_rng(k + clamp)
    n_u, n_i = 150, 7000
    U, V = _random(rng, n_u, n_i, 20)
    if clamp:
        U[4] = -np.abs(U[4]); V[:] = np.abs(V)  # row 4: every score <= 0, the fillers come from the first slab
    mask = rng.random((n_u, n_i)) < 0.1
    mask[4, :300] = True
    mask[5] = True; mask[5, 6000:6050] = False  # unseen items only in the last slab
    ptr, idx = _csr(mask)
    bounds = [0, 2500, 2600, n_i]  # the middle slab holds fewer than k items of some rows
    outs = [masked_topk(U, V[a:b], min(k, b - a), clamp, ptr, idx, item_offset=a) for a, b in zip(bounds[:-1], bounds[1:])]
    pad_i = lambda x: np.pad(x, ((0, 0), (0, k - x.shape[1])), constant_values=PAD)  # noqa: E731
    pad_s = lambda x: np.pad(x, ((0, 0), (0, k - x.shape[1])), constant_values=-np.inf)  # noqa: E731
    idx_in = torch.as_tensor(np.stack([pad_i(i) for i, _ in outs]), device="cuda").contiguous()
    sc_in = torch.as_tensor(np.stack([pad_s(s) for _, s in outs]), device="cuda").contiguous()
    out_i = torch.empty(n_u, k, dtype=torch.int32, device="cuda")
    out_s = torch.empty(n_u, k, dtype=torch.float32, device="cuda")
    _abi.call("tmf_topk_merge", _abi.ptr(idx_in), _abi.ptr(sc_in), len(outs), n_u, k, _abi.ptr(out_i), _abi.ptr(out_s))
    want_i, want_s = masked_topk(U, V, k, clamp, ptr, idx)
    assert np.array_equal(cpu(out_i), want_i) and np.array_equal(cpu(out_s), want_s)
    widx, wsc = oracle_masked(U, V, k, clamp, ptr, idx)
    assert np.array_equal(want_i, widx) and np.array_equal(want_s, wsc)


@pytest.mark.parametrize("k", [50, 500])
@pytest.mark.parametrize("clamp", [False, True])
def test_masked_topk_empty_exclusion_equals_unmasked(k, clamp):
    rng = np.random.default_rng(k)
    U, V = _random(rng, 300, 5000, 48)
    ptr, idx = np.zeros(301, np.int32), np.zeros(0, np.int32)
    got_i, got_s = masked_topk(U, V, k, clamp, ptr, idx)
    want_i, want_s = fused_topk(U, V, k, clamp)
    assert np.array_equal(got_i, want_i) and np.array_equal(got_s, want_s)


def test_masked_topk_is_deterministic():
    rng = np.random.default_rng(3)
    U, V = _random(rng, 400, 20000, 64)
    ptr, idx = _csr(rng.random((400, 20000)) < 0.03)
    for k, clamp in ((64, False), (600, True)):
        a = masked_topk(U, V, k, clamp, ptr, idx)
        b = masked_topk(U, V, k, clamp, ptr, idx)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("k", [100, 1000])
def test_masked_topk_beyond_the_dense_path_sampled_rows(k):
    # 40,000 x 60,000 = 2.4e9 scores: more than the dense canonical path takes
    rng = np.random.default_rng(k)
    n_u, n_i = 40_000, 60_000
    U, V = _random(rng, n_u, n_i, 64)
    lens = rng.integers(0, 400, n_u)
    lists = [np.unique(rng.integers(0, n_i, n)) for n in lens]
    rows = np.sort(rng.choice(n_u, 64, replace=False))
    lists[rows[0]] = np.arange(5000)  # one sampled row with its first 5000 ids seen
    _check(U, V, k, False, *_csr_from_lists(lists), rows=rows)


# ---------------------------------------------------------------------- evaluation and recommend


def _doubled(table):
    """scipy CSR with every non-zero cell of ``table`` stored twice, next to each other (not in canonical format)"""
    r, c = np.nonzero(table)
    v = np.asarray(table)[r, c].astype(np.float32)
    ptr = np.r_[0, np.cumsum(2 * np.count_nonzero(table, axis=1))]
    m = sparse.csr_matrix((np.repeat(v, 2), np.repeat(c, 2), ptr), shape=table.shape)
    assert m.nnz == 2 * r.size
    return m


def _split(rng, n_u, n_i, density):
    from teamoflow_b200.mf import input_utils as iu
    cells = np.nonzero(rng.random((n_u, n_i)) < density)
    vals = rng.integers(1, 6, cells[0].size).astype(np.float64)
    rows = [[int(u), int(i), float(v)] for u, i, v in zip(cells[0], cells[1], vals)]
    train, test = iu.mask_train_test_split(rows, n_u, n_i, return_indices=False)
    return train, test


def _oracle_metrics(U, V, A, train, k):
    A = np.asarray(A, np.float32)
    ptr, idx = _csr(train != 0)
    kk = min(k, V.shape[0])
    ci, _ = oracle_masked(U, V, kk, True, ptr, idx)
    hit = np.array([np.count_nonzero(A[u, ci[u][ci[u] != PAD]]) for u in range(A.shape[0])], np.float32)
    rel = np.count_nonzero(A > 0, axis=1).astype(np.float32)
    recall = hit[rel != 0] / rel[rel != 0]
    precision = hit[rel != 0] / np.float32(k)
    ri, _ = oracle_masked(U, V, kk, False, ptr, idx)
    disc = (np.log1p(np.arange(1, kk + 1, dtype=np.float32)) / np.log(np.float32(2.0))).astype(np.float32)
    gains = np.array([[A[u, i] if i != PAD else 0.0 for i in ri[u]] for u in range(A.shape[0])], np.float32)
    dcg = ((np.power(np.float32(2.0), gains) - np.float32(1.0)) / disc[None, :]).sum(axis=1, dtype=np.float32)
    P = o.canonical_scores(U, V)
    with np.errstate(all="ignore"):
        ndcg = dcg / o.idcg_at_k(P, A, k)
    return recall, precision, ndcg[np.count_nonzero(A, axis=1) > 0]


@pytest.mark.parametrize("k", [10, 200, 1500])
def test_evaluation_with_exclude_matches_oracle(k):
    from teamoflow_b200.mf import evaluation as ev
    from teamoflow_b200.mf._tensors import SparseInteractions
    rng = np.random.default_rng(k)
    n_u, n_i, r = 300, 2000, 16
    U, V = _random(rng, n_u, n_i, r)
    train, test = _split(rng, n_u, n_i, 0.04)
    Ut = train.toarray().astype(np.float32)
    m = model_with(U, V)
    want_rec, want_prec, want_ndcg = _oracle_metrics(U, V, test.toarray(), Ut, k)
    coo = train.tocoo()
    excl = [Ut, train, SparseInteractions(np.stack([coo.row, coo.col], 1), coo.data.astype(np.float32), (n_u, n_i)), _doubled(Ut)]
    for ex in excl:
        np.testing.assert_array_equal(cpu(ev.recall_at_k(m, test, k, exclude=ex)), want_rec)
        np.testing.assert_array_equal(cpu(ev.precision_at_k(m, test, k, exclude=ex)), want_prec)
        np.testing.assert_allclose(cpu(ev.ndcg_at_k(m, test, k, exclude=ex)), want_ndcg, rtol=5e-6, atol=1e-6)


@pytest.mark.parametrize("k", [10, 300])
def test_evaluation_without_exclude_equals_model_methods(k):
    from teamoflow_b200.mf import evaluation as ev
    rng = np.random.default_rng(k)
    U, V = _random(rng, 250, 1500, 16)
    m = model_with(U, V)
    _, test = _split(rng, 250, 1500, 0.05)
    for pr in (False, True):
        assert torch.equal(ev.recall_at_k(m, test, k, preserve_rows=pr), m.recall_at_k(test, k, preserve_rows=pr))
        assert torch.equal(ev.precision_at_k(m, test, k, preserve_rows=pr), m.precision_at_k(test, k, preserve_rows=pr))
        assert torch.equal(ev.ndcg_at_k(m, test, k, preserve_rows=pr), m.ndcg_at_k(test, k, preserve_rows=pr))


@pytest.mark.parametrize("k", [10, 500])
def test_recommend_trained_like_rows(k):
    rng = np.random.default_rng(k)
    n_u, n_i = 160, 6000
    U, V = _random(rng, n_u, n_i, 32)
    lists = _top_n_by_score(U, V, 400)  # every user's best 400 items are seen
    mask = np.zeros((n_u, n_i), bool)
    for u, l in enumerate(lists):
        mask[u, l] = True
    mask[0] = True; mask[0, :7] = False  # 7 unseen items: -1 padding
    m = model_with(U, V)
    ptr, idx = _csr(mask)
    widx, _ = oracle_masked(U, V, k, False, ptr, idx)
    want = np.where(widx == PAD, -1, widx)
    A = sparse.csr_matrix(mask.astype(np.float32))
    np.testing.assert_array_equal(cpu(m.recommend(A, k=k)), want)
    # the same table with every cell stored twice (a scipy matrix not in canonical format)
    np.testing.assert_array_equal(cpu(m.recommend(_doubled(mask), k=k)), want)
    np.testing.assert_array_equal(cpu(m.recommend(A, k=k, users=[0, 5, 159])), want[[0, 5, 159]])
