"""Held-out evaluation: recall, precision and NDCG at k with chosen items (a user's training items) removed from every
user's ranking, and the masked fused top-k behind them and behind ``MatrixFactorization.recommend``.

The split ``input_utils.mask_train_test_split`` produces is used by fitting on the train table and measuring on the test
table with the train items excluded: ``recall_at_k(model, test, k, exclude=train)``.  The model's own ``recall_at_k`` ranks
every item, like the reference; on a trained model the train items fill the top of each list, so the held-out numbers would
mostly count how many train items outrank each test item.

Without ``exclude`` the functions here return exactly what the model's methods return.  The metric arithmetic after the
top-k (hits / relevant, the ``preserve_rows`` masking, the DCG / IDCG combination) exists once, in this module; the model's
methods call it.
"""
import torch

from .. import _abi
from . import _engine as eng
from .matrix_factorization import TOPK_FUSED_MAX_K, _csr_of, _rank_rows

# item id of a padding slot: a row with fewer than k unseen items ends in (PAD_ID, -inf) entries
PAD_ID = 0x7FFFFFFF


def score_topk_masked(U, V, r, k, clamp, ex_ptr, ex_idx, item_offset=0):
    """Fused tcgen05 ``U V^T`` + per-row top-k over each row's UNSEEN items (``tmf_score_topk_masked``).  ``U``/``V`` are
    padded storages; ``ex_ptr`` [n_u + 1] / ``ex_idx`` (int32, on the device) the CSR of the global item ids to exclude, each
    row sorted ascending with distinct ids.  Returns ``(idx int32 [n_u, k], score fp32 [n_u, k])``, ranked by (score desc,
    id asc) -- clamped scores with ``clamp`` -- and padded with ``(PAD_ID, -inf)`` where a row has fewer than k unseen items."""
    n_u, n_i = U.shape[0], V.shape[0]
    idx = torch.empty(n_u, k, dtype=torch.int32, device=U.device)
    score = torch.empty(n_u, k, dtype=torch.float32, device=U.device)
    ws_bytes = _abi.query("tmf_score_topk_ws_bytes", n_u, n_i, r, k)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=U.device)
    _abi.call("tmf_score_topk_masked", _abi.ptr(U), n_u, _abi.ptr(V), n_i, r, U.shape[1], k, int(bool(clamp)), int(item_offset),
              _abi.ptr(ex_ptr), _abi.ptr(ex_idx), _abi.ptr(idx), _abi.ptr(score), _abi.ptr(ws), ws_bytes)
    return idx, score


def masked_topk(U, V, r, k, clamp, ex_ptr, ex_idx):
    """Top-``min(k, n_items)`` item ids per row of ``U`` over its unseen items, ``PAD_ID`` padding.  The fused kernel up to
    ``TOPK_FUSED_MAX_K``; beyond it (full rankings) exact dense blocks of at most 2^27 scores: canonical scores, clamped
    first in clamp mode, excluded cells at -inf, stable ranking."""
    n_u, n_i = U.shape[0], V.shape[0]
    k = min(int(k), n_i)
    if k <= TOPK_FUSED_MAX_K:
        return score_topk_masked(U, V, r, k, clamp, ex_ptr, ex_idx)[0]
    dev = U.device
    out = torch.empty(n_u, k, dtype=torch.int32, device=dev)
    row_nnz = (ex_ptr[1:] - ex_ptr[:-1]).to(torch.int64)
    block = max(1, min(4096, (1 << 27) // n_i))
    for b0 in range(0, n_u, block):
        b1 = min(n_u, b0 + block)
        Ub = U[b0:b1].contiguous()
        P = torch.empty(b1 - b0, n_i, dtype=torch.float32, device=dev)
        _abi.call("tmf_predict_dense", _abi.ptr(Ub), b1 - b0, _abi.ptr(V), n_i, r, U.shape[1], _abi.ptr(P))
        if clamp:  # tf.where(p > 0, p, 0.0): the ranking key, before the excluded cells leave the ranking
            P = torch.where(P > 0, P, torch.zeros_like(P))
        c = row_nnz[b0:b1]
        rr = torch.repeat_interleave(torch.arange(b1 - b0, device=dev), c)
        P[rr, ex_idx[int(ex_ptr[b0]):int(ex_ptr[b1])].long()] = float("-inf")
        order = _rank_rows(P, clamp=False)[:, :k]
        unseen = (n_i - torch.isneginf(P).sum(1)).clamp(max=k)  # a repeated excluded id counts once
        out[b0:b1] = torch.where(torch.arange(k, device=dev)[None, :] < unseen[:, None], order, torch.full_like(order, PAD_ID))
    return out


# ---------------------------------------------------------------------- metric arithmetic after the top-k


def hits_relevant(topk, a_csr):
    """hits[u] = #{i in topk[u] : A[u, i] != 0} (padding never hits), relevant[u] = #{i : A[u, i] > 0} (``tmf_metrics_hits``)."""
    a_ptr, a_idx, a_val = a_csr
    n_u = topk.shape[0]
    hits = torch.empty(n_u, dtype=torch.float32, device=topk.device)
    relevant = torch.empty(n_u, dtype=torch.float32, device=topk.device)
    _abi.call("tmf_metrics_hits", _abi.ptr(topk), n_u, topk.shape[1], _abi.ptr(a_ptr), _abi.ptr(a_idx), _abi.ptr(a_val),
              _abi.ptr(hits), _abi.ptr(relevant))
    return hits, relevant


def recall_from_hits(hits, relevant, preserve_rows):
    if not preserve_rows:
        m = relevant != 0.0
        return hits[m] / relevant[m]
    recall = hits / relevant
    return torch.where(torch.isnan(recall), torch.zeros_like(recall), recall)


def precision_from_hits(hits, relevant, k, preserve_rows):
    kk = torch.full_like(hits, float(k))  # tensor / tensor is a true IEEE division (tensor / scalar multiplies by 1/k)
    if not preserve_rows:
        m = relevant != 0.0
        return hits[m] / kk[m]
    return hits / kk


def dcg_of(topk, a_csr):
    """dcg[u] = sum_q (2^A[u, topk[u, q]] - 1) / log2(q + 2) (``tmf_dcg``); a padding slot adds 0."""
    a_ptr, a_idx, a_val = a_csr
    n_u = topk.shape[0]
    dcg = torch.empty(n_u, dtype=torch.float32, device=topk.device)
    _abi.call("tmf_dcg", _abi.ptr(topk), n_u, topk.shape[1], _abi.ptr(a_ptr), _abi.ptr(a_idx), _abi.ptr(a_val), _abi.ptr(dcg))
    return dcg


def ndcg_from_dcg(dcg, idcg, row_nnz, preserve_rows):
    ndcg = dcg / idcg
    if not preserve_rows:
        return ndcg[row_nnz > 0]
    return torch.where(~torch.isnan(ndcg), ndcg, torch.zeros_like(ndcg))


# ---------------------------------------------------------------------- held-out metrics


def exclusion_csr(table, n_users, n_items):
    """CSR ``(ptr, idx)`` of the non-zero cells of an interaction table, each row sorted with distinct ids as
    ``tmf_score_topk_masked`` takes it (a table may hold a cell twice, e.g. a scipy matrix not in canonical format)."""
    ptr, idx, _ = _csr_of(table, n_users, n_items, drop_zeros=True)
    if idx.numel() < 2:
        return ptr, idx
    rows = torch.repeat_interleave(torch.arange(n_users, device=idx.device), (ptr[1:] - ptr[:-1]).to(torch.int64))
    keep = torch.ones_like(idx, dtype=torch.bool)
    keep[1:] = (idx[1:] != idx[:-1]) | (rows[1:] != rows[:-1])
    if bool(keep.all()):
        return ptr, idx
    dedup = torch.zeros(n_users + 1, dtype=torch.int64, device=idx.device)
    dedup[1:] = torch.cumsum(torch.bincount(rows[keep], minlength=n_users), 0)
    return dedup.to(torch.int32), idx[keep].contiguous()


def _ranking(model, k, clamp, exclude):
    if exclude is None:
        return model._topk(k, clamp=clamp)
    n_u, n_i = model.user_embedding.shape[0], model.item_embedding.shape[0]
    ex_ptr, ex_idx = exclusion_csr(exclude, n_u, n_i)
    return masked_topk(eng.storage_of(model.user_embedding), eng.storage_of(model.item_embedding), model.n_components, k, clamp,
                       ex_ptr, ex_idx)


def _a_csr(model, A):
    return _csr_of(A, model.user_embedding.shape[0], model.item_embedding.shape[0])


def recall_at_k(model, A, k=10, exclude=None, preserve_rows=False):
    """``model.recall_at_k(A, k, preserve_rows)`` with the non-zero cells of ``exclude`` (an interaction table: dense, scipy,
    torch sparse or ``SparseInteractions``) removed from every user's ranking.  Slots a user cannot fill are misses;
    ``relevant`` still counts the positive cells of ``A``."""
    hits, relevant = hits_relevant(_ranking(model, k, True, exclude), _a_csr(model, A))
    return recall_from_hits(hits, relevant, preserve_rows)


def precision_at_k(model, A, k=10, exclude=None, preserve_rows=False):
    """``model.precision_at_k`` with ``exclude`` as in ``recall_at_k``; hits are still divided by k, like the reference."""
    hits, relevant = hits_relevant(_ranking(model, k, True, exclude), _a_csr(model, A))
    return precision_from_hits(hits, relevant, k, preserve_rows)


def ndcg_at_k(model, A, k=10, exclude=None, preserve_rows=False):
    """``model.ndcg_at_k`` with ``exclude`` as in ``recall_at_k``: DCG over the masked ranking of raw scores (a padding slot
    adds 0), IDCG from ``A`` as before."""
    dcg = dcg_of(_ranking(model, k, False, exclude), _a_csr(model, A))
    idcg, row_nnz = model._idcg(A, k)
    return ndcg_from_dcg(dcg, idcg, row_nnz, preserve_rows)
