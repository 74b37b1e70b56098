"""CPU checks that the multi-batch top-k shapes of test_gpu_topk_batches.py really span several user batches.

score_topk_impl (score_topk.cu) ranks the users in batches of user blocks of 128 rows: UB_BATCH blocks per main-kernel and
rerank launch for k <= 128, UB_BATCH_W blocks for 128 < k <= 1024.  Only the candidate lists are sized by the batch, so
tmf_score_topk_ws_bytes grows by one 128-row candidate slab per extra 128 users until the users fill a batch, and by the
per-user terms alone after that.  The batch size is recovered from that query (no GPU needed): if UB_BATCH or UB_BATCH_W
changes, this file fails instead of the GPU sweep silently falling back to a single batch.
"""
import functools

import pytest

BM = 128             # users per block (score_topk.cu: BM)
UB_BATCH = 2048      # blocks per launch, k <= 128 (score_topk.cu: UB_BATCH)
UB_BATCH_W = 592     # blocks per launch, 128 < k <= 1024 (score_topk.cu: UB_BATCH_W)
NARROW_MAX_K = 128
BATCH_USERS = BM * UB_BATCH      # 262,144
BATCH_USERS_W = BM * UB_BATCH_W  # 75,776


def n_batches(n_users, k):
    """main-kernel (and rerank) launches of one tmf_score_topk* call"""
    blocks = -(-n_users // BM)
    return -(-blocks // (UB_BATCH if k <= NARROW_MAX_K else UB_BATCH_W))


def batch_users(k):
    return BATCH_USERS if k <= NARROW_MAX_K else BATCH_USERS_W


def straddles(n_users, k):
    """several batches, or exactly one full batch (the boundary from the other side)"""
    return n_batches(n_users, k) >= 2 or n_users == batch_users(k)


# The GPU cases.  test_gpu_topk_batches.py parametrizes its tests from these lists and test_gpu_cases_straddle_the_batches
# checks every one of them.  Each family's data set is built at its n_users; smaller cases rank a prefix of its rows.
FAMILIES = {
    "narrow": dict(n_users=262_344, n_items=2_000, r=32),
    "narrow3": dict(n_users=525_288, n_items=300, r=16),
    "wide": dict(n_users=80_000, n_items=6_000, r=64),
    "ml20m": dict(n_users=138_493, n_items=26_744, r=64),  # the ML-20M shape
}
# (family, n_users, k, clamp)
PLAIN = [("narrow", n, k, c) for n, ks in ((262_144, (10, 128)), (262_145, (10,)), (262_344, (10, 128))) for k in ks
         for c in (False, True)] + [("narrow3", 525_288, 10, False)] + \
        [("wide", n, 200, c) for n in (75_776, 75_777) for c in (False, True)] + \
        [("ml20m", 138_493, k, c) for k in (200, 1024) for c in (False, True)]
MASKED = [("narrow", 262_344, 100, c) for c in (False, True)] + \
         [("ml20m", 138_493, k, c) for k in (200, 1024) for c in (False, True)]
# (family, n_users, k, item slab bounds, clamp)
BOUNDED = [("wide", 80_000, 300, (0, 2000, 4100, 6000), c) for c in (False, True)] + \
          [("narrow", 262_344, 25, (0, 700, 1400, 2000), c) for c in (False, True)]
# (family, k, clamp, masked), over the whole family
INVARIANCE = [("narrow", 10, False, False), ("ml20m", 1024, True, False), ("ml20m", 200, False, True)]
LAUNCHES = [("narrow3", 10, False, False), ("narrow", 100, True, True), ("ml20m", 200, False, False),
            ("ml20m", 1024, True, True)]


def gpu_cases():
    """(test, family, n_users, k) of every GPU case"""
    return ([("plain", f, n, k) for f, n, k, _ in PLAIN] + [("masked", f, n, k) for f, n, k, _ in MASKED] +
            [("bounded", f, n, k) for f, n, k, _, _ in BOUNDED] +
            [(t, f, FAMILIES[f]["n_users"], k) for t, cases in (("invariance", INVARIANCE), ("launches", LAUNCHES))
             for f, k, _, _ in cases])


def _ws(n_users, n_items, r, k):
    from teamoflow_b200 import _abi
    return _abi.query("tmf_score_topk_ws_bytes", n_users, n_items, r, k)


@functools.lru_cache(maxsize=None)
def batch_users_from_workspace(n_items, r, k):
    """smallest multiple n of 128 at which 128 more users no longer add a candidate slab (>= 2 MB): the users per batch"""
    grows = lambda m: _ws(BM * (m + 1), n_items, r, k) - _ws(BM * m, n_items, r, k) >= 1 << 20  # noqa: E731
    lo, hi = 1, 1 << 16  # grows(lo) holds, grows(hi) does not
    assert grows(lo) and not grows(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if grows(mid):
            lo = mid
        else:
            hi = mid
    return BM * hi


@pytest.mark.parametrize("k,want", [(1, BATCH_USERS), (10, BATCH_USERS), (128, BATCH_USERS), (129, BATCH_USERS_W),
                                    (200, BATCH_USERS_W), (1024, BATCH_USERS_W)])
def test_batch_size_recovered_from_the_workspace(k, want):
    assert batch_users_from_workspace(2_000, 32, k) == want
    # one candidate slab per 128 users below the batch size: 128 rows x 2048 (narrow) or 8192 (wide) slots x 8 bytes
    slab = BM * (2048 if k <= NARROW_MAX_K else 8192) * 8
    per_user = _ws(want + BM, 2_000, 32, k) - _ws(want, 2_000, 32, k)  # packed operands, norms, counts (256-byte aligned)
    assert per_user < 64 << 10
    assert 0 <= _ws(want, 2_000, 32, k) - _ws(want - BM, 2_000, 32, k) - slab < 64 << 10


@pytest.mark.parametrize("case", gpu_cases(), ids=lambda c: f"{c[0]}-{c[1]}-{c[2]}-k{c[3]}")
def test_gpu_cases_straddle_the_batches(case):
    _, name, n_users, k = case
    shape = FAMILIES[name]
    assert n_users <= shape["n_users"]
    per_batch = batch_users_from_workspace(shape["n_items"], shape["r"], k)
    got = -(-n_users // per_batch)
    assert got == n_batches(n_users, k), f"n_users {n_users}, k {k}: {got} batches of {per_batch} users"
    assert got >= 2 or n_users == per_batch, f"n_users {n_users}, k {k}: one batch of {per_batch} users"
    assert straddles(n_users, k)


def test_gpu_cases_reach_three_batches_and_both_configurations():
    got = {(n_batches(n, k), k > NARROW_MAX_K) for _, _, n, k in gpu_cases()}
    assert {(1, False), (2, False), (3, False), (1, True), (2, True)} <= got
