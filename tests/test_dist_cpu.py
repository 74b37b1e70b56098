"""world_size-2 gloo tests (CPU) of the multi-GPU plumbing: shard bounds, the all-reduce hooks of
user-sharded training and the all-gather + merge of item-sharded top-k.  The compute legs are played by the
oracle (test infrastructure) so that only the host-side sharding / collective logic is under test."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import mf_oracle as o
from teamoflow_b200.mf import dist as tdist


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _spawn(fn, world=2):
    port = _free_port()
    mp.spawn(_entry, args=(world, port, fn), nprocs=world, join=True)


def _entry(rank, world, port, fn):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        fn(rank, world)
    finally:
        dist.destroy_process_group()


def test_shard_bounds():
    assert tdist.shard_bounds(10, 3) == [0, 4, 7, 10]
    assert tdist.shard_bounds(2, 4) == [0, 1, 2, 2, 2]
    b = tdist.balanced_user_bounds([100, 1, 1, 1, 100, 1, 1, 95], 2)
    assert b[0] == 0 and b[-1] == 8 and 1 <= b[1] <= 5
    lens = np.random.default_rng(0).integers(0, 50, 1000)
    b = tdist.balanced_user_bounds(lens, 4)
    per = [lens[b[i]:b[i + 1]].sum() for i in range(4)]
    assert max(per) - min(per) <= 2 * lens.max()


class _FakeTower:
    def __init__(self, kind, grads, params):
        self.kind, self.grads, self._p = kind, grads, params

    def trainables(self):
        return self._p


def _problem():
    rng = np.random.default_rng(3)
    n_u, n_i, r, S = 40, 30, 6, 5
    (rows, cols, vals), _ = o.generate_random_interaction(n_u, n_i, density=0.2, random_state=4)
    U = o.uniform_initializer(n_u, r, rng).astype(np.float64)
    V = o.uniform_initializer(n_i, r, rng).astype(np.float64)
    samp = np.stack([rng.choice(n_i, S, replace=False) for _ in range(n_u)])
    return n_u, n_i, r, S, rows, cols, vals.astype(np.float64), U, V, samp


def _dp_training(rank, world):
    n_u, n_i, r, S, rows, cols, vals, U, V, samp = _problem()
    full = o.train_step_sparse("wmrb", np.eye(n_u), np.eye(n_i), "linear", "linear", {"W": U}, {"W": V}, rows, cols, vals,
                               samp, n_i, S, update=False)
    lens = np.bincount(rows, minlength=n_u)
    b = tdist.balanced_user_bounds(lens, world)
    lo, hi = b[rank], b[rank + 1]
    m = (rows >= lo) & (rows < hi)
    local = o.train_step_sparse("wmrb", np.eye(hi - lo), np.eye(n_i), "linear", "linear", {"W": U[lo:hi]}, {"W": V},
                                rows[m] - lo, cols[m], vals[m], samp[lo:hi], n_i, S, update=False)
    comm = tdist.GradientSync()
    dEi = torch.from_numpy(local[2]["W"].copy())
    comm.sync_item_grad(dEi)  # one all-reduce per epoch: the summed item gradient
    np.testing.assert_allclose(dEi.numpy(), full[2]["W"], rtol=1e-12, atol=1e-14)
    # the user rows are owned by the shard: no communication, identical to the corresponding rows of the full run
    np.testing.assert_allclose(local[1]["W"], full[1]["W"][lo:hi], rtol=1e-12, atol=1e-14)
    assert comm.bytes_reduced == dEi.numel() * 8

    # shared user-side parameters (side-feature rows, bias) are reduced; rank-local identity rows are not
    g = {"W": torch.full((7, 2), float(rank + 1)), "b": torch.full((1, 2), float(rank + 1))}
    tower = _FakeTower("biased", g, {"W": torch.zeros(7, 2), "b": torch.zeros(1, 2)})
    tdist.GradientSync(shared_user_rows=5).sync_shared_grads(tower, None)
    assert torch.all(g["W"][:5] == rank + 1) and torch.all(g["W"][5:] == 3.0) and torch.all(g["b"] == 3.0)

    # replicated parameters start identical (rank 0 wins)
    pu = {"W": torch.full((7, 2), float(rank)), "b": torch.full((1, 2), float(rank))}
    pi = {"W": torch.full((4, 2), float(rank + 10))}
    tdist.GradientSync(shared_user_rows=5).broadcast_params(_FakeTower("biased", {}, pu), _FakeTower("linear", {}, pi))
    assert torch.all(pi["W"] == 10.0) and torch.all(pu["W"][5:] == 0.0) and torch.all(pu["W"][:5] == rank) and torch.all(pu["b"] == 0)


def test_user_sharded_training_allreduce():
    _spawn(_dp_training)


class _FakePlan:
    """What GradientSync.sync_grads touches of a TrainPlan: the item tower's dE and the user tower's grads."""

    def __init__(self, u, i):
        self.u, self.i = u, i


def _sync_grads_and_kl(rank, world):
    # ---- one call exchanges the item gradient AND the shared user-side slices (NCCL/gloo form: no peer arena on CPU)
    class IT:
        kind = "linear"
    it = IT()
    it.dE = torch.full((6, 4), float(rank + 1))
    g = {"W": torch.full((7, 4), float(rank + 1)), "b": torch.full((1, 4), float(10 * (rank + 1)))}
    u = _FakeTower("biased", g, {"W": torch.zeros(7, 4), "b": torch.zeros(1, 4)})
    comm = tdist.GradientSync(shared_user_rows=5, peer=False)  # CPU tensors: the collective path, also where CUDA is present
    assert comm.peer is False
    fused = comm.sync_grads(_FakePlan(u, it), lr=0.1)
    assert fused is False
    assert torch.all(it.dE == 3.0)
    assert torch.all(g["W"][:5] == rank + 1) and torch.all(g["W"][5:] == 3.0) and torch.all(g["b"] == 30.0)
    # ---- KL under user sharding: the six additive moments of the rank's interactions, summed, give the global statistics
    rng = np.random.default_rng(5)
    p = rng.standard_normal(400) * 0.3 + 0.1
    vals = rng.choice([-1.0, 1.0, 2.0], 400)
    mine = slice(0, 150) if rank == 0 else slice(150, 400)

    def moments(pp, vv):
        pos = vv > 0
        return np.array([pos.sum(), pp[pos].sum(), (pp[pos] ** 2).sum(), (~pos).sum(), pp[~pos].sum(), (pp[~pos] ** 2).sum()])
    m = torch.from_numpy(moments(p[mine], vals[mine]))
    comm.allreduce_kl_moments(m)
    np.testing.assert_allclose(m.numpy(), moments(p, vals), rtol=1e-13)
    n_p, s_p, q_p, n_n, s_n, q_n = m.numpy()
    mp, mn = s_p / n_p, s_n / n_n
    vp, vn = q_p / n_p - mp ** 2, q_n / n_n - mn ** 2
    from scipy import special
    loss = 1.0 - special.ndtr((mp - mn) / np.sqrt(vp + vn))
    np.testing.assert_allclose(loss, float(o.kl_loss(p, vals)), rtol=1e-10)  # == the single-process KL of all interactions

    class KLPlan:
        loss = "kl"

        def mean_loss(self):
            return 0.25
    assert comm.mean_loss(KLPlan()) == 0.25  # already global: no second reduction


def test_sync_grads_collective_form_and_kl_moments():
    _spawn(_sync_grads_and_kl)


def _sharded_topk(rank, world):
    rng = np.random.default_rng(9)
    n_u, n_i, r, k = 25, 90, 8, 7
    U = rng.integers(-4, 5, (n_u, r)).astype(np.float32) / 8
    V = rng.integers(-4, 5, (n_i, r)).astype(np.float32) / 8  # grid values: many exact ties across shards
    P = o.canonical_scores(U, V)
    want = o.topk_stable(P, k)
    b = tdist.shard_bounds(n_i, world)
    lo, hi = b[rank], b[rank + 1]
    loc = o.topk_stable(P[:, lo:hi], k)
    loc_idx = torch.from_numpy((loc + lo).astype(np.int32))
    loc_sc = torch.from_numpy(np.take_along_axis(P[:, lo:hi], loc.astype(np.int64), 1))
    all_idx = [torch.empty_like(loc_idx) for _ in range(world)]
    all_sc = [torch.empty_like(loc_sc) for _ in range(world)]
    dist.all_gather(all_idx, loc_idx)
    dist.all_gather(all_sc, loc_sc)
    idx, sc = tdist.merge_topk_lists([t.numpy() for t in all_idx], [t.numpy() for t in all_sc], k)
    assert np.array_equal(idx, want)  # a global top-k member is always in its slab's local top-k
    assert np.array_equal(sc, np.take_along_axis(P, want.astype(np.int64), 1))


def test_item_sharded_topk_merge():
    _spawn(_sharded_topk)


def _mean_loss(rank, world):
    class IP:
        loss = "wmrb"
        n_pos = 3 + rank
        vals = torch.zeros(1)

        def mean_loss(self):
            return 2.0 + rank
    got = tdist.GradientSync().mean_loss(IP())
    assert abs(got - (3 * 2.0 + 4 * 3.0) / 7) < 1e-12


def test_mean_loss_is_weighted_over_ranks():
    _spawn(_mean_loss)


# ---- the full item-sharded protocol (bound pass -> bounded slab lists -> all-to-all -> merge -> all-gather) with the
# two kernels replaced by oracle-backed CPU stand-ins: only dist.sharded_topk's host logic is under test


def _fake_score_topk(U, V, r, k, clamp, item_offset=0, row_bound=None, out=None):
    P = o.canonical_scores(U[:, :r].numpy(), V[:, :r].numpy())
    if clamp:
        P = np.where(P > 0, P, np.float32(0))
    loc = o.topk_stable(P, k)
    sc = np.take_along_axis(P, loc.astype(np.int64), 1)
    idx = (loc + item_offset).astype(np.int32)
    if row_bound is not None:  # what tmf_score_topk_bounded may drop: entries strictly below the bound
        rb = row_bound.numpy()[:, None]
        drop = sc < rb
        if clamp:
            drop &= rb > 0
        # surviving entries stay sorted in front, dropped slots become padding
        order = np.argsort(drop, axis=1, kind="stable")
        idx, sc, drop = (np.take_along_axis(a, order, 1) for a in (idx, sc, drop))
        idx = np.where(drop, np.int32(2 ** 31 - 1), idx)
        sc = np.where(drop, np.float32(-np.inf), sc)
    ti, ts = torch.from_numpy(idx.copy()), torch.from_numpy(sc.astype(np.float32).copy())
    if out is not None:
        out[0].copy_(ti); out[1].copy_(ts)
        return out
    return ti, ts


class _FakeAbi:
    @staticmethod
    def ptr(t):
        return t

    @staticmethod
    def call(name, idx_in, sc_in, n_lists, n_users, k, out_idx, out_sc):
        assert name == "tmf_topk_merge"
        i = idx_in.reshape(n_lists, n_users, k).numpy()
        s = sc_in.reshape(n_lists, n_users, k).numpy()
        mi, ms = tdist.merge_topk_lists(list(i), list(s), k)
        out_idx.copy_(torch.from_numpy(mi.astype(np.int32)))
        out_sc.copy_(torch.from_numpy(ms.astype(np.float32)))


def _bounded_protocol(rank, world):
    import teamoflow_b200 as pkg
    import teamoflow_b200.mf.matrix_factorization as mfm
    mfm.score_topk = _fake_score_topk
    pkg._abi = _FakeAbi  # `from .. import _abi` inside sharded_topk resolves to the package attribute
    rng = np.random.default_rng(21)
    n_u, n_i, r, k = 23, 120, 8, 6  # 23 users over 2 ranks: unequal slices
    U = rng.integers(-4, 5, (n_u, r)).astype(np.float32) / 8
    V = rng.integers(-4, 5, (n_i, r)).astype(np.float32) / 8
    b = tdist.shard_bounds(n_i, world)
    lo, hi = b[rank], b[rank + 1]
    for clamp in (False, True):
        P = o.canonical_scores(U, V)
        if clamp:
            P = np.where(P > 0, P, np.float32(0))
        want = o.topk_stable(P, k)
        for bound in ("force", False):
            idx, sc = tdist.sharded_topk(torch.from_numpy(U), torch.from_numpy(V[lo:hi].copy()), r, k, clamp, lo,
                                         exchange="nccl", bound=bound)
            assert np.array_equal(idx.numpy(), want), (clamp, bound)
            assert np.array_equal(sc.numpy(), np.take_along_axis(P, want.astype(np.int64), 1))


def test_item_sharded_bounded_protocol_host_logic():
    _spawn(_bounded_protocol)


def test_rebalanced_user_bounds_equalises_measured_cost():
    """Ranges with different cost per unit of weight: after one pass the boundaries sit at equal shares of the measured cost."""
    import numpy as np
    from teamoflow_b200.mf import dist as tdist
    rng = np.random.default_rng(0)
    w = np.sort(rng.pareto(1.2, 20000) * 10 + 1)[::-1].astype(np.int64) + 32   # heavy users first, like the Zipf generators
    world = 4
    b0 = tdist.balanced_user_bounds(w, world)
    assert b0[0] == 0 and b0[-1] == w.size and all(x <= y for x, y in zip(b0, b0[1:]))
    density = np.array([1.0, 1.4, 0.9, 0.6])                                 # cost per unit of weight of each CURRENT range
    times = [density[r] * w[b0[r]:b0[r + 1]].sum() for r in range(world)]
    b1 = tdist.rebalanced_user_bounds(w, b0, times)
    assert b1[0] == 0 and b1[-1] == w.size and all(x <= y for x, y in zip(b1, b1[1:]))
    cost = np.concatenate([w[b0[r]:b0[r + 1]] * density[r] for r in range(world)])  # the model the pass assumes
    new_t = np.array([cost[b1[r]:b1[r + 1]].sum() for r in range(world)])
    assert new_t.max() / new_t.mean() < 1.01 < max(times) / np.mean(times)
    # equal times are a fixed point
    assert tdist.rebalanced_user_bounds(w, b1, list(new_t)) == b1 or \
        np.abs(np.array(tdist.rebalanced_user_bounds(w, b1, list(new_t))) - np.array(b1)).max() <= 2
