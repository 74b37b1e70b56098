"""GPU parity tests at the EXACT shapes of BASELINE.json configs[0] (C1) and configs[1] (C2) -- the two configurations the
NumPy oracle finishes in seconds (VERDICT r1, "no parity test runs a BASELINE config").

For each: one full training step from the configuration's own initialisation against the fp64 oracle (per-interaction
losses, dU, dV within north_star's 1e-5 relative), the update against the oracle's Adam step-1, a short ``fit`` trajectory
against ``oracle.fit`` (sign-like update => compared by fraction, DESIGN 4), and the evaluation metrics the configuration
names (recall / precision / f1 @ 10, and NDCG) BIT-EXACT against the oracle on the fitted embeddings.
"""
import numpy as np
import pytest
import torch

import _baseline_configs as cfg
from oracle import mf_oracle as o
from test_gpu_train import _mods, build_model, close, cpu

pytestmark = pytest.mark.gpu


def _dense_A(c):
    A = np.zeros((c["n_u"], c["n_i"]), np.float32)
    A[c["rows"], c["cols"]] = c["vals"]
    return A


def _run_config(c, epochs):
    n_u, n_i, r, S, loss, lr = c["n_u"], c["n_i"], c["r"], c["S"], c["loss"], c["lr"]
    rows, cols, vals, samp = c["rows"], c["cols"], c["vals"], c["samp"]
    _, _, _, _, FM, SI, _ = _mods()
    inter = SI(np.stack([rows, cols], 1), vals, (n_u, n_i))
    pu, pi = {"W": c["U0"]}, {"W": c["V0"]}
    eye_u, eye_i = np.eye(n_u), np.eye(n_i)

    # ---- one step from the configuration's initialisation
    want = o.train_step_sparse(loss, eye_u, eye_i, "linear", "linear", {"W": c["U0"].astype(np.float64)},
                               {"W": c["V0"].astype(np.float64)}, rows, cols, vals.astype(np.float64), samp, n_i, S or None, lr=lr,
                               update=False)
    samp_gpu = samp if samp is not None else np.zeros((n_u, 1), np.int64)
    m = build_model(loss, ("linear", "linear"), pu, pi, r, n_u, n_i, S or None, samp_gpu)
    plan = m._prepare(FM.eye(n_u), FM.eye(n_i), inter)
    plan.forward_backward()
    close(cpu(plan.ip.loss_vector()), want[0], name=f"{c['name']} loss vector")
    close(cpu(plan.u.grads["W"])[:, :r], want[1]["W"], name=f"{c['name']} dU")
    close(cpu(plan.i.grads["W"])[:, :r], want[2]["W"], name=f"{c['name']} dV")
    assert abs(plan.ip.mean_loss() - float(np.mean(want[0]))) <= 1e-5 * abs(float(np.mean(want[0])))
    gU, gV = cpu(plan.u.grads["W"]).copy(), cpu(plan.i.grads["W"]).copy()
    U_before, V_before = cpu(plan.u.W).copy(), cpu(plan.i.W).copy()
    plan.u.update(lr)
    plan.i.update(lr)
    np.testing.assert_allclose(cpu(plan.u.W), o.adam_step1(U_before, gU, lr), rtol=2e-6, atol=1e-9)
    np.testing.assert_allclose(cpu(plan.i.W), o.adam_step1(V_before, gV, lr), rtol=2e-6, atol=1e-9)

    # ---- a short fit through the public API against oracle.fit
    m = build_model(loss, ("linear", "linear"), pu, pi, r, n_u, n_i, S or None, samp_gpu)
    m.fit(epochs, FM.eye(n_u), FM.eye(n_i), inter, lr=lr, verbose=False)
    _, _, Eu, Ei, hist = o.fit(epochs, loss, eye_u, eye_i, "linear", "linear", {"W": c["U0"].astype(np.float64)},
                               {"W": c["V0"].astype(np.float64)}, rows, cols, vals.astype(np.float64), samp, n_i, S or None,
                               lr=lr, dense=False)
    for got, ref, tag in ((cpu(m.user_embedding), Eu, "E_u"), (cpu(m.item_embedding), Ei, "E_i")):
        d = np.abs(got - ref)
        assert (d < 1e-4).mean() > 0.99, f"{c['name']} {tag}: only {(d < 1e-4).mean():.4f} of the weights track the oracle trajectory"
    return m


def _check_metrics(m, A, k=10):
    U, V = cpu(m.user_embedding), cpu(m.item_embedding)
    P = o.canonical_scores(U, V)
    At = torch.as_tensor(A)
    from scipy import sparse
    np.testing.assert_array_equal(m.retrieve_user_recs(k=k), o.retrieve_user_recs(P, k=k))
    for Ain in (At, sparse.csr_matrix(A)):
        np.testing.assert_array_equal(cpu(m.recall_at_k(Ain, k)), o.recall_at_k(P, A, k))
        np.testing.assert_array_equal(cpu(m.recall_at_k(Ain, k, True)), o.recall_at_k(P, A, k, True))
        np.testing.assert_array_equal(cpu(m.precision_at_k(Ain, k)), o.precision_at_k(P, A, k))
    np.testing.assert_allclose(float(m.f1_at_k(At, k)), float(o.f1_at_k(P, A, k)), rtol=1e-6)
    np.testing.assert_allclose(cpu(m.ndcg_at_k(At, k)), o.ndcg_at_k(P, A, k), rtol=5e-6, atol=1e-6)


def test_c1_toy_1k_x_1k_rank10_mse():
    c = cfg.c1()
    assert c["rows"].size == 10_000
    m = _run_config(c, epochs=5)
    _check_metrics(m, _dense_A(c))


def test_c2_ml100k_shape_rank32_wmrb_recall_at_10():
    c = cfg.c2()
    assert (c["n_u"], c["n_i"], c["S"]) == (943, 1682, 336) and 50_000 < c["rows"].size < 62_000
    m = _run_config(c, epochs=3)
    _check_metrics(m, _dense_A(c))
    # recall@10 against ALL ratings >= 4 of the synthetic set is what the configuration names; it must equal the oracle bit for bit
    rec = cpu(m.recall_at_k(torch.as_tensor(_dense_A(c)), 10))
    assert rec.shape[0] == np.count_nonzero(np.bincount(c["rows"], minlength=c["n_u"]))


# ------------------------------------------------------------------------------- round-2 extensions (SURVEY 8f)


def test_minibatch_mode_matches_oracle_per_block():
    """fit(batch_size=B): one optimizer step per contiguous block of B users, each on that block's interactions only."""
    from test_gpu_train import make_problem
    n_u, n_i, r, S, B = 50, 70, 8, 10, 16
    rng, rows, cols, vals, samp = make_problem(n_u, n_i, r, 500, S, 31, values=(1.0, 2.0, 5.0))
    U0, V0 = o.uniform_initializer(n_u, r, rng), o.uniform_initializer(n_i, r, rng)
    _, _, _, _, FM, SI, _ = _mods()
    for loss in ("wmrb", "mse"):
        m = build_model(loss, ("linear", "linear"), {"W": U0}, {"W": V0}, r, n_u, n_i, S, samp)
        m.fit(2, FM.eye(n_u), FM.eye(n_i), SI(np.stack([rows, cols], 1), vals, (n_u, n_i)), lr=0.1, verbose=False, batch_size=B)
        pu, pi = {"W": U0.astype(np.float64)}, {"W": V0.astype(np.float64)}
        last = []
        for _ in range(2):
            last = []
            for lo in range(0, n_u, B):
                hi = min(lo + B, n_u)
                sel = (rows >= lo) & (rows < hi)
                # the block's step on the FULL parameter set: other users simply have no interactions (zero gradient rows)
                # (their samples carry no gradient either: G_uj sums over the user's own positives)
                lv, _, _, pu, pi = o.train_step_sparse(loss, np.eye(n_u), np.eye(n_i), "linear", "linear", pu, pi, rows[sel], cols[sel],
                                                       vals[sel].astype(np.float64), samp, n_i, S, lr=0.1)
                last.append(lv)
        d = np.abs(cpu(m.user_embedding) - pu["W"])
        assert (d < 1e-4).mean() > 0.99, (loss, (d < 1e-4).mean())
        d = np.abs(cpu(m.item_embedding) - pi["W"])
        assert (d < 1e-4).mean() > 0.99, (loss, (d < 1e-4).mean())
        got, ref = cpu(m._plan.ip.loss_vector()), np.concatenate(last)
        assert got.shape == ref.shape
        assert (np.abs(got - ref) < 1e-4 * max(np.abs(ref).max(), 1.0)).mean() > 0.97, loss


def _kl_from_moments(shards, p, val, ws):
    """KL loss and coefficients with the interactions split into ``shards`` (ranks): each shard's six moments, summed on
    the host side of the ABI, then each shard's coefficients from the global moments."""
    from teamoflow_b200 import _abi
    n = p.numel()
    mom = torch.zeros(len(shards), 6, dtype=torch.float64, device="cuda")
    for g, (a, b) in enumerate(shards):
        _abi.call("tmf_kl_moments", b - a, _abi.ptr(p[a:b]), _abi.ptr(val[a:b]), _abi.ptr(mom[g]), _abi.ptr(ws))
    tot = mom.sum(0).contiguous()
    loss, coef = torch.zeros(1, device="cuda"), torch.zeros(n, device="cuda")
    for a, b in shards:
        _abi.call("tmf_kl_coef_from_moments", b - a, _abi.ptr(p[a:b]), _abi.ptr(val[a:b]), _abi.ptr(tot), _abi.ptr(loss),
                  _abi.ptr(coef[a:b]), _abi.ptr(ws))
    torch.cuda.synchronize()
    return cpu(loss), cpu(coef)


def test_kl_moments_summed_over_shards_equal_one_shard():
    """Two ranks' moments summed give the KL loss and coefficients of one rank holding every interaction."""
    from teamoflow_b200 import _abi
    rng = np.random.default_rng(3)
    n = 5000
    p = torch.as_tensor(rng.standard_normal(n).astype(np.float32) * 0.3 + 0.1, device="cuda")
    val = torch.as_tensor(rng.choice([-1.0, 1.0, 2.0], n).astype(np.float32), device="cuda")
    ws = torch.empty(_abi.query("tmf_reduce_ws_bytes"), dtype=torch.uint8, device="cuda")
    l1, c1 = _kl_from_moments(((0, n),), p, val, ws)
    h = n // 3
    l2, c2 = _kl_from_moments(((0, h), (h, n)), p, val, ws)
    np.testing.assert_allclose(l2, l1, rtol=1e-6)
    np.testing.assert_allclose(c2, c1, rtol=2e-5, atol=1e-9)
    want_loss, want_c = o.kl_loss(cpu(p).astype(np.float64), cpu(val)), o.kl_coef(cpu(val), cpu(p).astype(np.float64))
    np.testing.assert_allclose(l2[0], float(want_loss), rtol=1e-5)
    close(c2, want_c, name="kl coef from moments")


def test_kl_moments_stay_inside_the_reduce_workspace():
    """tmf_reduce_ws_bytes() covers the widest reduction: 4M interactions take 977 blocks of six partial sums each, which
    must all land inside the workspace (a canary right after it stays intact) and add up to the float64 host sums."""
    from teamoflow_b200 import _abi
    rng = np.random.default_rng(11)
    n = 4_000_000
    p_h = (rng.standard_normal(n) * 0.5 + 0.25).astype(np.float32)
    val_h = rng.choice([-1.0, 0.0, 1.0, 3.0], n).astype(np.float32)
    p, val = torch.as_tensor(p_h, device="cuda"), torch.as_tensor(val_h, device="cuda")
    ws_bytes, tail = _abi.query("tmf_reduce_ws_bytes"), 4096
    buf = torch.zeros(ws_bytes + tail, dtype=torch.uint8, device="cuda")
    buf[ws_bytes:] = 0xA5
    mom = torch.zeros(6, dtype=torch.float64, device="cuda")
    _abi.call("tmf_kl_moments", n, _abi.ptr(p), _abi.ptr(val), _abi.ptr(mom), _abi.ptr(buf))
    torch.cuda.synchronize()
    assert bool((buf[ws_bytes:] == 0xA5).all()), "tmf_kl_moments wrote past tmf_reduce_ws_bytes()"
    x, pos = p_h.astype(np.float64), val_h > 0
    want = [pos.sum(), x[pos].sum(), (x[pos] ** 2).sum(), (~pos).sum(), x[~pos].sum(), (x[~pos] ** 2).sum()]
    got = cpu(mom)
    assert got[0] == want[0] and got[3] == want[3]
    np.testing.assert_allclose(got, want, rtol=1e-11)


def test_predict_with_sparse_A_and_predict_ranks_without_densifying():
    from scipy import sparse
    from test_gpu_score import model_with
    rng = np.random.default_rng(8)
    n_u, n_i, r = 37, 91, 8
    U = rng.integers(-4, 5, (n_u, r)).astype(np.float32) / 8
    V = rng.integers(-4, 5, (n_i, r)).astype(np.float32) / 8
    A = np.where(rng.random((n_u, n_i)) < 0.1, rng.choice([-1.0, 1.0, 4.0], (n_u, n_i)), 0.0).astype(np.float32)
    A[5] = 0.0
    m = model_with(U, V)
    P_want, un_want = o.predict(U, V, A)
    for Ain in (torch.as_tensor(A), sparse.csr_matrix(A)):
        P, un = m.predict(Ain)
        np.testing.assert_array_equal(cpu(P), P_want)
        np.testing.assert_array_equal(cpu(un), un_want)
        np.testing.assert_array_equal(cpu(m.predict_ranks(Ain)), o.predict_ranks(U, V, A))


def test_recommend_excludes_seen_items_bit_exact():
    from scipy import sparse
    from test_gpu_score import model_with
    rng = np.random.default_rng(12)
    n_u, n_i, r, k = 60, 400, 16, 10
    U = rng.integers(-4, 5, (n_u, r)).astype(np.float32) / 8   # grid values: exact ties, the id tie-break matters
    V = rng.integers(-4, 5, (n_i, r)).astype(np.float32) / 8
    A = np.where(rng.random((n_u, n_i)) < 0.05, 1.0, 0.0).astype(np.float32)
    A[3] = 0.0                      # a user who has seen nothing
    A[4, :] = 1.0; A[4, 7] = 0.0    # a user with ONE unseen item -> padded with -1
    A[6, :300] = 1.0                # a heavy user: more seen items than the fused list can absorb -> exact fallback
    m = model_with(U, V)
    P = o.canonical_scores(U, V).astype(np.float64)
    P[A != 0] = -np.inf
    want = o.topk_stable(P, k)
    n_unseen = (A == 0).sum(1)
    want = np.where(np.arange(k)[None, :] < n_unseen[:, None], want, -1)
    for seen in (sparse.csr_matrix(A), torch.as_tensor(A)):
        got = cpu(m.recommend(seen, k=k))
        np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(m.retrieve_user_recs(user=6, k=k, exclude=sparse.csr_matrix(A)), want[6])
    np.testing.assert_array_equal(cpu(m.recommend(sparse.csr_matrix(A), k=k, users=[4, 0, 6])), want[[4, 0, 6]])
    # default behaviour is still the reference's: seen items are NOT excluded (SURVEY A.7)
    np.testing.assert_array_equal(m.retrieve_user_recs(k=k), o.topk_stable(o.canonical_scores(U, V), k))


def test_out_of_range_interaction_ids_raise():
    _, _, _, _, FM, SI, _ = _mods()
    with pytest.raises(ValueError, match="out of range"):
        SI(np.array([[0, 1], [2, 5]]), np.ones(2, np.float32), (3, 5)).csr()      # 1-based column id
    with pytest.raises(ValueError, match="out of range"):
        SI(np.array([[0, 1], [-1, 2]]), np.ones(2, np.float32), (3, 5)).csr()
    SI(np.array([[0, 1], [2, 4]]), np.ones(2, np.float32), (3, 5)).csr()


def test_load_resolves_class_names_through_a_fixed_table(tmp_path):
    _, _, L, _, FM, SI, MF = _mods()
    m = MF(4, loss_graph=L.WMRBLoss(), n_users=5, n_items=6, n_samples=2, generate_sample=True)
    path = str(tmp_path / "m.pt")
    m.save(path)
    back = MF.load(path)
    assert isinstance(back.loss_graph, L.WMRBLoss) and back.generate_sample is True
    assert torch.equal(back.random_ind, m.random_ind)
    blob = torch.load(path, weights_only=True)
    blob["config"]["loss_graph"] = "new_relu_params"   # an exported zero-argument callable that is not a graph class
    torch.save(blob, path)
    with pytest.raises(ValueError, match="not one of the package's graph classes"):
        MF.load(path)
    assert isinstance(MF.load(path, graphs={"loss_graph": L.MSELoss()}).loss_graph, L.MSELoss)
