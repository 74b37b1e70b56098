"""GPU parity tests of the training path: CUDA kernels (through the C ABI and the reference-shaped
Python surface) against the oracle on identical inputs, weights and negatives.

Tolerance: north_star's "losses, gradients and scores agree within 1e-5 relative in fp32" -- checked
against the fp64 oracle twin as max-abs error relative to the tensor's max-abs value (plus elementwise
rtol where no cancellation is involved).
"""
import json
import os

import numpy as np
import pytest
import torch
from scipy import sparse

from oracle import mf_oracle as o

pytestmark = pytest.mark.gpu

G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))
REL = 1e-5


def _mods():
    from teamoflow_b200.mf import embedding_graphs as E, initializer_graphs as I, loss_graphs as L
    from teamoflow_b200.mf import _engine as eng
    from teamoflow_b200.mf._tensors import FeatureMatrix, SparseInteractions
    from teamoflow_b200.mf.matrix_factorization import MatrixFactorization
    return E, I, L, eng, FeatureMatrix, SparseInteractions, MatrixFactorization


def fixed_init(W):
    from teamoflow_b200.mf.initializer_graphs import Initializer

    class Fixed(Initializer):
        def initialize_weights(self, n_features, n_components):
            assert W.shape == (n_features, n_components)
            return torch.as_tensor(np.asarray(W, dtype=np.float32), device="cuda")
    return Fixed()


def close(got, want, rel=REL, name="", floor=0.0):
    """max-abs error relative to the tensor's max-abs value; `floor` = magnitude of the summands for sums
    that cancel to ~0 (e.g. the item-bias gradient under WMRB is identically zero in exact arithmetic)"""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, f"{name}: shape {got.shape} vs {want.shape}"
    scale = max(np.abs(want).max() if want.size else 0.0, floor, 1e-30)
    err = np.abs(got - want).max() if want.size else 0.0
    assert err <= rel * scale, f"{name}: max abs err {err:.3e} > {rel} * {scale:.3e}"


def cpu(t):
    return t.detach().cpu().numpy()


LOSS_OBJ = {"mse": "MSELoss", "wmrb": "WMRBLoss", "kl": "KLDivergenceLoss"}
EMB_OBJ = {"linear": "LinearEmbedding", "biased": "BiasedLinearEmbedding", "relu": "ReLUEmbedding"}


def make_problem(n_u, n_i, r, nnz, S, seed, values=(1.0, 2.0, 3.0, -1.0, -2.0), wscale=0.5):
    rng = np.random.default_rng(seed)
    cells = rng.choice(n_u * n_i, size=min(nnz, n_u * n_i), replace=False)
    cells.sort()
    rows, cols = (cells // n_i).astype(np.int64), (cells % n_i).astype(np.int64)
    vals = rng.choice(np.array(values, dtype=np.float32), size=rows.size)
    samp = np.stack([rng.choice(n_i, S, replace=False) for _ in range(n_u)]).astype(np.int64)
    return rng, rows, cols, vals, samp


def params_for(kind, F, r, rng, wscale):
    if kind == "relu":
        return {"W": (rng.standard_normal((5 * r, r)) * wscale * 0.3).astype(np.float32),
                "Wr": rng.standard_normal((F, 5 * r)).astype(np.float32) * 0.5,
                "br": (rng.standard_normal((1, 5 * r)) * 0.1).astype(np.float32)}
    p = {"W": (rng.standard_normal((F, r)) * wscale).astype(np.float32)}
    if kind == "biased":
        p["b"] = (rng.standard_normal((1, r)) * 0.1).astype(np.float32)
    return p


def build_model(loss, kinds, pu, pi, r, n_u, n_i, S, samp):
    E, I, L, eng, FM, SI, MF = _mods()
    m = MF(r, user_repr_graph=getattr(E, EMB_OBJ[kinds[0]])(), item_repr_graph=getattr(E, EMB_OBJ[kinds[1]])(),
           loss_graph=getattr(L, LOSS_OBJ[loss])(), user_weight_graph=fixed_init(pu["W"]), item_weight_graph=fixed_init(pi["W"]),
           n_users=n_u, n_items=n_i, n_samples=S)
    m.random_ind = torch.as_tensor(samp, device="cuda")
    for side, p in (("user", pu), ("item", pi)):
        if "b" in p:
            setattr(m, f"{side}_linear_bias", torch.as_tensor(p["b"], device="cuda"))
        if "Wr" in p:
            setattr(m, f"{side}_relu_weight", torch.as_tensor(p["Wr"], device="cuda"))
            setattr(m, f"{side}_relu_bias", torch.as_tensor(p["br"], device="cuda"))
    return m


def oracle64(loss, Xu, Xi, kinds, pu, pi, rows, cols, vals, samp, n_i, S, lr, update=False):
    f = lambda d: {k: v.astype(np.float64) for k, v in d.items()}  # noqa: E731
    return o.train_step_sparse(loss, Xu.astype(np.float64), Xi.astype(np.float64), kinds[0], kinds[1], f(pu), f(pi),
                               rows, cols, vals.astype(np.float64), samp, n_i, S, lr=lr, update=update)


def min_hinge_gap(Xu, Xi, kinds, pu, pi, rows, cols, vals, samp):
    """smallest |1 - p + s| over (positive, sample) pairs in fp64: the WMRB indicator is discontinuous there."""
    f = lambda d: {k: v.astype(np.float64) for k, v in d.items()}  # noqa: E731
    Eu, _ = o.embed_forward(kinds[0], Xu.astype(np.float64), f(pu))
    Ei, _ = o.embed_forward(kinds[1], Xi.astype(np.float64), f(pi))
    P = Eu @ Ei.T
    pos = vals > 0
    h = 1.0 - P[rows[pos], cols[pos]][:, None] + np.take_along_axis(P, samp, 1)[rows[pos]]
    return np.abs(h).min() if h.size else 1.0


def features(kind, n, F, seed):
    if kind == "eye":
        return np.eye(n, dtype=np.float32), None
    X = sparse.random(n, F, density=min(1.0, 4.0 / F), random_state=seed, format="csr", dtype=np.float32)
    X = (X + sparse.eye(n, F, dtype=np.float32, format="csr")).tocsr()  # [I | M]-like: every row non-empty
    return X.toarray().astype(np.float32), X


# ------------------------------------------------------------------------------- golden vectors


@pytest.mark.parametrize("name,loss", [("wmrb_3x4", "wmrb"), ("mse_2x2", "mse"), ("kl_2p2n", "kl"),
                                       ("rand_mse", "mse"), ("rand_wmrb", "wmrb"), ("rand_kl", "kl")])
def test_golden_vectors_through_cuda(name, loss):
    c = G[name]
    it = c["inter"]
    rows = np.array([x[0] for x in it]); cols = np.array([x[1] for x in it]); vals = np.array([x[2] for x in it], np.float32)
    U, V = np.array(c["U"], np.float32), np.array(c["V"], np.float32)
    n_u, n_i, r = U.shape[0], V.shape[0], U.shape[1]
    samp = np.array(c["samp"], np.int64) if "samp" in c else np.zeros((n_u, 1), np.int64)
    S = samp.shape[1]
    m = build_model(loss, ("linear", "linear"), {"W": U}, {"W": V}, r, n_u, n_i, S, samp)
    _, _, _, _, FM, SI, _ = _mods()
    plan = m._prepare(FM.eye(n_u), FM.eye(n_i), SI(np.stack([rows, cols], 1), vals, (n_u, n_i)))
    plan.forward_backward()
    close(cpu(plan.ip.loss_vector()), np.array(c["loss"]), name="loss")
    close(cpu(plan.u.grads["W"])[:, :r], np.array(c["dU"]), name="dU")
    close(cpu(plan.i.grads["W"])[:, :r], np.array(c["dV"]), name="dV")


# ------------------------------------------------------------------------------- step parity matrix


@pytest.mark.parametrize("loss", ["mse", "wmrb", "kl"])
@pytest.mark.parametrize("kinds", [("linear", "linear"), ("biased", "biased"), ("relu", "linear"), ("linear", "relu")])
@pytest.mark.parametrize("feat", ["eye", "sparse"])
def test_step_parity(loss, kinds, feat):
    n_u, n_i, r, S = 61, 83, 12, 9
    for seed in range(20):
        rng, rows, cols, vals, samp = make_problem(n_u, n_i, r, 900, S, 100 + seed)
        Xu_d, Xu_s = features(feat, n_u, n_u + 7 if feat == "sparse" else n_u, 1)
        Xi_d, Xi_s = features(feat, n_i, n_i + 5 if feat == "sparse" else n_i, 2)
        pu = params_for(kinds[0], Xu_d.shape[1], r, rng, 0.4)
        pi = params_for(kinds[1], Xi_d.shape[1], r, rng, 0.4)
        if loss != "wmrb" or min_hinge_gap(Xu_d, Xi_d, kinds, pu, pi, rows, cols, vals, samp) > 1e-4:
            break
    lr = 0.05
    want = oracle64(loss, Xu_d, Xi_d, kinds, pu, pi, rows, cols, vals, samp, n_i, S, lr)
    m = build_model(loss, kinds, pu, pi, r, n_u, n_i, S, samp)
    _, _, _, _, FM, SI, _ = _mods()
    plan = m._prepare(Xu_s if Xu_s is not None else torch.as_tensor(Xu_d), Xi_s if Xi_s is not None else torch.as_tensor(Xi_d),
                      SI(np.stack([rows, cols], 1), vals, (n_u, n_i)))
    plan.forward_backward()
    close(cpu(plan.ip.loss_vector()), want[0], name="loss")
    for tower, g in ((plan.u, want[1]), (plan.i, want[2])):
        for k in g:
            got = cpu(tower.grads[k])[:, :g[k].shape[1]]
            # column sums (bias gradients) are sums over all rows of dE: their rounding scale is sum |dE|
            floor = np.abs(cpu(tower.dE)).sum(axis=0).max() if k in ("b", "br") else 0.0
            close(got, g[k], name=f"{tower.kind}.{k}", floor=floor)
    # update: w_new must equal the oracle's Adam step-1 applied to the GPU's own gradient (the update is
    # sign-like, so comparing against the oracle's gradient would amplify 1e-7 differences near g = 0)
    before = {(s, k): cpu(w).copy() for s, t in (("u", plan.u), ("i", plan.i)) for k, w in t.trainables().items()}
    grads = {(s, k): cpu(t.grads[k]).copy() for s, t in (("u", plan.u), ("i", plan.i)) for k in t.trainables()}
    plan.u.update(lr)
    plan.i.update(lr)
    for (s, k), w0 in before.items():
        t = plan.u if s == "u" else plan.i
        np.testing.assert_allclose(cpu(t.trainables()[k]), o.adam_step1(w0, grads[(s, k)], lr), rtol=2e-6, atol=1e-9)


@pytest.mark.parametrize("r,S", [(3, 5), (10, 40), (32, 336), (64, 128), (128, 32), (200, 17), (64, 700)])
def test_wmrb_shapes(r, S):
    """WMRB through the engine at seven (rank, samples) shapes.  They launch seven of the 27 user-pass instantiations,
    (LPR, VPL, JPL) = (4, 1, 2), (4, 1, 16), (16, 1, 8), (32, 1, 2), (32, 1, 16), (32, 1, -1) (G in shared memory) and
    (32, 2, 2): no LPR 8 kernel, and two float4 columns per lane only with JPL 2.  (32, 336) and (64, 700) run the narrow
    sample gather.  tests/test_gpu_train_variants.py compares every instantiation with an fp64 reference."""
    n_u, n_i = 97, max(S + 3, 211)
    for seed in range(20):
        rng, rows, cols, vals, samp = make_problem(n_u, n_i, r, 2500, S, 7 + seed, values=(1.0, 4.0, -1.0))
        pu = {"W": (rng.standard_normal((n_u, r)) / np.sqrt(r)).astype(np.float32)}
        pi = {"W": (rng.standard_normal((n_i, r)) / np.sqrt(r)).astype(np.float32)}
        eye_u, eye_i = np.eye(n_u, dtype=np.float32), np.eye(n_i, dtype=np.float32)
        if min_hinge_gap(eye_u, eye_i, ("linear", "linear"), pu, pi, rows, cols, vals, samp) > 1e-4:
            break
    want = oracle64("wmrb", eye_u, eye_i, ("linear", "linear"), pu, pi, rows, cols, vals, samp, n_i, S, 0.1)
    m = build_model("wmrb", ("linear", "linear"), pu, pi, r, n_u, n_i, S, samp)
    _, _, _, _, FM, SI, _ = _mods()
    plan = m._prepare(FM.eye(n_u), FM.eye(n_i), SI(np.stack([rows, cols], 1), vals, (n_u, n_i)))
    plan.forward_backward()
    close(cpu(plan.ip.loss_vector()), want[0], name="loss")
    close(cpu(plan.u.grads["W"])[:, :r], want[1]["W"], name="dU")
    close(cpu(plan.i.grads["W"])[:, :r], want[2]["W"], name="dV")


def test_midsize_wmrb_with_side_features_and_skew():
    """C3-shaped in miniature: [I | M] sparse features, Zipf-skewed users/items (long segments that span
    several spmm chunks, empty users and items), r=64, S=128."""
    n_u, n_i, r, S, nnz = 3000, 1500, 64, 128, 150_000
    rng = np.random.default_rng(5)
    pu_w = 1.0 / np.arange(1, n_u + 1); pi_w = 1.0 / np.arange(1, n_i + 1)
    u = rng.choice(n_u, size=3 * nnz, p=pu_w / pu_w.sum()); i = rng.choice(n_i, size=3 * nnz, p=pi_w / pi_w.sum())
    cells = np.unique(u.astype(np.int64) * n_i + i)[:nnz]
    rows, cols = cells // n_i, cells % n_i
    vals = np.ones(rows.size, np.float32)
    samp = np.stack([rng.choice(n_i, S, replace=False) for _ in range(n_u)]).astype(np.int64)
    Mu = sparse.random(n_u, 64, density=4 / 64, random_state=1, format="csr", dtype=np.float32); Mu.data[:] = 1
    Mi = sparse.random(n_i, 256, density=16 / 256, random_state=2, format="csr", dtype=np.float32); Mi.data[:] = 1
    Xu = sparse.hstack([sparse.eye(n_u, dtype=np.float32), Mu]).tocsr()
    Xi = sparse.hstack([sparse.eye(n_i, dtype=np.float32), Mi]).tocsr()
    pu = {"W": o.uniform_initializer(Xu.shape[1], r, rng)}
    pi = {"W": o.uniform_initializer(Xi.shape[1], r, rng)}
    want = o.train_step_sparse("wmrb", Xu.astype(np.float64), Xi.astype(np.float64), "linear", "linear",
                               {"W": pu["W"].astype(np.float64)}, {"W": pi["W"].astype(np.float64)}, rows, cols,
                               vals.astype(np.float64), samp, n_i, S, update=False)
    m = build_model("wmrb", ("linear", "linear"), pu, pi, r, n_u, n_i, S, samp)
    _, _, _, _, FM, SI, _ = _mods()
    plan = m._prepare(Xu, Xi, SI(np.stack([rows, cols], 1), vals, (n_u, n_i)))
    plan.forward_backward()
    close(cpu(plan.ip.loss_vector()), want[0], name="loss")
    close(cpu(plan.u.grads["W"])[:, :r], want[1]["W"], name="dWu")
    close(cpu(plan.i.grads["W"])[:, :r], want[2]["W"], name="dWi")
    # bitwise determinism: fixed summation order, no float atomics
    g1 = plan.i.grads["W"].clone(); l1 = plan.ip.loss_k.clone()
    plan.forward_backward()
    assert torch.equal(g1, plan.i.grads["W"]) and torch.equal(l1, plan.ip.loss_k)


def test_unsorted_interactions_keep_stored_order():
    n_u, n_i, r = 20, 30, 8
    rng, rows, cols, vals, samp = make_problem(n_u, n_i, r, 120, 4, 3)
    perm = rng.permutation(rows.size)
    pu = {"W": (rng.standard_normal((n_u, r)) * 0.3).astype(np.float32)}
    pi = {"W": (rng.standard_normal((n_i, r)) * 0.3).astype(np.float32)}
    m = build_model("mse", ("linear", "linear"), pu, pi, r, n_u, n_i, 4, samp)
    _, _, _, _, FM, SI, _ = _mods()
    plan = m._prepare(FM.eye(n_u), FM.eye(n_i), SI(np.stack([rows[perm], cols[perm]], 1), vals[perm], (n_u, n_i)))
    plan.forward_backward()
    P = pu["W"].astype(np.float64) @ pi["W"].astype(np.float64).T
    close(cpu(plan.ip.loss_vector()), (vals[perm] - P[rows[perm], cols[perm]]) ** 2, name="loss order")


def test_short_trajectory_matches_oracle_fit():
    n_u, n_i, r, S = 50, 70, 8, 10
    rng, rows, cols, vals, samp = make_problem(n_u, n_i, r, 400, S, 11, values=(1.0, 2.0, 5.0))
    U0, V0 = o.uniform_initializer(n_u, r, rng), o.uniform_initializer(n_i, r, rng)
    m = build_model("wmrb", ("linear", "linear"), {"W": U0}, {"W": V0}, r, n_u, n_i, S, samp)
    _, _, _, _, FM, SI, _ = _mods()
    m.fit(5, FM.eye(n_u), FM.eye(n_i), SI(np.stack([rows, cols], 1), vals, (n_u, n_i)), lr=0.1, verbose=False)
    _, _, Eu, Ei, _ = o.fit(5, "wmrb", np.eye(n_u), np.eye(n_i), "linear", "linear", {"W": U0.astype(np.float64)},
                            {"W": V0.astype(np.float64)}, rows, cols, vals.astype(np.float64), samp, n_i, S, lr=0.1, dense=False)
    # the update is ~ lr*sign(g): a sign flip near g=0 moves one weight by 2*lr, so compare loosely and by fraction
    d = np.abs(cpu(m.user_embedding) - Eu)
    assert (d < 1e-4).mean() > 0.995, f"only {(d < 1e-4).mean():.4f} of user weights track the oracle trajectory"
    d = np.abs(cpu(m.item_embedding) - Ei)
    assert (d < 1e-4).mean() > 0.995


# ------------------------------------------------------------------------------- kernels through the raw C ABI


def test_spmm_seg_raw_abi_random_segments():
    from teamoflow_b200 import _abi
    from teamoflow_b200.mf._engine import spmm
    rng = np.random.default_rng(0)
    n_seg, n_src, r = 500, 300, 20
    lens = rng.integers(0, 6, n_seg)
    lens[7] = 4000; lens[8] = 0; lens[9] = 700; lens[499] = 1300  # spans many chunks, empty, long at the end
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    T = int(ptr[-1])
    idx = rng.integers(0, n_src, T).astype(np.int32)
    cpos = rng.permutation(T).astype(np.int32)
    coef = rng.standard_normal(T).astype(np.float32)
    src = np.zeros((n_src, 20), np.float32); src[:, :r] = rng.standard_normal((n_src, r))
    want = np.zeros((n_seg, r))
    seg_of = np.repeat(np.arange(n_seg), lens)
    np.add.at(want, seg_of, coef[cpos].astype(np.float64)[:, None] * src[idx].astype(np.float64))
    dev = "cuda"
    out = spmm(n_seg, torch.as_tensor(ptr, device=dev), T, torch.as_tensor(idx, device=dev), torch.as_tensor(cpos, device=dev),
               torch.as_tensor(coef, device=dev), torch.as_tensor(src, device=dev), r)
    close(cpu(out)[:, :r], want, name="spmm")
    assert _abi.call_count > 0


def test_transpose_and_sampler_and_initializers():
    from teamoflow_b200.mf._tensors import build_transpose
    from teamoflow_b200.mf.utils import random_sampler
    from teamoflow_b200.mf.initializer_graphs import NormalInitializer, UniformInitializer
    rng = np.random.default_rng(1)
    keys = rng.integers(0, 50, 10_000).astype(np.int32)
    ptr, perm = build_transpose(torch.as_tensor(keys, device="cuda"), 50)
    want_perm = np.argsort(keys, kind="stable")
    assert np.array_equal(cpu(perm), want_perm)
    assert np.array_equal(cpu(ptr), np.searchsorted(keys[want_perm], np.arange(51)))
    s = cpu(random_sampler(1000, 300, 64, seed=5))
    assert s.shape == (300, 64) and s.min() >= 0 and s.max() < 1000
    assert all(len(set(row)) == 64 for row in s)          # without replacement
    assert abs(s.mean() - 499.5) < 10                     # roughly uniform
    np.random.seed(3)
    a = cpu(random_sampler(40, 10, 7))
    np.random.seed(3)
    assert np.array_equal(a, o.random_sampler(40, 10, 7))  # the reference's own numpy statement, same stream
    W = cpu(NormalInitializer(seed=1).initialize_weights(1000, 10))
    assert abs(np.linalg.norm(W.astype(np.float64)) - 1.0) < 1e-5 and abs(W.mean()) < 2e-3
    Wn = W * np.sqrt(W.size)
    assert abs(Wn.std() - 1.0) < 0.05
    Wu = cpu(UniformInitializer(seed=2).initialize_weights(1000, 10))
    assert Wu.min() >= 0 and abs(np.linalg.norm(Wu.astype(np.float64)) - 1.0) < 1e-5


# ------------------------------------------------------------------------------- reference-test-shaped API smoke tests


def _toy():
    from teamoflow_b200.mf.utils import generate_random_interaction
    np.random.seed(0)
    sp, dense = generate_random_interaction(n_users=50, n_items=100, density=0.05)  # test/test_loss.py:14-16
    return sp, dense, torch.eye(50), torch.eye(100)


def test_reference_style_fit_all_losses_embeddings_initializers():
    """test/test_loss.py, test_embedding.py, test_initializer.py, test_predict.py of the reference, with the
    exception-swallowing removed."""
    E, I, L, eng, FM, SI, MF = _mods()
    from teamoflow_b200.mf.utils import generate_random_interaction
    sp, dense, uf, itf = _toy()
    m = MF(3)
    m.fit(epochs=25, user_features=uf, item_features=itf, tf_interactions=sp, verbose=False)
    assert m.predict().shape == (50, 100) and len(m.loss_history) == 1
    m = MF(3, loss_graph=L.WMRBLoss(), n_users=50, n_items=100, generate_sample=True)
    assert tuple(m.random_ind.shape) == (50, 50) and m.random_ind.dtype == torch.int64
    m.fit(25, user_features=uf, item_features=itf, tf_interactions=sp, lr=0.1, verbose=False)
    first = m.loss_history[0][1]
    assert np.isfinite(first)
    mixed, _ = generate_random_interaction(n_users=50, n_items=100, min_val=-5.0, max_val=5.0, density=0.01)
    m = MF(3, loss_graph=L.KLDivergenceLoss())
    m.fit(25, user_features=uf, item_features=itf, tf_interactions=mixed, lr=0.1, verbose=False)
    for emb in (E.LinearEmbedding(), E.BiasedLinearEmbedding(), E.ReLUEmbedding()):
        m = MF(3, user_repr_graph=emb)
        m.fit(epochs=25, user_features=uf, item_features=itf, tf_interactions=sp, verbose=False)
        assert len(m.user_trainable) == {"LinearEmbedding": 1, "BiasedLinearEmbedding": 2, "ReLUEmbedding": 3}[type(emb).__name__]
    for init in (I.NormalInitializer(), I.UniformInitializer()):
        m = MF(3, user_weight_graph=init, item_weight_graph=init)
        m.fit(epochs=25, user_features=uf, item_features=itf, tf_interactions=sp, verbose=False)
    cfg, res = m.save_model()
    assert cfg["Latent Dimension"] == 3 and res["User Embedding"].shape == (50, 3)
    with pytest.raises(TypeError):
        MF.from_saved(cfg)  # same quirk as the reference (keys are not constructor kwargs)
    assert isinstance(MF.from_saved({"n_components": 4}), MF)


def test_training_reduces_loss():
    E, I, L, eng, FM, SI, MF = _mods()
    sp, dense, uf, itf = _toy()
    m = MF(8, loss_graph=L.WMRBLoss(), user_weight_graph=I.UniformInitializer(seed=1), item_weight_graph=I.UniformInitializer(seed=2),
           n_users=50, n_items=100, n_samples=20, generate_sample=True)
    m.fit(100, uf, itf, sp, lr=0.05, verbose=False)
    losses = [l for _, l in m.loss_history]
    assert losses[-1] < losses[0]


def test_standalone_get_loss_and_get_repr_entry_points():
    E, I, L, eng, FM, SI, MF = _mods()
    from teamoflow_b200.mf.utils import gather_matrix_indices
    g = G["gather_matrix_indices"]
    out = gather_matrix_indices(torch.tensor(g["input"], dtype=torch.float32), torch.tensor(g["index"]))
    assert np.array_equal(cpu(out), np.array(g["expected"], np.float32))  # reference test/test_utils.py:47-61
    rng, rows, cols, vals, samp = make_problem(15, 22, 4, 90, 6, 2)
    P = rng.standard_normal((15, 22)).astype(np.float32)
    sp = SI(np.stack([rows, cols], 1), vals, (15, 22))
    close(cpu(L.MSELoss().get_loss(sp, torch.as_tensor(P))), o.mse_loss(rows, cols, vals, P.astype(np.float64)), name="mse")
    ss = o.gather_matrix_indices(P, samp)
    serial = P[rows, cols]
    got = L.WMRBLoss().get_loss(sp, torch.as_tensor(ss), torch.as_tensor(serial), 22, 6)
    close(cpu(got), o.wmrb_loss(rows, vals, ss.astype(np.float64), serial.astype(np.float64), 22, 6), name="wmrb")
    got = L.KLDivergenceLoss().get_loss(torch.as_tensor(serial), sp)
    close(cpu(got), o.kl_loss(serial.astype(np.float64), vals), name="kl")
    X = rng.standard_normal((15, 9)).astype(np.float32) * (rng.random((15, 9)) < 0.4)
    W = rng.standard_normal((9, 4)).astype(np.float32)
    emb, tr = E.LinearEmbedding().get_repr(torch.as_tensor(X), torch.as_tensor(W, device="cuda"))
    close(cpu(emb), X.astype(np.float64) @ W, name="linear repr")
    emb, tr = E.BiasedLinearEmbedding().get_repr(torch.as_tensor(X), torch.as_tensor(W, device="cuda"))
    assert len(tr) == 2 and float(tr[1].abs().sum()) == 0.0
    W5 = rng.standard_normal((20, 4)).astype(np.float32)
    emb, tr = E.ReLUEmbedding().get_repr(torch.as_tensor(X), torch.as_tensor(W5, device="cuda"))
    want = np.maximum(X.astype(np.float64) @ cpu(tr[1]) + cpu(tr[2]), 0) @ W5
    close(cpu(emb), want, name="relu repr")


# ------------------------------------------------------------------------------- edge cases


def test_edge_cases_empty_and_degenerate_inputs():
    E, I, L, eng, FM, SI, MF = _mods()
    rng = np.random.default_rng(0)
    # (1) no interactions at all: a step is a no-op on the weights (all gradients are exactly zero => Adam moves nothing)
    n_u, n_i, r = 9, 11, 4
    U0 = rng.standard_normal((n_u, r)).astype(np.float32); V0 = rng.standard_normal((n_i, r)).astype(np.float32)
    for loss, S in (("mse", 1), ("wmrb", 3)):
        samp = np.stack([rng.choice(n_i, S, replace=False) for _ in range(n_u)]).astype(np.int64)
        m = build_model(loss, ("linear", "linear"), {"W": U0}, {"W": V0}, r, n_u, n_i, S, samp)
        plan = m._prepare(FM.eye(n_u), FM.eye(n_i), SI(np.zeros((0, 2), np.int64), np.zeros(0, np.float32), (n_u, n_i)))
        plan.step(0.1)
        assert np.array_equal(cpu(plan.u.W)[:, :r], U0) and np.array_equal(cpu(plan.i.W)[:, :r], V0)
        assert plan.ip.loss_vector().numel() == 0
    # (2) WMRB where one user has only non-positive interactions and another has none
    rows = np.array([0, 0, 1, 3, 3]); cols = np.array([1, 4, 2, 0, 5]); vals = np.array([2.0, 1.0, -3.0, 5.0, -1.0], np.float32)
    S = 4
    samp = np.stack([rng.choice(n_i, S, replace=False) for _ in range(n_u)]).astype(np.int64)
    m = build_model("wmrb", ("linear", "linear"), {"W": U0}, {"W": V0}, r, n_u, n_i, S, samp)
    plan = m._prepare(FM.eye(n_u), FM.eye(n_i), SI(np.stack([rows, cols], 1), vals, (n_u, n_i)))
    plan.forward_backward()
    want = oracle64("wmrb", np.eye(n_u, dtype=np.float32), np.eye(n_i, dtype=np.float32), ("linear", "linear"), {"W": U0}, {"W": V0},
                    rows, cols, vals, samp, n_i, S, 0.1)
    close(cpu(plan.ip.loss_vector()), want[0], name="loss")
    close(cpu(plan.u.grads["W"])[:, :r], want[1]["W"], name="dU")
    assert np.all(cpu(plan.u.grads["W"])[1] == 0) and np.all(cpu(plan.u.grads["W"])[2] == 0)  # user 1: only a negative; user 2: nothing
    # (3) rank-1 model, a single sample, one interaction
    m = build_model("wmrb", ("linear", "linear"), {"W": U0[:, :1].copy()}, {"W": V0[:, :1].copy()}, 1, n_u, n_i, 1, samp[:, :1].copy())
    plan = m._prepare(FM.eye(n_u), FM.eye(n_i), SI(np.array([[2, 3]]), np.array([1.0], np.float32), (n_u, n_i)))
    plan.forward_backward()
    want = oracle64("wmrb", np.eye(n_u, dtype=np.float32), np.eye(n_i, dtype=np.float32), ("linear", "linear"), {"W": U0[:, :1]},
                    {"W": V0[:, :1]}, np.array([2]), np.array([3]), np.array([1.0], np.float32), samp[:, :1], n_i, 1, 0.1)
    close(cpu(plan.ip.loss_vector()), want[0], name="loss r=1")
    close(cpu(plan.i.grads["W"])[:, :1], want[2]["W"], name="dV r=1")
    # (4) argument validation mirrors numpy / the reference's failure modes
    from teamoflow_b200.mf.utils import random_sampler
    with pytest.raises(ValueError):
        random_sampler(5, 3, 6)  # n_samples > n_items without replacement
    with pytest.raises(ValueError):
        MF(3, loss_graph=L.WMRBLoss()).fit(1, torch.eye(4), torch.eye(5), SI(np.array([[0, 1]]), np.array([1.0], np.float32), (4, 5)))
    with pytest.raises(TypeError):
        MF(3, loss_graph=object()).fit(1, torch.eye(4), torch.eye(5), SI(np.array([[0, 1]]), np.array([1.0], np.float32), (4, 5)))


def test_heavy_users_are_split_and_still_deterministic_and_exact():
    """users above InteractionPlan.SPLIT interactions are processed as several slices + a fix-up; results must not change"""
    E, I, L, eng, FM, SI, MF = _mods()
    n_u, n_i, r, S = 6, 9000, 16, 20
    rng = np.random.default_rng(21)
    SP = eng.InteractionPlan.SPLIT
    eng.InteractionPlan.SPLIT_MIN, keep_min = SP, eng.InteractionPlan.SPLIT_MIN  # fixed slice length for this test
    lens = [2 * SP + 807, SP + 904, SP + 1, SP, 3, 0]  # 3, 2, 2, 1, 1, 0 slices
    rows = np.concatenate([np.full(n, u) for u, n in enumerate(lens)])
    cols = np.concatenate([np.sort(rng.choice(n_i, n, replace=False)) for n in lens]).astype(np.int64)
    vals = rng.choice(np.array([1.0, 2.0, -1.0], np.float32), rows.size)
    samp = np.stack([rng.choice(n_i, S, replace=False) for _ in range(n_u)]).astype(np.int64)
    pu = {"W": (rng.standard_normal((n_u, r)) * 0.2).astype(np.float32)}
    pi = {"W": (rng.standard_normal((n_i, r)) * 0.2).astype(np.float32)}
    for loss in ("wmrb", "mse"):
        m = build_model(loss, ("linear", "linear"), pu, pi, r, n_u, n_i, S, samp)
        plan = m._prepare(FM.eye(n_u), FM.eye(n_i), SI(np.stack([rows, cols], 1), vals, (n_u, n_i)))
        assert plan.ip.n_split == 3 and plan.ip.n_slots == 3 + 2 + 2
        plan.forward_backward()
        want = oracle64(loss, np.eye(n_u, dtype=np.float32), sparse.eye(n_i, dtype=np.float32, format="csr"), ("linear", "linear"),
                        pu, pi, rows, cols, vals, samp, n_i, S, 0.1)
        close(cpu(plan.ip.loss_vector()), want[0], name="loss")
        close(cpu(plan.u.grads["W"])[:, :r], want[1]["W"], name="dU")
        close(cpu(plan.i.grads["W"])[:, :r], want[2]["W"], name="dV")
        g1 = plan.u.grads["W"].clone()
        plan.forward_backward()
        assert torch.equal(g1, plan.u.grads["W"])
    eng.InteractionPlan.SPLIT_MIN = keep_min


# ------------------------------------------------------------------ SURVEY 8(f) extensions (defaults stay reference behaviour)


def _small_wmrb_model(seed=31, n_u=60, n_i=80, r=8, S=10, nnz=700):
    E, I, L, eng, FeatureMatrix, SparseInteractions, MatrixFactorization = _mods()
    rng, rows, cols, vals, samp = make_problem(n_u, n_i, r, nnz, S, seed, values=(1.0, 2.0, -1.0))
    U0 = (rng.standard_normal((n_u, r)) * 0.3).astype(np.float32)
    V0 = (rng.standard_normal((n_i, r)) * 0.3).astype(np.float32)
    model = MatrixFactorization(r, loss_graph=L.WMRBLoss(), user_weight_graph=fixed_init(U0), item_weight_graph=fixed_init(V0),
                                n_users=n_u, n_items=n_i, n_samples=S)
    model.random_ind = torch.as_tensor(samp, device="cuda")
    inter = SparseInteractions(np.stack([rows, cols], 1), vals, (n_u, n_i))
    return model, inter, FeatureMatrix, (rows, cols, vals, samp, U0, V0, n_u, n_i, r, S)


def test_stateful_adam_extension_matches_oracle():
    model, inter, FeatureMatrix, (rows, cols, vals, samp, U0, V0, n_u, n_i, r, S) = _small_wmrb_model()
    lr, epochs = 0.05, 3
    model.fit(epochs, FeatureMatrix.eye(n_u), FeatureMatrix.eye(n_i), inter, lr=lr, verbose=False, optimizer="adam")
    Xu, Xi = np.eye(n_u, dtype=np.float32), np.eye(n_i, dtype=np.float32)
    pu, pi = {"W": U0.copy()}, {"W": V0.copy()}
    mu, vu, mi, vi = (np.zeros_like(U0), np.zeros_like(U0), np.zeros_like(V0), np.zeros_like(V0))
    for t in range(1, epochs + 1):
        _, gu, gi, _, _ = o.train_step_sparse("wmrb", Xu, Xi, "linear", "linear", pu, pi, rows, cols, vals, samp, n_i, S, update=False)
        pu["W"], mu, vu = o.adam_step(pu["W"], gu["W"], mu, vu, t, lr)
        pi["W"], mi, vi = o.adam_step(pi["W"], gi["W"], mi, vi, t, lr)
    for got, want in ((model.user_trainable[0], pu["W"]), (model.item_trainable[0], pi["W"])):
        d = np.abs(cpu(got).astype(np.float64) - want)
        assert (d <= 2 * lr * epochs).all() and (d > 5e-5).mean() < 0.01


def test_cuda_graph_epoch_loop_is_bitwise_the_eager_loop():
    """fit() replays ONE captured CUDA graph of a step after the first epoch (TrainPlan.run); the trajectory must be the
    eager loop's bit for bit, for every loss / tower combination the step can launch."""
    E, I, L, eng, FM, SI, MF = _mods()
    n_u, n_i, r, S = 50, 70, 8, 12
    for loss, kinds in (("wmrb", ("linear", "linear")), ("mse", ("biased", "relu")), ("kl", ("relu", "biased"))):
        rng, rows, cols, vals, samp = make_problem(n_u, n_i, r, 600, S, 41, values=(1.0, 2.0, -1.0))
        pu, pi = params_for(kinds[0], n_u, r, rng, 0.5), params_for(kinds[1], n_i, r, rng, 0.5)
        out = []
        for use_graph in (True, False):
            m = build_model(loss, kinds, pu, pi, r, n_u, n_i, S, samp)
            keep = eng.TrainPlan.USE_CUDA_GRAPH
            eng.TrainPlan.USE_CUDA_GRAPH = use_graph
            try:
                m.fit(7, FM.eye(n_u), FM.eye(n_i), SI(np.stack([rows, cols], 1), vals, (n_u, n_i)), lr=0.05, verbose=False)
            finally:
                eng.TrainPlan.USE_CUDA_GRAPH = keep
            assert getattr(m._plan, "graph_replays", 0) == (6 if use_graph else 0)
            assert getattr(m._plan, "_graph", None) is None  # the captured step does not outlive fit()
            out.append([w.clone() for w in m.user_trainable + m.item_trainable] + [m.user_embedding.clone(), m.item_embedding.clone()])
        for a, b in zip(*out):
            assert torch.equal(a, b)


def test_fresh_optimizer_is_the_default_and_differs_from_stateful():
    model, inter, FeatureMatrix, (rows, cols, vals, samp, U0, V0, n_u, n_i, r, S) = _small_wmrb_model()
    model.fit(3, FeatureMatrix.eye(n_u), FeatureMatrix.eye(n_i), inter, lr=0.05, verbose=False)
    fresh = cpu(model.item_trainable[0]).copy()
    _, _, _, Ei_ref, _ = o.fit(3, "wmrb", np.eye(n_u, dtype=np.float32), np.eye(n_i, dtype=np.float32), "linear", "linear",
                               {"W": U0.copy()}, {"W": V0.copy()}, rows, cols, vals, samp, n_i, S, lr=0.05, dense=False)[:5]
    assert (np.abs(fresh - Ei_ref) > 5e-5).mean() < 0.02
    model.fit(3, FeatureMatrix.eye(n_u), FeatureMatrix.eye(n_i), inter, lr=0.05, verbose=False, optimizer="adam")
    assert np.abs(cpu(model.item_trainable[0]) - fresh).max() > 1e-3


def test_resample_every_extension_matches_oracle_with_the_drawn_tables():
    model, inter, FeatureMatrix, (rows, cols, vals, samp, U0, V0, n_u, n_i, r, S) = _small_wmrb_model(seed=32)
    lr = 0.05
    model.fit(4, FeatureMatrix.eye(n_u), FeatureMatrix.eye(n_i), inter, lr=lr, verbose=False, resample_every=2, resample_seed=99)
    assert [e for e, _ in model._sample_log] == [2]
    samp2 = cpu(model._sample_log[0][1])
    assert samp2.shape == samp.shape and not np.array_equal(samp2, samp)
    assert all(len(set(row)) == S and min(row) >= 0 and max(row) < n_i for row in samp2.tolist())  # without replacement
    Xu, Xi = np.eye(n_u, dtype=np.float32), np.eye(n_i, dtype=np.float32)
    pu, pi, _, _, _ = o.fit(2, "wmrb", Xu, Xi, "linear", "linear", {"W": U0.copy()}, {"W": V0.copy()}, rows, cols, vals, samp, n_i, S,
                            lr=lr, dense=False)
    pu, pi, _, _, _ = o.fit(2, "wmrb", Xu, Xi, "linear", "linear", pu, pi, rows, cols, vals, samp2, n_i, S, lr=lr, dense=False)
    for got, want in ((model.user_trainable[0], pu["W"]), (model.item_trainable[0], pi["W"])):
        d = np.abs(cpu(got).astype(np.float64) - want)
        assert (d <= 2 * lr * 4).all() and (d > 5e-5).mean() < 0.02
    # same seed, same draws
    model.fit(4, FeatureMatrix.eye(n_u), FeatureMatrix.eye(n_i), inter, lr=lr, verbose=False, resample_every=2, resample_seed=99)
    assert np.array_equal(cpu(model._sample_log[0][1]), samp2)


def test_save_and_load_round_trip(tmp_path):
    from teamoflow_b200.mf.matrix_factorization import MatrixFactorization
    model, inter, FeatureMatrix, (rows, cols, vals, samp, U0, V0, n_u, n_i, r, S) = _small_wmrb_model(seed=33)
    model.fit(2, FeatureMatrix.eye(n_u), FeatureMatrix.eye(n_i), inter, lr=0.05, verbose=False)
    path = str(tmp_path / "model.pt")
    model.save(path)
    again = MatrixFactorization.load(path)
    assert torch.equal(again.user_embedding, model.user_embedding) and torch.equal(again.item_embedding, model.item_embedding)
    assert torch.equal(again.random_ind, model.random_ind) and again.n_samples == model.n_samples
    assert type(again.loss_graph).__name__ == "WMRBLoss"
    assert np.array_equal(again.retrieve_user_recs(k=7), model.retrieve_user_recs(k=7))
    A = np.zeros((n_u, n_i), np.float32); A[rows, cols] = vals
    assert torch.equal(again.recall_at_k(torch.as_tensor(A), k=5), model.recall_at_k(torch.as_tensor(A), k=5))
    # and it can be trained again (weights are re-initialised by fit like the reference does)
    again.fit(1, FeatureMatrix.eye(n_u), FeatureMatrix.eye(n_i), inter, lr=0.05, verbose=False)


# ------------------------------------------------------------------------------- tensor-core GEMM (tcgen05, split-bf16)


@pytest.mark.parametrize("ta,tb", [(0, 0), (1, 0), (0, 1), (1, 1)])
@pytest.mark.parametrize("m,n,k", [(300, 70, 1000), (128, 64, 64), (1000, 160, 32), (320, 64, 50_000), (5, 3, 7)])
def test_gemm_tc_matches_fp64_to_fp32_accuracy(ta, tb, m, n, k):
    """tmf_gemm_tc (three exact bf16 planes per operand, six plane products per 64-wide k-block in TMEM, k-blocks added in fp32
    registers with round-to-nearest) against an fp64 product.  The error stays at the level of ONE k-block's tensor-core
    chain (measured 4-6e-7 sum|a||b|) however large K is -- without the per-block promotion it grew to 5e-6 at K = 2048."""
    from teamoflow_b200 import _abi
    rng = np.random.default_rng(m * 7 + n * 3 + k + ta * 2 + tb)
    A = (rng.standard_normal((k, m) if ta else (m, k)) * np.exp(rng.standard_normal((1, 1)))).astype(np.float32)
    B = (rng.standard_normal((n, k) if tb else (k, n))).astype(np.float32)
    A[0, 0] = 1e-20; B[0, 0] = 3e4  # small / large magnitudes survive the split
    want = (A.T if ta else A).astype(np.float64) @ (B.T if tb else B).astype(np.float64)
    bound = np.abs(A.T if ta else A).astype(np.float64) @ np.abs(B.T if tb else B).astype(np.float64)
    pad = lambda x: torch.nn.functional.pad(torch.as_tensor(x, device="cuda"), (0, (-x.shape[1]) % 4)).contiguous()  # noqa: E731
    At, Bt = pad(A), pad(B)
    out = torch.full((m, (n + 3) // 4 * 4 + 4), 7.0, device="cuda")  # an ldc wider than n: columns >= n must stay untouched
    need = _abi.query("tmf_gemm_tc_ws_bytes", m, n, k)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    _abi.call("tmf_gemm_tc", ta, tb, m, n, k, _abi.ptr(At), At.shape[1], _abi.ptr(Bt), Bt.shape[1], _abi.ptr(out), out.shape[1],
              _abi.ptr(ws), need)
    got = cpu(out)
    assert np.all(got[:, n:] == 7.0)
    err = np.abs(got[:, :n] - want)
    assert np.all(err <= 1.2e-6 * bound + 1e-30), f"max err/bound {np.max(err / (bound + 1e-300)):.3e}"
    # and in north_star's own terms (relative to the tensor's magnitude) on this random-sign, cancellation-heavy product
    assert err[1:, 1:].max() <= 1e-5 * np.abs(want[1:, 1:]).max(), f"max err / max|C| {err[1:, 1:].max() / np.abs(want[1:, 1:]).max():.3e}"
    out2 = torch.full_like(out, 7.0)
    _abi.call("tmf_gemm_tc", ta, tb, m, n, k, _abi.ptr(At), At.shape[1], _abi.ptr(Bt), Bt.shape[1], _abi.ptr(out2), out2.shape[1],
              _abi.ptr(ws), need)
    assert torch.equal(out, out2)  # deterministic (fixed K-split order)


@pytest.mark.parametrize("kinds", [("relu", "linear"), ("linear", "relu")])
def test_relu_tower_midsize_runs_its_gemms_on_the_tensor_cores(kinds):
    """Large enough that H.W, H^T.dE and dE.W^T go through tmf_gemm_tc (>= TC_GEMM_MIN_MACS): parity like test_step_parity."""
    _, _, _, eng, FM, SI, _ = _mods()
    n_u, n_i, r, S = 2500, 1800, 24, 6
    assert min(n_u, n_i) * r * 5 * r >= eng.TC_GEMM_MIN_MACS
    for seed in range(20):
        rng, rows, cols, vals, samp = make_problem(n_u, n_i, r, 30_000, S, 900 + seed)
        pu = params_for(kinds[0], n_u, r, rng, 0.3)
        pi = params_for(kinds[1], n_i, r, rng, 0.3)
        for p in (pu, pi):
            if "Wr" in p:  # identity features: X W_r is a row gather of the [n, 5r] table
                p["Wr"] = (p["Wr"] * 0.4).astype(np.float32)
        break
    from scipy import sparse
    Xu, Xi = sparse.identity(n_u, format="csr", dtype=np.float64), sparse.identity(n_i, format="csr", dtype=np.float64)
    f = lambda d: {k: v.astype(np.float64) for k, v in d.items()}  # noqa: E731
    want = o.train_step_sparse("mse", Xu, Xi, kinds[0], kinds[1], f(pu), f(pi), rows, cols, vals.astype(np.float64), samp, n_i, S, update=False)
    m = build_model("mse", kinds, pu, pi, r, n_u, n_i, S, samp)
    calls0 = dict(tc=0)
    from teamoflow_b200 import _abi
    real_call = _abi.call

    def counting(name, *a):
        calls0["tc"] += name == "tmf_gemm_tc"
        return real_call(name, *a)
    _abi.call = counting
    try:
        plan = m._prepare(FM.eye(n_u), FM.eye(n_i), SI(np.stack([rows, cols], 1), vals, (n_u, n_i)))
        plan.forward_backward()
    finally:
        _abi.call = real_call
    assert calls0["tc"] >= 3, "the ReLU tower's contractions did not reach the tensor-core GEMM"
    close(cpu(plan.ip.loss_vector()), want[0], name="loss")
    for tower, g in ((plan.u, want[1]), (plan.i, want[2])):
        for k in g:
            got = cpu(tower.grads[k])[:, :g[k].shape[1]]
            floor = np.abs(cpu(tower.dE)).sum(axis=0).max() if k in ("b", "br") else 0.0
            close(got, g[k], name=f"{tower.kind}.{k}", floor=floor)


def test_dense_features_stay_dense_and_use_the_tensor_core_gemm():
    """A genuinely dense feature matrix (every entry non-zero) is not exploded into CSR: X.W and X^T.dE are tmf_gemm_tc calls
    (embedding_graphs.py:38 with dense X; north_star: "a dense tcgen05/TMA GEMM only when the feature matrices are dense")."""
    _, _, _, eng, FM, SI, _ = _mods()
    from teamoflow_b200.mf._tensors import as_features
    n_u, n_i, r, S, Fu, Fi = 2000, 1500, 32, 8, 96, 80
    rng, rows, cols, vals, samp = make_problem(n_u, n_i, r, 20_000, S, 77)
    Xu = rng.standard_normal((n_u, Fu)).astype(np.float32)
    Xi = rng.standard_normal((n_i, Fi)).astype(np.float32)
    assert as_features(torch.as_tensor(Xu)).dense is not None
    sparse_like = np.where(rng.random((50, 40)) < 0.1, 1.0, 0.0).astype(np.float32)
    assert as_features(torch.as_tensor(sparse_like)).dense is None  # a mostly-zero dense tensor still becomes CSR
    pu = {"W": (rng.standard_normal((Fu, r)) * 0.1).astype(np.float32), "b": np.zeros((1, r), np.float32)}
    pi = {"W": (rng.standard_normal((Fi, r)) * 0.1).astype(np.float32)}
    want = oracle64("mse", Xu, Xi, ("biased", "linear"), pu, pi, rows, cols, vals, samp, n_i, S, 0.01)
    m = build_model("mse", ("biased", "linear"), pu, pi, r, n_u, n_i, S, samp)
    plan = m._prepare(torch.as_tensor(Xu), torch.as_tensor(Xi), SI(np.stack([rows, cols], 1), vals, (n_u, n_i)))
    assert plan.u.X.dense is not None and plan.i.X.dense is not None
    plan.forward_backward()
    close(cpu(plan.ip.loss_vector()), want[0], name="loss")
    close(cpu(plan.u.grads["W"])[:, :r], want[1]["W"], name="dWu (X^T dE, dense X)")
    close(cpu(plan.u.grads["b"])[:, :r], want[1]["b"], name="db", floor=np.abs(cpu(plan.u.dE)).sum(axis=0).max())
    close(cpu(plan.i.grads["W"])[:, :r], want[2]["W"], name="dWi")
    Eu, _ = o.embed_forward("biased", Xu.astype(np.float64), {k: v.astype(np.float64) for k, v in pu.items()})
    close(cpu(plan.u.E)[:, :r], Eu, name="E_u = X W + b")


def test_item_major_coefficient_layout_is_bitwise_the_gather_layout():
    """The user pass may store c_k / G_uj straight into the item-major slots (coef_pos) so that the item pass streams them;
    the sums run over the same values in the same order, so every gradient is bit-identical to the gather layout --
    including split (heavy) users, whose G is finished by the fix-up kernel, and users without interactions."""
    _, _, _, eng, FM, SI, _ = _mods()
    n_u, n_i, r, S = 700, 900, 16, 24
    rng = np.random.default_rng(4)
    lens = np.minimum((3000.0 / np.arange(1, n_u + 1)).astype(np.int64), n_i)
    lens[5] = 0
    rows = np.repeat(np.arange(n_u), lens)
    cols = np.concatenate([np.sort(rng.choice(n_i, l, replace=False)) for l in lens])
    vals = rng.choice(np.array([1.0, 2.0, -1.0], np.float32), rows.size)
    samp = np.stack([rng.choice(n_i, S, replace=False) for _ in range(n_u)]).astype(np.int64)
    pu = {"W": (rng.standard_normal((n_u, r)) * 0.3).astype(np.float32)}
    pi = {"W": (rng.standard_normal((n_i, r)) * 0.3).astype(np.float32)}
    res = {}
    keep = eng.InteractionPlan.DIRECT_COEF, eng.InteractionPlan.SPLIT
    try:
        eng.InteractionPlan.SPLIT = 128  # the heaviest users (up to 900 interactions) are processed as slices
        for loss in ("wmrb", "mse"):
            for direct in (True, False):
                eng.InteractionPlan.DIRECT_COEF = direct
                m = build_model(loss, ("linear", "linear"), pu, pi, r, n_u, n_i, S, samp)
                plan = m._prepare(FM.eye(n_u), FM.eye(n_i), SI(np.stack([rows, cols], 1), vals, (n_u, n_i)))
                assert (plan.ip.coef_pos is not None) == direct and plan.ip.n_split > 0
                plan.forward_backward()
                res[(loss, direct)] = (plan.u.dE.clone(), plan.i.dE.clone(), plan.ip.loss_k.clone())
            for a, b in zip(res[(loss, True)], res[(loss, False)]):
                assert torch.equal(a, b), loss
    finally:
        eng.InteractionPlan.DIRECT_COEF, eng.InteractionPlan.SPLIT = keep
    want = oracle64("wmrb", np.eye(n_u, dtype=np.float32), np.eye(n_i, dtype=np.float32), ("linear", "linear"), pu, pi, rows, cols, vals,
                    samp, n_i, S, 0.1)
    close(cpu(res[("wmrb", True)][1])[:, :r], want[2]["W"], name="dE_i (item-major coefficients)")
