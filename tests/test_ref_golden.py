"""The oracle against golden vectors produced by the REFERENCE'S OWN SOURCE run over tests/golden/tf_shim
(tests/golden/make_ref_golden.py; TensorFlow itself is not installable here).  CPU only."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import mf_oracle as o

HERE = os.path.dirname(os.path.abspath(__file__))
G = json.load(open(os.path.join(HERE, "golden", "ref_golden.json")))


def arr(x, dtype=np.float32):
    def conv(v):
        if isinstance(v, list):
            return [conv(t) for t in v]
        return float(v) if isinstance(v, str) else v
    return np.asarray(conv(x), dtype=dtype)


D = G["data"]
ROWS, COLS, VALS = arr(D["rows"], np.int64), arr(D["cols"], np.int64), arr(D["vals"])
SAMP = arr(D["samp"], np.int64)
N_U, N_I, R, S = D["n_users"], D["n_items"], D["r"], D["S"]


def fit_inputs(case):
    Xu = np.eye(N_U, dtype=np.float32) if case["features"] == "id" else arr(G["fit"]["Xu_feat"])
    Xi = np.eye(N_I, dtype=np.float32) if case["features"] == "id" else arr(G["fit"]["Xi_feat"])
    pu, pi = {"W": arr(case["Wu0"])}, {"W": arr(case["Wi0"])}
    for side, kind, p in (("u", case["user"], pu), ("i", case["item"], pi)):
        if kind == "biased":
            p["b"] = np.zeros((1, R), np.float32)  # created as zeros on the first get_repr (embedding_graphs.py:55)
        if kind == "relu":
            p["Wr"], p["br"] = arr(case["relu"][f"{side}_rw"]), arr(case["relu"][f"{side}_rb"])
    return Xu, Xi, pu, pi


def trainables(kind, p):
    return [p["W"]] if kind == "linear" else [p["W"], p["b"]] if kind == "biased" else [p["W"], p["Wr"], p["br"]]


def close_update(got, want, lr, what):
    """Weights after fresh-Adam steps: |delta| ~ lr per entry with a sign-like dependence on the gradient, so an entry whose
    gradient is ~1e-6 may legitimately land elsewhere; everything else must agree to fp32 accuracy."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape, what
    diff = np.abs(got - want)
    assert (diff <= 2.0 * lr + 1e-6).all(), what
    assert (diff > 2e-5).mean() <= 0.01, f"{what}: {(diff > 2e-5).mean():.3%} of the entries differ"


def test_gather_matrix_indices_reference_vector():
    c = G["gather_matrix_indices"]
    assert np.array_equal(o.gather_matrix_indices(arr(c["input"]), arr(c["index"], np.int64)), arr(c["out"]))


def test_loss_graphs_match_reference_source():
    c = G["loss_graphs"]
    P = arr(c["P"])
    p = P[ROWS, COLS]
    np.testing.assert_allclose(o.mse_loss(ROWS, COLS, VALS, P), arr(c["mse"]), rtol=1e-6, atol=1e-7)
    ss = o.gather_matrix_indices(P, SAMP)
    np.testing.assert_allclose(o.wmrb_loss(ROWS, VALS, ss, p, N_I, S), arr(c["wmrb"]), rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(o.kl_loss(p, VALS), arr(c["kl"]), rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("ci", range(len(G["fit"]["cases"])))
@pytest.mark.parametrize("dense", [True, False])
def test_fit_steps_match_reference_source(ci, dense):
    case = G["fit"]["cases"][ci]
    Xu, Xi, pu, pi = fit_inputs(case)
    for epochs, key in ((1, "after1"), (2, "after2")):
        npu, npi, Eu, Ei, _ = o.fit(epochs, case["loss"], Xu, Xi, case["user"], case["item"], dict(pu), dict(pi), ROWS, COLS, VALS,
                                    SAMP, N_I, S, lr=case["lr"], dense=dense)
        want = case[key]
        tag = f"{case['loss']}/{case['user']}/{case['item']}/{case['features']} epochs={epochs}"
        for got, w in zip(trainables(case["user"], npu), want["user_trainable"]):
            close_update(got, arr(w), case["lr"], tag + " user trainable")
        for got, w in zip(trainables(case["item"], npi), want["item_trainable"]):
            close_update(got, arr(w), case["lr"], tag + " item trainable")
        if case["user"] != "relu":
            close_update(Eu, arr(want["user_embedding"]), case["lr"] * (1 + np.abs(Xu).sum(1).max()), tag + " user embedding")
        if case["item"] != "relu":
            close_update(Ei, arr(want["item_embedding"]), case["lr"] * (1 + np.abs(Xi).sum(1).max()), tag + " item embedding")


def test_embedding_graphs_match_reference_source():
    c = G["embeddings"]
    X = arr(c["X"])
    np.testing.assert_allclose(o.embed_forward("linear", X, {"W": arr(c["W"])})[0], arr(c["linear"]), rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(o.embed_forward("biased", X, {"W": arr(c["W"]), "b": arr(c["b"])})[0], arr(c["biased"]), rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(o.embed_forward("relu", X, {"W": arr(c["W5"]), "Wr": arr(c["Wr"]), "br": arr(c["br"])})[0], arr(c["relu"]),
                               rtol=1e-5, atol=1e-5)


def test_evaluation_surface_matches_reference_source():
    e = G["evaluate"]
    U, V, A = arr(e["U"]), arr(e["V"]), arr(e["A"])
    P = o.canonical_scores(U, V)
    assert np.array_equal(P, arr(e["predict"]))  # grid-valued embeddings: exact in any summation order
    assert np.array_equal(o.predict(U, V, A)[1], arr(e["predict_unobserved"]))
    assert np.array_equal(o.predict_ranks(U, V, A), arr(e["predict_ranks"], np.int64))
    for k in (3, 5, 17):
        w = e[f"k{k}"]
        np.testing.assert_array_equal(o.recall_at_k(P, A, k), arr(w["recall"]))
        np.testing.assert_array_equal(o.recall_at_k(P, A, k, preserve_rows=True), arr(w["recall_keep"]))
        np.testing.assert_array_equal(o.precision_at_k(P, A, k), arr(w["precision"]))
        np.testing.assert_array_equal(o.precision_at_k(P, A, k, preserve_rows=True), arr(w["precision_keep"]))
        np.testing.assert_allclose(o.f1_at_k(P, A, k), arr(w["f1"]), rtol=1e-6)
        np.testing.assert_allclose(o.f1_at_k(P, A, k, beta=2.0), arr(w["f1_beta2"]), rtol=1e-6)
        np.testing.assert_allclose(o.dcg_at_k(P, A, k), arr(w["dcg"]), rtol=2e-6, atol=1e-6)
        np.testing.assert_allclose(o.idcg_at_k(P, A, k), arr(w["idcg"]), rtol=2e-6, atol=1e-6)
        np.testing.assert_allclose(o.ndcg_at_k(P, A, k), arr(w["ndcg"]), rtol=4e-6, atol=1e-6)
        np.testing.assert_allclose(o.ndcg_at_k(P, A, k, preserve_rows=True), arr(w["ndcg_keep"]), rtol=4e-6, atol=1e-6)
        assert np.array_equal(o.retrieve_user_recs(P, k=k), arr(w["recs_all"], np.int64))
        assert np.array_equal(o.retrieve_user_recs(P, user=2, k=k), arr(w["recs_user2"], np.int64))
    assert np.array_equal(o.retrieve_user_recs(P, user=9), arr(e["recs_user9_full"], np.int64))
    assert np.array_equal(o.retrieve_user_recs(P), arr(e["recs_full"], np.int64))


def test_generate_random_interaction_structure():
    c = G["generate_random_interaction"]
    rows, cols, vals, A = arr(c["rows"], np.int64), arr(c["cols"], np.int64), arr(c["vals"]), arr(c["A"])
    order = np.lexsort((cols, rows))
    assert np.array_equal(order, np.arange(rows.size))        # row-major sorted indices (utils.py:53-57)
    assert (vals != 0).all() and np.array_equal(vals, np.round(vals)) and np.array_equal(A[rows, cols], vals)
    assert np.count_nonzero(A) == rows.size
    (r2, c2, v2), A2 = o.generate_random_interaction(14, 17, 0.0, 5.0, 0.3, random_state=1)
    assert np.array_equal(np.lexsort((c2, r2)), np.arange(r2.size)) and (v2 != 0).all() and np.array_equal(A2[r2, c2], v2)


def test_initializer_properties():
    c = G["initializers"]
    assert abs(c["normal_fro"] - 1) < 1e-5 and abs(c["uniform_fro"] - 1) < 1e-5 and c["uniform_min"] >= 0 and c["shape"] == [9, 4]
    W = o.uniform_initializer(9, 4, np.random.default_rng(0))
    assert abs(np.sqrt((W.astype(np.float64) ** 2).sum()) - 1) < 1e-6 and W.min() >= 0


REF_ROOT = os.environ.get("TMF_REFERENCE_ROOT")


@pytest.mark.skipif(not (REF_ROOT and os.path.isdir(os.path.join(REF_ROOT, "src", "teamoflow", "mf"))),
                    reason="needs TMF_REFERENCE_ROOT: a checkout of the original TeAMOFlow source")
def test_committed_goldens_are_what_the_reference_source_produces():
    """Re-run the generator (reference source over the shim) and compare with the committed JSON."""
    code = ("import sys, json; sys.path.insert(0, %r); import make_ref_golden as m; print(json.dumps(m.build()))"
            % os.path.join(HERE, "golden"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    fresh = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("gather_matrix_indices", "loss_graphs", "evaluate", "embeddings", "data"):
        assert fresh[key] == G[key], key
    for a, b in zip(fresh["fit"]["cases"], G["fit"]["cases"]):
        for k in ("after1", "after2"):
            for got, want in zip(a[k]["item_trainable"] + a[k]["user_trainable"], b[k]["item_trainable"] + b[k]["user_trainable"]):
                np.testing.assert_allclose(arr(got), arr(want), rtol=0, atol=1e-6)
