"""Golden vectors produced by the REFERENCE'S OWN SOURCE (``$TMF_REFERENCE_ROOT/src/teamoflow/mf``, imported unmodified)
executed over the TensorFlow stand-in in ``tests/golden/tf_shim`` (no TensorFlow needed).

    TMF_REFERENCE_ROOT=<checkout of the original TeAMOFlow> python tests/golden/make_ref_golden.py   # writes tests/golden/ref_golden.json

Needs a checkout of the original project, which is not part of this repository; the JSON travels with the repo.  See
tf_shim/README.md for what these vectors pin (the reference's Python logic) and what they do not (TensorFlow's kernels).
"""
import contextlib
import io
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("TMF_REFERENCE_ROOT", "")


def load_reference():
    if not os.path.isdir(os.path.join(REF, "src", "teamoflow", "mf")):
        sys.exit("make_ref_golden.py: set TMF_REFERENCE_ROOT to a checkout of the original TeAMOFlow project "
                 f"(no src/teamoflow/mf under {REF!r})")
    sys.path.insert(0, os.path.join(HERE, "tf_shim"))
    sys.path.insert(0, REF)
    import tensorflow as tf  # the shim
    from src.teamoflow.mf import embedding_graphs, initializer_graphs, loss_graphs, matrix_factorization, utils
    return tf, matrix_factorization, loss_graphs, embedding_graphs, initializer_graphs, utils


def L(x):
    """tensor / ndarray -> nested python lists (floats survive a JSON round trip exactly: repr of float32 as float64)."""
    if hasattr(x, "detach"):
        x = x.detach().cpu().numpy()
    x = np.asarray(x)
    out = x.astype(np.float64) if x.dtype.kind == "f" else x
    return json.loads(json.dumps(out.tolist()).replace("NaN", '"nan"').replace("-Infinity", '"-inf"').replace("Infinity", '"inf"'))


def build():
    tf, mfm, lg, eg, ig, ut = load_reference()
    rng = np.random.default_rng(20241018)
    G = {"_about": "made by tests/golden/make_ref_golden.py: reference source over tests/golden/tf_shim (torch-CPU fp32)"}

    class Fixed(ig.Initializer):  # the reference's own ABC: only initialize_weights(n_features, n_components) is called (fit :115-123)
        def __init__(self, W):
            self.W = W

        def initialize_weights(self, n_features, n_components):
            assert self.W.shape == (n_features, n_components)
            return tf.Variable(tf.constant(self.W, dtype=tf.float32), trainable=True)

    # ---- utils.gather_matrix_indices: the reference's only known-answer vector (test/test_utils.py:47-61)
    inp = [[1, 4, 2], [5, 7, 8], [6, 2, 1]]
    idx = [[0, 2, 0], [2, 2, 2], [2, 1, 0]]
    G["gather_matrix_indices"] = {"input": inp, "index": idx,
                                  "out": L(ut.gather_matrix_indices(tf.constant(inp, dtype=tf.float32), tf.constant(idx, dtype=tf.int64)))}

    # ---- interaction table with positive, negative and empty rows (the reference's generator, then signs / holes)
    n_u, n_i, r, S = 14, 17, 5, 6
    np.random.seed(7)  # scipy.sparse.random inside generate_random_interaction draws from numpy's global RNG
    inter, A = ut.generate_random_interaction(n_u, n_i, min_val=0.0, max_val=5.0, density=0.3)
    rows = inter.indices[:, 0].numpy(); cols = inter.indices[:, 1].numpy(); vals = inter.values.numpy().copy()
    G["generate_random_interaction"] = {"rows": L(rows), "cols": L(cols), "vals": L(vals), "A": L(A)}
    neg = rng.random(vals.size) < 0.25
    vals[neg] *= -1
    keep = rows != 3  # user 3 has no interactions at all
    rows, cols, vals = rows[keep], cols[keep], vals[keep]
    A2 = np.zeros((n_u, n_i), np.float32); A2[rows, cols] = vals
    inter2 = tf.sparse.SparseTensor(indices=np.stack([rows, cols], 1), values=tf.constant(vals, dtype=tf.float32), dense_shape=(n_u, n_i))
    samp = np.stack([rng.choice(n_i, S, replace=False) for _ in range(n_u)]).astype(np.int64)
    G["data"] = {"n_users": n_u, "n_items": n_i, "r": r, "S": S, "rows": L(rows), "cols": L(cols), "vals": L(vals), "samp": L(samp)}

    # ---- loss graphs called directly (loss_graphs.py:36-122) on given predictions
    P = (rng.standard_normal((n_u, n_i)) * 0.7).astype(np.float32)
    Pt = tf.constant(P, dtype=tf.float32)
    serial = tf.gather_nd(params=Pt, indices=inter2.indices)
    sample_preds = ut.gather_matrix_indices(Pt, tf.constant(samp, dtype=tf.int64))
    G["loss_graphs"] = {
        "P": L(P),
        "mse": L(lg.MSELoss().get_loss(tf_interactions=inter2, predictions=Pt)),
        "wmrb": L(lg.WMRBLoss().get_loss(tf_interactions=inter2, tf_sample_predictions=sample_preds, tf_prediction_serial=serial,
                                         n_items=n_i, n_samples=S)),
        "kl": L(lg.KLDivergenceLoss().get_loss(tf_prediction_serial=serial, tf_interactions=inter2)),
    }

    # ---- fit: one and two full-batch steps from injected weights (matrix_factorization.py:96-187)
    Xu_id, Xi_id = np.eye(n_u, dtype=np.float32), np.eye(n_i, dtype=np.float32)
    Xu_ft = np.concatenate([Xu_id, (rng.random((n_u, 4)) < 0.4).astype(np.float32)], 1)   # [I | M] side features, dense like the reference needs
    Xi_ft = np.concatenate([Xi_id, (rng.random((n_i, 3)) < 0.4).astype(np.float32)], 1)
    embed_cls = {"linear": eg.LinearEmbedding, "biased": eg.BiasedLinearEmbedding, "relu": eg.ReLUEmbedding}
    loss_cls = {"mse": lg.MSELoss, "wmrb": lg.WMRBLoss, "kl": lg.KLDivergenceLoss}
    fits = []
    cases = [("mse", "linear", "linear", "id", 1e-2), ("wmrb", "linear", "linear", "id", 0.1), ("kl", "linear", "linear", "id", 1e-2),
             ("wmrb", "linear", "linear", "feat", 0.1), ("mse", "biased", "biased", "feat", 1e-2), ("wmrb", "biased", "linear", "id", 0.05),
             ("wmrb", "relu", "relu", "id", 0.05), ("mse", "relu", "biased", "feat", 1e-2), ("kl", "biased", "relu", "id", 1e-2)]
    for loss, ku, ki, feat, lr in cases:
        Xu, Xi = (Xu_id, Xi_id) if feat == "id" else (Xu_ft, Xi_ft)
        Fu, Fi = Xu.shape[1], Xi.shape[1]
        aux = 5 * r
        Wu0 = (rng.standard_normal((aux if ku == "relu" else Fu, r)) * 0.3).astype(np.float32)
        Wi0 = (rng.standard_normal((aux if ki == "relu" else Fi, r)) * 0.3).astype(np.float32)
        extra = {}
        for epochs in (1, 2):
            model = mfm.MatrixFactorization(r, user_repr_graph=embed_cls[ku](), item_repr_graph=embed_cls[ki](), loss_graph=loss_cls[loss](),
                                            user_weight_graph=Fixed(Wu0), item_weight_graph=Fixed(Wi0), n_users=n_u, n_items=n_i, n_samples=S)
            model.random_ind = tf.constant(samp, dtype=tf.int64)  # read at matrix_factorization.py:153
            if ku == "relu":
                if "u_rw" not in extra:
                    extra["u_rw"] = (rng.standard_normal((Fu, aux)) * 0.5).astype(np.float32)
                    extra["u_rb"] = (rng.standard_normal((1, aux)) * 0.1).astype(np.float32)
                model.user_relu_weight = tf.Variable(tf.constant(extra["u_rw"], dtype=tf.float32))
                model.user_relu_bias = tf.Variable(tf.constant(extra["u_rb"], dtype=tf.float32))
            if ki == "relu":
                if "i_rw" not in extra:
                    extra["i_rw"] = (rng.standard_normal((Fi, aux)) * 0.5).astype(np.float32)
                    extra["i_rb"] = (rng.standard_normal((1, aux)) * 0.1).astype(np.float32)
                model.item_relu_weight = tf.Variable(tf.constant(extra["i_rw"], dtype=tf.float32))
                model.item_relu_bias = tf.Variable(tf.constant(extra["i_rb"], dtype=tf.float32))
            with contextlib.redirect_stdout(io.StringIO()):
                model.fit(epochs, tf.constant(Xu), tf.constant(Xi), inter2, lr=lr)
            rec = {"user_embedding": L(model.user_embedding), "item_embedding": L(model.item_embedding),
                   "user_trainable": [L(v) for v in model.user_trainable], "item_trainable": [L(v) for v in model.item_trainable]}
            if epochs == 1:
                one = rec
        fits.append({"loss": loss, "user": ku, "item": ki, "features": feat, "lr": lr, "Wu0": L(Wu0), "Wi0": L(Wi0),
                     "relu": {k: L(v) for k, v in extra.items()}, "after1": one, "after2": rec})
    G["fit"] = {"Xu_feat": L(Xu_ft), "Xi_feat": L(Xi_ft), "cases": fits}

    # ---- evaluation surface on GRID-VALUED embeddings (every score exact in fp32 => order independent of blocking, many ties)
    Ug = rng.integers(-4, 5, (n_u, r)).astype(np.float32) / 8
    Vg = rng.integers(-4, 5, (n_i, r)).astype(np.float32) / 8
    Ug[5] = -np.abs(Ug[5]); Vg[:] = Vg  # keep mixed signs; row 5 mostly non-positive scores
    Ug[6] = 0.0                          # an all-zero score row: clamp ties resolve to the lowest item ids
    model = mfm.MatrixFactorization(r)
    model.user_embedding, model.item_embedding = tf.constant(Ug), tf.constant(Vg)
    At = tf.constant(A2)
    ev = {"U": L(Ug), "V": L(Vg), "A": L(A2), "predict": L(model.predict()), "predict_unobserved": L(model.predict(At)[1]),
          "predict_ranks": L(model.predict_ranks(At))}
    for k in (3, 5, 17):
        ev[f"k{k}"] = {
            "recall": L(model.recall_at_k(At, k=k)), "recall_keep": L(model.recall_at_k(At, k=k, preserve_rows=True)),
            "precision": L(model.precision_at_k(At, k=k)), "precision_keep": L(model.precision_at_k(At, k=k, preserve_rows=True)),
            "f1": L(model.f1_at_k(At, k=k)), "f1_beta2": L(model.f1_at_k(At, k=k, beta=2.0)),
            "dcg": L(model.dcg_at_k(At, k=k)), "idcg": L(model.idcg_at_k(At, k=k)),
            "ndcg": L(model.ndcg_at_k(At, k=k)), "ndcg_keep": L(model.ndcg_at_k(At, k=k, preserve_rows=True)),
            "recs_all": L(model.retrieve_user_recs(k=k)), "recs_user2": L(model.retrieve_user_recs(user=2, k=k)),
        }
    ev["recs_user9_full"] = L(model.retrieve_user_recs(user=9))
    ev["recs_full"] = L(model.retrieve_user_recs())
    G["evaluate"] = ev

    # ---- embedding graphs called directly (embedding_graphs.py:30-87)
    X = tf.constant(Xu_ft)
    W = (rng.standard_normal((Xu_ft.shape[1], r)) * 0.3).astype(np.float32)
    b = (rng.standard_normal((1, r)) * 0.2).astype(np.float32)
    Wr = (rng.standard_normal((Xu_ft.shape[1], 5 * r)) * 0.5).astype(np.float32)
    br = (rng.standard_normal((1, 5 * r)) * 0.1).astype(np.float32)
    W5 = (rng.standard_normal((5 * r, r)) * 0.3).astype(np.float32)
    G["embeddings"] = {
        "X": L(Xu_ft), "W": L(W), "b": L(b), "Wr": L(Wr), "br": L(br), "W5": L(W5),
        "linear": L(eg.LinearEmbedding().get_repr(X, tf.constant(W))[0]),
        "biased": L(eg.BiasedLinearEmbedding().get_repr(X, tf.constant(W), linear_bias=tf.constant(b))[0]),
        "relu": L(eg.ReLUEmbedding().get_repr(X, tf.constant(W5), relu_weight=tf.constant(Wr), relu_bias=tf.constant(br))[0]),
    }
    # ---- initializers: only properties can be pinned (the RNG streams differ): ||W||_F == 1, shape, trainable
    Wn = ig.NormalInitializer().initialize_weights(9, 4)
    Wuf = ig.UniformInitializer().initialize_weights(9, 4)
    G["initializers"] = {"normal_fro": float((Wn.detach() ** 2).sum().sqrt()), "uniform_fro": float((Wuf.detach() ** 2).sum().sqrt()),
                         "uniform_min": float(Wuf.detach().min()), "shape": list(Wn.shape)}
    return G


if __name__ == "__main__":
    G = build()
    out = os.path.join(HERE, "ref_golden.json")
    with open(out, "w") as f:
        json.dump(G, f)
    print("wrote", out, os.path.getsize(out), "bytes")
