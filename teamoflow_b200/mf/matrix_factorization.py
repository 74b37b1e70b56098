"""``MatrixFactorization`` -- same class, constructor, methods and attributes as the reference
``src/teamoflow/mf/matrix_factorization.py`` (cited below as ``ref:LINE``), with the TensorFlow op
sequence replaced by hand-written sm_100a kernels behind the C ABI of ``include/tmf.h``.

Differences that are deliberate and documented in DESIGN.md:
  * tensors are torch CUDA tensors; sparse interactions are ``SparseInteractions``
    (``indices`` / ``values`` / ``dense_shape`` like ``tf.sparse.SparseTensor``);
  * features / interaction tables may also be given sparse (scipy / torch) -- the reference's dense
    ``[n_users, n_items]`` prediction matrix is never formed during training or top-k;
  * scores used for ranking are the canonical fp32 score (fp64-accumulated dot product rounded to
    fp32), which makes top-k indices independent of GEMM blocking.
"""
import timeit as t

import numpy as np
import torch

from .. import _abi
from . import _engine as eng
from ._tensors import FeatureMatrix, SparseInteractions, as_features, as_interactions, device, to_device
from .embedding_graphs import *  # noqa: F401,F403  (the reference re-exports these, ref:16)
from .embedding_graphs import BiasedLinearEmbedding, LinearEmbedding, ReLUEmbedding, new_relu_params
from .initializer_graphs import NormalInitializer
from .loss_graphs import *  # noqa: F401,F403  (ref:17)
from .loss_graphs import KLDivergenceLoss, MSELoss, WMRBLoss
from .predict_graphs import dense_scores
from .utils import gather_matrix_indices, random_sampler  # noqa: F401  (ref:20)

# the fused tcgen05 top-k kernel keeps at most this many results per row; larger k (full rankings)
# go through dense canonical scores + a segmented sort
TOPK_FUSED_MAX_K = 1024


def _public(st, r):
    return st[:, :r]


class MatrixFactorization:
    """Standard matrix-factorization model with pluggable embeddings, loss and initializers (ref:23)."""

    def __init__(self, n_components, user_repr_graph=LinearEmbedding(), item_repr_graph=LinearEmbedding(), loss_graph=MSELoss(), user_weight_graph=NormalInitializer(), item_weight_graph=NormalInitializer(), n_users=None, n_items=None, n_samples=None, generate_sample=False):
        """Same arguments and defaults as ref:28-50."""
        self.n_components = n_components
        self.user_repr_graph = user_repr_graph
        self.item_repr_graph = item_repr_graph
        self.loss_graph = loss_graph
        self.user_weight_graph = user_weight_graph
        self.item_weight_graph = item_weight_graph

        self.n_users = n_users
        self.n_items = n_items
        self.n_samples = n_samples
        self.random_ind = None
        self.generate_sample = generate_sample

        # ref:68-69 -- default sample size is half of the items
        if n_samples is None and n_items is not None:
            self.n_samples = n_items // 2

        # ref:72-73 -- negatives are sampled ONCE per model and never refreshed
        if generate_sample == True:  # noqa: E712
            self.random_ind = random_sampler(n_items, n_users, self.n_samples)

        # ref:76-79
        if isinstance(self.user_repr_graph, ReLUEmbedding):
            self.user_aux_dim = 5 * self.n_components
        if isinstance(self.item_repr_graph, ReLUEmbedding):
            self.item_aux_dim = 5 * self.n_components

        # ref:82-90
        self.user_relu_bias = None
        self.user_relu_weight = None
        self.item_relu_bias = None
        self.item_relu_weight = None
        self.user_linear_bias = None
        self.item_linear_bias = None

        # ref:93-94
        self.user_trainable = None
        self.item_trainable = None

        self.loss_history = []
        self._plan = None

    # ------------------------------------------------------------------ training

    def _loss_kind(self):
        # the reference dispatches on isinstance (ref:152-162); an unknown LossGraph fails there too
        for cls, kind in ((WMRBLoss, eng.WMRB), (MSELoss, eng.MSE), (KLDivergenceLoss, eng.KL)):
            if isinstance(self.loss_graph, cls):
                return kind
        raise TypeError("loss_graph must be an MSELoss, WMRBLoss or KLDivergenceLoss instance "
                        "(the reference's fit dispatches on exactly these, matrix_factorization.py:152-162)")

    @staticmethod
    def _embed_kind(graph):
        for cls, kind in ((ReLUEmbedding, eng.RELU), (BiasedLinearEmbedding, eng.BIASED), (LinearEmbedding, eng.LINEAR)):
            if isinstance(graph, cls):
                return kind
        raise TypeError("embedding graphs must be LinearEmbedding, BiasedLinearEmbedding or ReLUEmbedding instances")

    def _make_tower(self, side, graph, weight_graph, X):
        r = self.n_components
        kind = self._embed_kind(graph)
        n_features = X.shape[1]
        # ref:115-123 -- weights are re-initialised by every fit call
        rows = n_features if kind != eng.RELU else getattr(self, f"{side}_aux_dim")
        W0 = weight_graph.initialize_weights(rows, r)
        if tuple(W0.shape) != (rows, r):
            raise ValueError(f"{type(weight_graph).__name__}.initialize_weights returned {tuple(W0.shape)}, expected {(rows, r)}")
        W = eng.storage_of(W0)
        b = Wr = br = None
        if kind == eng.BIASED:  # ref:136-137,142-143: the bias persists on the model across fits
            cur = getattr(self, f"{side}_linear_bias")
            b = eng.storage_of(cur) if cur is not None else eng.new_storage(1, r)
            setattr(self, f"{side}_linear_bias", _public(b, r))
        if kind == eng.RELU:  # ref:139-140,145-146
            aux = rows
            rw, rb = getattr(self, f"{side}_relu_weight"), getattr(self, f"{side}_relu_bias")
            if rw is None or rb is None:
                nrw, nrb = new_relu_params(n_features, aux)
                rw = nrw if rw is None else rw
                rb = nrb if rb is None else rb
            Wr, br = eng.storage_of(rw), eng.storage_of(rb)
            setattr(self, f"{side}_relu_weight", _public(Wr, aux))
            setattr(self, f"{side}_relu_bias", _public(br, aux))
        tower = eng.Tower(kind, X, r, W, b=b, Wr=Wr, br=br)
        if kind == eng.RELU:
            tower.aux = rows
        return tower

    def _trainable_list(self, tower):
        r = self.n_components
        if tower.kind == eng.LINEAR:
            return [_public(tower.W, r)]
        if tower.kind == eng.BIASED:
            return [_public(tower.W, r), _public(tower.b, r)]
        return [_public(tower.W, r), _public(tower.Wr, tower.aux), _public(tower.br, tower.aux)]

    def _prepare(self, user_features, item_features, tf_interactions, comm=None, batch_size=None):
        """Everything ``fit`` does before its epoch loop (ref:110-123) plus the one-time device
        structures (CSR / item-major lists).  Returns the ``TrainPlan``."""
        Xu, Xi = as_features(user_features), as_features(item_features)
        inter = as_interactions(tf_interactions)
        n_users, n_items = Xu.shape[0], Xi.shape[0]  # ref:110-111
        if inter.dense_shape != (n_users, n_items):
            raise ValueError(f"interactions have dense_shape {inter.dense_shape}, features imply {(n_users, n_items)}")
        loss = self._loss_kind()
        tu = self._make_tower("user", self.user_repr_graph, self.user_weight_graph, Xu)
        ti = self._make_tower("item", self.item_repr_graph, self.item_weight_graph, Xi)
        if batch_size is None:
            ip = eng.InteractionPlan(inter, loss, self.random_ind if loss == eng.WMRB else None)
        else:
            ip = eng.BatchedInteractions(inter, loss, self.random_ind if loss == eng.WMRB else None, batch_size)
        if loss == eng.WMRB:
            # the reference passes the constructor's n_items / n_samples to the loss (ref:165-167)
            if self.n_items is not None and self.n_items != n_items:
                raise ValueError("model n_items disagrees with item_features")
            if self.n_samples is not None and self.n_samples != ip.S:
                raise ValueError("model n_samples disagrees with random_ind")
        self._plan = eng.TrainPlan(tu, ti, ip, self.n_components, comm=comm)
        self.user_trainable = self._trainable_list(tu)
        self.item_trainable = self._trainable_list(ti)
        return self._plan

    def fit(self, epochs, user_features, item_features, tf_interactions, lr=1e-2, comm=None, verbose=True,
            optimizer="fresh", resample_every=None, resample_seed=None, batch_size=None):
        """Full-batch training, one gradient step per epoch (ref:96-187).

        Each epoch: embeddings -> scores of the observed (and sampled) pairs -> loss -> gradient of the
        SUMMED loss (ref:170-171) -> a brand-new Adam's first step on every trainable (ref:176).
        Extensions (defaults = reference behaviour; SURVEY 8f):
          ``comm``            a ``teamoflow_b200.mf.dist.GradientSync`` for user-sharded data parallelism;
          ``optimizer``       ``"fresh"`` = a new Adam every epoch like the reference; ``"adam"`` = ONE Adam whose moments
                              and step count persist over the epochs of this fit (``tmf_adam``);
          ``resample_every``  redraw the WMRB negatives every that many epochs with the device sampler (the reference
                              samples once per model, ref:72-73); ``resample_seed`` makes the draws reproducible.  The new
                              table replaces ``self.random_ind``; every table drawn is also kept in ``self._sample_log``.
          ``batch_size``      mini-batch mode: USERS per mini-batch (contiguous blocks; MSE / WMRB).  An epoch is then one
                              optimizer step per block, each on the summed loss of that block's interactions; ``None`` = the
                              reference's full batch (ref:128).
        """
        if optimizer not in ("fresh", "adam"):
            raise ValueError("optimizer must be 'fresh' (reference behaviour) or 'adam'")
        plan = self._prepare(user_features, item_features, tf_interactions, comm=comm, batch_size=batch_size)
        if optimizer == "adam":
            plan.opt_state = ({}, {})
        if comm is not None:
            comm.broadcast_params(plan.u, plan.i)
        cumulative_time = 0
        self.loss_history = []
        self._sample_log = []
        span_left = 0
        for epoch in range(epochs):
            start = t.default_timer()
            if resample_every and epoch > 0 and epoch % int(resample_every) == 0 and plan.ip.loss == eng.WMRB:
                seed = None if resample_seed is None else int(resample_seed) + epoch
                if seed is None:
                    seed = int(np.random.randint(0, 2 ** 62))
                self.random_ind = random_sampler(plan.ip.n_items, plan.ip.n_users, plan.ip.S, seed=seed)
                self._sample_log.append((epoch, self.random_ind))
                plan.ip.set_samples(self.random_ind)
                plan.invalidate_graph()
            if span_left == 0:
                # epochs up to the next loss report / resampling point run as one span (TrainPlan.run: first step
                # eager, the rest replayed from a CUDA graph of the step)
                span_left = min(25 - epoch % 25, epochs - epoch)
                if resample_every and plan.ip.loss == eng.WMRB:
                    span_left = min(span_left, int(resample_every) - epoch % int(resample_every))
                plan.run(span_left, lr)
            span_left -= 1
            report = (epoch + 1) % 25 == 0
            if report:
                torch.cuda.synchronize()
            end = t.default_timer()
            cumulative_time += (end - start)
            if report:  # ref:179-183
                loss_one_epoch = plan.ip.mean_loss() if comm is None else comm.mean_loss(plan.ip)
                self.loss_history.append((epoch + 1, loss_one_epoch))
                if verbose:
                    print(f'Epoch {epoch + 1} Complete | Loss {loss_one_epoch} | Runtime {cumulative_time:.5} s')
        plan.invalidate_graph()  # the captured step does not outlive fit (with comm it holds NCCL work)
        if comm is not None and hasattr(comm, "detach"):
            comm.detach(plan)
        # ref:186-187 -- embeddings recomputed from the final weights
        r = self.n_components
        self.user_embedding = _public(plan.u.forward(), r)
        self.item_embedding = _public(plan.i.forward(), r)
        self.user_trainable = self._trainable_list(plan.u)
        self.item_trainable = self._trainable_list(plan.i)

    # ------------------------------------------------------------------ prediction / ranking

    def predict(self, A=None):
        """Dense ``U V^T`` (ref:189-201); with ``A`` also the scores of the unobserved cells (``A == 0``) flattened
        row-major (ref:197-198).  A sparse ``A`` (``SparseInteractions`` / scipy / torch sparse, distinct cells) is never
        densified: the unobserved scores are gathered against its CSR (``tmf_gather_unobserved``)."""
        all_predictions = dense_scores(self.user_embedding, self.item_embedding)
        if A is not None:
            if _is_sparse_table(A):
                n_u, n_i = all_predictions.shape
                a_ptr, a_idx, _ = _csr_of(A, n_u, n_i, drop_zeros=True)
                out = torch.empty(n_u * n_i - int(a_idx.numel()), dtype=torch.float32, device=all_predictions.device)
                _abi.call("tmf_gather_unobserved", _abi.ptr(all_predictions), n_u, n_i, _abi.ptr(a_ptr), _abi.ptr(a_idx), _abi.ptr(out))
                return all_predictions, out
            A = to_device(A, torch.float32)
            return all_predictions, all_predictions[A == 0]
        return all_predictions

    def predict_ranks(self, A):
        """Descending order of the unobserved scores (ref:203-216)."""
        _, tf_predictions = self.predict(A)
        return _rank_rows(tf_predictions.reshape(1, -1), clamp=False).reshape(-1)

    def _topk(self, k, clamp, users=None):
        """Top-k item ids per user, ties -> lower item id (``tf.math.top_k``, ref:245,:429)."""
        U = eng.storage_of(self.user_embedding)
        V = eng.storage_of(self.item_embedding)
        if users is not None:
            U = U[users].contiguous()
        n_u, n_i = U.shape[0], V.shape[0]
        k = min(int(k), n_i)
        if k <= TOPK_FUSED_MAX_K:
            idx, _ = score_topk(U, V, self.n_components, k, clamp)
            return idx
        P = torch.empty(n_u, n_i, dtype=torch.float32, device=U.device)
        _abi.call("tmf_predict_dense", _abi.ptr(U), n_u, _abi.ptr(V), n_i, self.n_components, U.shape[1], _abi.ptr(P))
        return _rank_rows(P, clamp)[:, :k].contiguous()

    def _hits_relevant(self, A, k):
        from . import evaluation as ev
        a_csr = _csr_of(A, self.user_embedding.shape[0], self.item_embedding.shape[0])
        return ev.hits_relevant(self._topk(k, clamp=True), a_csr)  # ref:237,245

    def recall_at_k(self, A, k=10, preserve_rows=False):
        """ref:218-269 (hits count any non-zero interaction; relevant counts positive ones).  Held-out evaluation with
        the training items excluded: ``evaluation.recall_at_k``."""
        from . import evaluation as ev
        hits, relevant = self._hits_relevant(A, k)
        return ev.recall_from_hits(hits, relevant, preserve_rows)

    def precision_at_k(self, A, k=10, preserve_rows=False):
        """ref:271-304."""
        from . import evaluation as ev
        hits, relevant = self._hits_relevant(A, k)
        return ev.precision_from_hits(hits, relevant, k, preserve_rows)

    def f1_at_k(self, A, k=10, beta=1.0):
        """ref:306-318 (formula kept as written)."""
        precision, recall = self.precision_at_k(A, k=k), self.recall_at_k(A, k=k)
        prec, rec = precision.mean(), recall.mean()
        return ((1 + beta ** 2) * prec * rec) / (beta ** 2 * (prec + rec))

    def dcg_at_k(self, dense_interactions, k=10):
        """ref:320-351 -- DCG of the top-k RAW scores with gains ``2^A - 1``."""
        from . import evaluation as ev
        a_csr = _csr_of(dense_interactions, self.user_embedding.shape[0], self.item_embedding.shape[0])
        return ev.dcg_of(self._topk(k, clamp=False), a_csr)

    def idcg_at_k(self, dense_interactions, k=10):
        """ref:353-384 -- gains sorted descending, first k."""
        return self._idcg(dense_interactions, k)[0]

    def _idcg(self, A, k):
        n_u, n_i = self.user_embedding.shape[0], self.item_embedding.shape[0]
        a_ptr, a_idx, a_val = _csr_of(A, n_u, n_i)
        idcg = torch.empty(n_u, dtype=torch.float32, device=a_val.device)
        row_nnz = torch.empty(n_u, dtype=torch.float32, device=a_val.device)
        _abi.call("tmf_idcg", n_u, n_i, min(int(k), n_i), _abi.ptr(a_ptr), _abi.ptr(a_val), _abi.ptr(idcg), _abi.ptr(row_nnz))
        return idcg, row_nnz

    def ndcg_at_k(self, A, k=10, preserve_rows=False):
        """ref:386-413."""
        from . import evaluation as ev
        dcg = self.dcg_at_k(A, k)
        idcg, row_nnz = self._idcg(A, k)
        return ev.ndcg_from_dcg(dcg, idcg, row_nnz, preserve_rows)

    def retrieve_user_recs(self, user=None, k=None, exclude=None):
        """Item rankings on RAW scores as a numpy int32 array (ref:416-438).

        Extension (SURVEY 8f-3; default = reference behaviour, which does NOT exclude seen items): ``exclude`` = an
        interaction table (sparse or dense) whose non-zero cells are removed from every user's ranking -- "recommend k
        unseen items" -- see ``recommend``."""
        if exclude is not None:
            if k is None:
                raise ValueError("retrieve_user_recs(exclude=...) needs k")
            out = self.recommend(exclude, k=k, users=None if user is None else [int(user)]).cpu().numpy().astype(np.int32)
            return out if user is None else out[0]
        num_items = self.item_embedding.shape[0]
        users = None if user is None else torch.as_tensor([int(user)], device=self.user_embedding.device)
        idx = self._topk(num_items if k is None else k, clamp=False, users=users)
        out = idx.cpu().numpy().astype(np.int32)
        return out if user is None else out[0]

    def recommend(self, seen, k=10, users=None):
        """Masked top-k (extension, SURVEY 8f-3): the ``k`` best items per user by RAW canonical score, ties -> lower item id,
        EXCLUDING the non-zero cells of the interaction table ``seen`` (sparse or dense, never densified).  int32 ``[n, k]``
        on the device; a user with fewer than ``k`` unseen items has its row padded with -1.

        For ``k <= 1024`` the fused tcgen05 top-k drops the seen items itself (``tmf_score_topk_masked``), so the answer costs
        one ranking pass however many of a user's best items are seen; larger ``k`` ranks dense blocks of canonical scores
        (``evaluation.masked_topk``)."""
        from . import evaluation as ev
        n_u, n_i = self.user_embedding.shape[0], self.item_embedding.shape[0]
        a_ptr, a_idx = ev.exclusion_csr(seen, n_u, n_i)
        dev = self.user_embedding.device
        k = int(k)
        if k < 1:
            raise ValueError("k must be >= 1")
        U = eng.storage_of(self.user_embedding)
        if users is not None:
            rows = torch.as_tensor(users, device=dev, dtype=torch.int64).reshape(-1)
            cnt = (a_ptr[1:] - a_ptr[:-1])[rows]
            sub_ptr = torch.zeros(rows.numel() + 1, dtype=torch.int32, device=dev)
            sub_ptr[1:] = torch.cumsum(cnt, 0).to(torch.int32)
            take = torch.repeat_interleave(a_ptr[:-1][rows].to(torch.int64) - sub_ptr[:-1].to(torch.int64), cnt.to(torch.int64)) \
                + torch.arange(int(sub_ptr[-1]), device=dev)
            a_ptr, a_idx = sub_ptr, a_idx[take].contiguous()
            U = U[rows].contiguous()
        n = U.shape[0]
        out = torch.full((n, k), -1, dtype=torch.int32, device=dev)
        if n == 0:
            return out
        got = ev.masked_topk(U, eng.storage_of(self.item_embedding), self.n_components, k, False, a_ptr, a_idx)
        out[:, :got.shape[1]] = torch.where(got == ev.PAD_ID, torch.full_like(got, -1), got)
        return out

    # ------------------------------------------------------------------ save / load (in-memory, ref:440-475)

    def save_model(self):
        dict_config = {'Latent Dimension': self.n_components, 'User Embedding': self.user_repr_graph,
                       'Item Embedding': self.item_repr_graph, 'Loss': self.loss_graph,
                       'User Initialization': self.user_weight_graph, 'Item Initialization': self.item_weight_graph,
                       'Number of Users': self.n_users, 'Number of Items': self.n_items,
                       'Number of Samples': self.n_samples, 'Generate Sample': self.generate_sample}
        dict_results = {'User Embedding': self.user_embedding, 'Item Embedding': self.item_embedding,
                        'User Variables': self.user_trainable, 'Item Variables': self.item_trainable}
        return dict_config, dict_results

    def save(self, path):
        """Extension (SURVEY 8f): write the fitted model to ``path`` -- constructor kwargs (so ``load`` can rebuild it,
        unlike ``from_saved(save_model()[0])``, quirk 7), embeddings, trainables and the sampled negatives."""
        config = {"n_components": self.n_components, "user_repr_graph": type(self.user_repr_graph).__name__,
                  "item_repr_graph": type(self.item_repr_graph).__name__, "loss_graph": type(self.loss_graph).__name__,
                  "user_weight_graph": type(self.user_weight_graph).__name__, "item_weight_graph": type(self.item_weight_graph).__name__,
                  "n_users": self.n_users, "n_items": self.n_items, "n_samples": self.n_samples,
                  "generate_sample": bool(self.generate_sample)}
        c = lambda x: None if x is None else x.detach().cpu()  # noqa: E731
        state = {"user_embedding": c(getattr(self, "user_embedding", None)), "item_embedding": c(getattr(self, "item_embedding", None)),
                 "user_trainable": None if self.user_trainable is None else [c(v) for v in self.user_trainable],
                 "item_trainable": None if self.item_trainable is None else [c(v) for v in self.item_trainable],
                 "random_ind": c(self.random_ind),
                 "user_linear_bias": c(self.user_linear_bias), "item_linear_bias": c(self.item_linear_bias),
                 "user_relu_weight": c(self.user_relu_weight), "user_relu_bias": c(self.user_relu_bias),
                 "item_relu_weight": c(self.item_relu_weight), "item_relu_bias": c(self.item_relu_bias)}
        torch.save({"format": "teamoflow_b200.mf/1", "config": config, "state": state}, path)

    @classmethod
    def load(cls, path, initializers=None, graphs=None):
        """Rebuild a model written by ``save``.  Class names in the file are resolved through a fixed table of the
        package's own graph classes (nothing else can be instantiated from a file).  User-defined subclasses are not
        serialised: pass ``initializers=(user_weight_graph, item_weight_graph)`` and / or
        ``graphs={"user_repr_graph": obj, "item_repr_graph": obj, "loss_graph": obj}`` (instances) to restore them."""
        from . import embedding_graphs as _E, initializer_graphs as _I, loss_graphs as _L
        known = {"LinearEmbedding": _E.LinearEmbedding, "BiasedLinearEmbedding": _E.BiasedLinearEmbedding,
                 "ReLUEmbedding": _E.ReLUEmbedding, "MSELoss": _L.MSELoss, "WMRBLoss": _L.WMRBLoss,
                 "KLDivergenceLoss": _L.KLDivergenceLoss}
        known_init = {"NormalInitializer": _I.NormalInitializer, "UniformInitializer": _I.UniformInitializer}
        blob = torch.load(path, map_location="cpu", weights_only=True)
        if blob.get("format") != "teamoflow_b200.mf/1":
            raise ValueError("not a teamoflow_b200 model file")
        cfg, st = dict(blob["config"]), blob["state"]
        graphs = dict(graphs or {})
        for key in ("user_repr_graph", "item_repr_graph", "loss_graph"):
            if graphs.get(key) is not None:
                cfg[key] = graphs[key]
            elif cfg[key] in known:
                cfg[key] = known[cfg[key]]()
            else:
                raise ValueError(f"{key} = {cfg[key]!r} is not one of the package's graph classes {sorted(known)}; "
                                 f"pass an instance through load(..., graphs={{'{key}': obj}})")
        for j, key in enumerate(("user_weight_graph", "item_weight_graph")):
            given = None if initializers is None else initializers[j]
            cfg[key] = given if given is not None else known_init.get(cfg[key], _I.NormalInitializer)()
        # the sampled negatives are restored from the file below; do not draw a new table in the constructor
        generate_sample = bool(cfg.pop("generate_sample", False))
        model = cls(**cfg)
        model.generate_sample = generate_sample
        r = model.n_components
        g = lambda x: None if x is None else to_device(x, x.dtype)  # noqa: E731
        if st["user_embedding"] is not None:
            model.user_embedding = _public(eng.storage_of(g(st["user_embedding"])), r)
            model.item_embedding = _public(eng.storage_of(g(st["item_embedding"])), r)
        model.user_trainable = None if st["user_trainable"] is None else [g(v) for v in st["user_trainable"]]
        model.item_trainable = None if st["item_trainable"] is None else [g(v) for v in st["item_trainable"]]
        model.random_ind = g(st["random_ind"])
        for key in ("user_linear_bias", "item_linear_bias", "user_relu_weight", "user_relu_bias", "item_relu_weight", "item_relu_bias"):
            setattr(model, key, g(st[key]))
        return model

    @classmethod
    def from_saved(cls, config):
        """``cls(**config)`` like ref:466-475 (so, like the reference, it takes constructor kwargs --
        ``save_model()``'s own human-readable keys raise TypeError there too)."""
        return cls(**config)


# ---------------------------------------------------------------------- module helpers


def score_topk(U, V, r, k, clamp, item_offset=0, row_bound=None, out=None):
    """Fused tcgen05 ``U V^T`` + per-row top-k (``tmf_score_topk``).  ``U``/``V`` are padded storages.
    Returns ``(idx int32 [n_u, k], score fp32 [n_u, k])``.

    ``row_bound`` (fp32 ``[n_u]``, item-sharded scoring only): per-user lower bounds of the k-th best score over ALL
    slabs (``tmf_score_topk_bounded``); rows may then end in ``(-inf, INT32_MAX)`` padding.  ``out``: optional
    ``(idx, score)`` buffers to fill (e.g. views of a peer arena)."""
    n_u, n_i = U.shape[0], V.shape[0]
    if out is None:
        idx = torch.empty(n_u, k, dtype=torch.int32, device=U.device)
        score = torch.empty(n_u, k, dtype=torch.float32, device=U.device)
    else:
        idx, score = out
        assert idx.shape == (n_u, k) and score.shape == (n_u, k) and idx.is_contiguous() and score.is_contiguous()
    ws_bytes = _abi.query("tmf_score_topk_ws_bytes", n_u, n_i, r, k)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=U.device)
    if row_bound is None:
        _abi.call("tmf_score_topk", _abi.ptr(U), n_u, _abi.ptr(V), n_i, r, U.shape[1], k, int(bool(clamp)), int(item_offset),
                  _abi.ptr(idx), _abi.ptr(score), _abi.ptr(ws), ws_bytes)
    else:
        assert row_bound.dtype == torch.float32 and row_bound.numel() == n_u and row_bound.is_contiguous()
        _abi.call("tmf_score_topk_bounded", _abi.ptr(U), n_u, _abi.ptr(V), n_i, r, U.shape[1], k, int(bool(clamp)),
                  int(item_offset), _abi.ptr(row_bound), _abi.ptr(idx), _abi.ptr(score), _abi.ptr(ws), ws_bytes)
    return idx, score


def _rank_rows(P, clamp):
    n_rows, n_cols = P.shape
    out = torch.empty(n_rows, n_cols, dtype=torch.int32, device=P.device)
    ws_bytes = _abi.query("tmf_rank_rows_ws_bytes", n_rows, n_cols)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=P.device)
    _abi.call("tmf_rank_rows", _abi.ptr(P.contiguous()), n_rows, n_cols, int(bool(clamp)), _abi.ptr(out), _abi.ptr(ws), ws_bytes)
    return out


def _is_sparse_table(A):
    if isinstance(A, SparseInteractions):
        return True
    if isinstance(A, torch.Tensor):
        return A.layout != torch.strided
    try:
        from scipy import sparse as _sp
        return _sp.issparse(A)
    except Exception:  # pragma: no cover
        return False


def _csr_of(A, n_users, n_items, drop_zeros=False):
    """Interaction table (dense like the reference, or sparse) -> CSR on the device.  ``drop_zeros``: explicitly stored
    zeros are removed (they count as unobserved for ``A == 0``)."""
    inter = as_interactions(A)
    if inter.dense_shape != (n_users, n_items):
        raise ValueError(f"interaction table has shape {inter.dense_shape}, model has {(n_users, n_items)}")
    if drop_zeros and inter.nnz and bool((inter.values == 0).any()):
        keep = inter.values != 0
        inter = SparseInteractions(inter.indices[keep], inter.values[keep], inter.dense_shape)
    row_ptr, col_idx, vals, _, _ = inter.csr()
    return row_ptr, col_idx, vals
