"""``teamoflow_b200.mf``: the B200-native mirror of the reference package ``teamoflow.mf``.

The drop-in boundary is the module layout itself (SURVEY 8b): a user of the reference imports
``<pkg>.mf.matrix_factorization``, ``.loss_graphs`` and so on, so the same submodule names are imported here and
re-exported through ``__all__``, followed by this build's ``evaluation`` (held-out metrics; the reference has no
counterpart).  (``_engine``, ``_tensors`` and ``dist`` are this build's own internals and are not part of that surface.)
"""
import importlib as _importlib

__all__ = [
    "matrix_factorization",   # MatrixFactorization: fit / predict / top-k / metrics
    "loss_graphs",            # MSELoss, WMRBLoss, KLDivergenceLoss
    "predict_graphs",         # DotProductPrediction
    "embedding_graphs",       # LinearEmbedding, BiasedLinearEmbedding, ReLUEmbedding
    "initializer_graphs",     # NormalInitializer, UniformInitializer
    "input_utils",            # sparse-input adapters
    "utils",                  # random_sampler, generate_random_interaction, gather_matrix_indices
    "evaluation",             # held-out recall / precision / NDCG with training items excluded; masked top-k
]

for _name in __all__:
    globals()[_name] = _importlib.import_module(f"{__name__}.{_name}")
del _name
