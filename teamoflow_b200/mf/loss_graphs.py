"""Loss graphs -- same classes/signatures as the reference ``mf/loss_graphs.py``.

``get_loss`` keeps the reference's argument names and returns the same tensors (forward only --
there is no autodiff here).  During ``MatrixFactorization.fit`` the classes are descriptors: the
loss, its gradient and the embedding gradients come out of the fused kernels (``tmf_user_pass``;
``tmf_kl_moments`` then ``tmf_kl_coef_from_moments`` for KL) and the dense ``predictions`` matrix these
signatures expect is never formed.
"""
from abc import ABC, abstractmethod

import torch

from .. import _abi
from ._engine import KL, MSE, WMRB, reduce_ws
from ._tensors import as_interactions, to_device


class LossGraph(ABC):
    """Abstract base class of loss functions (reference ``loss_graphs.py:8-28``)."""
    kind = None

    @abstractmethod
    def get_loss(self, tf_interactions, tf_sample_predictions, tf_prediction_serial, predictions, n_items, n_samples):
        pass


def _gather_nd(predictions, indices):
    P = to_device(predictions, torch.float32)
    out = torch.empty(indices.shape[0], dtype=torch.float32, device=P.device)
    _abi.call("tmf_gather_nd2", _abi.ptr(P), P.shape[1], _abi.ptr(indices), indices.shape[0], _abi.ptr(out))
    return out


class MSELoss(LossGraph):
    """``square(values - predictions[indices])`` over the stored interactions (reference ``:36-52``)."""
    kind = MSE

    def get_loss(self, tf_interactions, predictions, tf_sample_predictions=None, tf_prediction_serial=None, n_items=None, n_samples=None):
        inter = as_interactions(tf_interactions)
        return torch.square(inter.values - _gather_nd(predictions, inter.indices))


class WMRBLoss(LossGraph):
    """Sampled weighted-margin-rank-batch loss on the positive interactions (reference ``:62-88``)."""
    kind = WMRB

    def get_loss(self, tf_interactions, tf_sample_predictions, tf_prediction_serial, n_items, n_samples, predictions=None):
        inter = as_interactions(tf_interactions)
        sp = to_device(tf_sample_predictions, torch.float32)
        serial = to_device(tf_prediction_serial, torch.float32).reshape(-1)
        mask = inter.values > 0                                   # :74
        pos_rows = inter.indices[:, 0][mask].to(torch.int32).contiguous()
        pos_pred = serial[mask].contiguous()
        out = torch.empty(pos_rows.numel(), dtype=torch.float32, device=sp.device)
        _abi.call("tmf_wmrb_forward", pos_rows.numel(), _abi.ptr(pos_rows), _abi.ptr(pos_pred), _abi.ptr(sp),
                  sp.shape[1], float(n_items / n_samples), _abi.ptr(out))
        return out


class KLDivergenceLoss(LossGraph):
    """``1 - Normal(mu_neg - mu_pos, sqrt(var_pos + var_neg)).cdf(0)`` (reference ``:100-122``), a scalar."""
    kind = KL

    def get_loss(self, tf_prediction_serial, tf_interactions, tf_sample_predictions=None, predictions=None, n_items=None, n_samples=None):
        inter = as_interactions(tf_interactions)
        serial = to_device(tf_prediction_serial, torch.float32).reshape(-1)
        loss = torch.empty(1, dtype=torch.float32, device=serial.device)
        coef = torch.empty(max(serial.numel(), 1), dtype=torch.float32, device=serial.device)
        moments = torch.empty(6, dtype=torch.float64, device=serial.device)
        ws = reduce_ws()
        _abi.call("tmf_kl_moments", serial.numel(), _abi.ptr(serial), _abi.ptr(inter.values), _abi.ptr(moments), _abi.ptr(ws))
        _abi.call("tmf_kl_coef_from_moments", serial.numel(), _abi.ptr(serial), _abi.ptr(inter.values), _abi.ptr(moments),
                  _abi.ptr(loss), _abi.ptr(coef), _abi.ptr(ws))
        return loss.reshape(())
