"""Host-side orchestration of the CUDA training step (one process per GPU).

``TrainPlan`` owns every device buffer of a ``MatrixFactorization.fit`` call and issues, per epoch,
the kernel sequence that replaces ``matrix_factorization.py:130-176``:

    embed fwd (spmm / alias)  ->  fused user pass (scores, loss, dL/dscore, dE_u)
    ->  item-major segment-sum (dE_i)  ->  [sum of dE_i over the ranks when user-sharded: one NVLink peer-memory
        kernel, Adam fused in when the item tower is an identity-feature Linear one; NCCL as the fallback]
    ->  embed bwd  ->  Adam step-1 on every trainable

Embedding matrices live in padded storage ``[n, ld]`` (``ld = ceil4(r)``, pad columns zero) so rows
are 16-byte aligned for 128-bit loads; the public tensors are the ``[:, :r]`` views.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from .. import _abi
from ._tensors import FeatureMatrix, SparseInteractions, build_transpose, device, pad4, to_device

LINEAR, BIASED, RELU = "linear", "biased", "relu"
MSE, WMRB, KL = "mse", "wmrb", "kl"
_LOSS_CODE = {MSE: 0, WMRB: 1}


# ----------------------------------------------------------------------------- storage helpers


def new_storage(n, r, fill=None):
    st = torch.zeros(int(n), pad4(r), dtype=torch.float32, device=device())
    if fill is not None:
        st[:, :r] = fill
    return st


def storage_of(W):
    """Padded ``[n, ld]`` storage behind a public ``[n, r]`` weight (copying when ``W`` is not one of ours)."""
    if isinstance(W, torch.Tensor) and W.is_cuda and W.dtype == torch.float32 and W.dim() == 2:
        base = W._base if W._base is not None else W
        n, r = W.shape
        if (base.dim() == 2 and base.is_contiguous() and base.shape == (n, pad4(r)) and base.data_ptr() == W.data_ptr()
                and W.stride() == (pad4(r), 1) and base.data_ptr() % 16 == 0):
            return base
    Wt = to_device(W.detach() if isinstance(W, torch.Tensor) else W, torch.float32)
    if Wt.dim() != 2:
        raise ValueError("weights must be 2-D")
    return new_storage(Wt.shape[0], Wt.shape[1], Wt)


def _ws(nbytes):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device())


def reduce_ws():
    return _ws(_abi.query("tmf_reduce_ws_bytes"))


def spmm(n_seg, seg_ptr, n_entries, idx, cpos, coef, src, n_cols, out=None, ws=None):
    """``out[s] = sum_e c(e) * src[idx[e]]`` -- see ``tmf_spmm_seg``."""
    ld_out = pad4(n_cols)
    if out is None:
        out = torch.empty(n_seg, ld_out, dtype=torch.float32, device=src.device)
        if ld_out != n_cols:
            out.zero_()
    need = _abi.query("tmf_spmm_ws_bytes", n_entries, out.shape[1])
    if ws is None or ws.numel() < need:
        ws = _ws(need)
    _abi.call("tmf_spmm_seg", n_seg, _abi.ptr(seg_ptr), n_entries, _abi.ptr(idx), _abi.ptr(cpos), _abi.ptr(coef),
              _abi.ptr(src), src.shape[1], _abi.ptr(out), out.shape[1], n_cols, _abi.ptr(ws), ws.numel())
    return out


# dense contractions with at least this many multiply-adds go to the tensor cores (tmf_gemm_tc: tcgen05, operands split
# exactly into three bf16 planes, fp32 accumulation in TMEM); smaller ones stay on the SIMT fp32 kernel (launch-bound anyway)
TC_GEMM_MIN_MACS = 1 << 22


def gemm(ta, tb, m, n, k, A, B, out=None, tc=None):
    """``out[m, n] = op(A) op(B)`` (``ta``: A is stored [k, m]; ``tb``: B is stored [n, k]); storages with padded leading dims."""
    if out is None:
        out = torch.zeros(m, pad4(n), dtype=torch.float32, device=A.device)
    use_tc = (m * n * k >= TC_GEMM_MIN_MACS) if tc is None else bool(tc)
    if use_tc:
        need = _abi.query("tmf_gemm_tc_ws_bytes", m, n, k)
        ws = _ws(need)
        _abi.call("tmf_gemm_tc", int(ta), int(tb), m, n, k, _abi.ptr(A), A.shape[1], _abi.ptr(B), B.shape[1],
                  _abi.ptr(out), out.shape[1], _abi.ptr(ws), ws.numel())
    else:
        _abi.call("tmf_gemm_f32", int(ta), int(tb), m, n, k, _abi.ptr(A), A.shape[1], _abi.ptr(B), B.shape[1],
                  _abi.ptr(out), out.shape[1])
    return out


def col_sum(dE, n_cols):
    out = torch.zeros(1, pad4(n_cols), dtype=torch.float32, device=dE.device)
    ws = _ws(1024 * dE.shape[1] * 4)
    _abi.call("tmf_col_sum", _abi.ptr(dE), dE.shape[0], n_cols, dE.shape[1], _abi.ptr(out), _abi.ptr(ws), ws.numel())
    return out


def adam1(w, g, lr):
    _abi.call("tmf_adam1", _abi.ptr(w), _abi.ptr(g), w.numel(), float(lr))


# ----------------------------------------------------------------------------- one embedding tower


class Tower:
    """One side (user or item) of the model: features, trainables, embedding and its backward.

    kind/params follow ``embedding_graphs.py``: Linear ``X W`` (:38); BiasedLinear ``X W + b`` (:58);
    ReLU ``relu(X W_r + b_r) W`` with hidden width ``5 r`` (:73-87).
    """

    def __init__(self, kind, X: FeatureMatrix, r, W, b=None, Wr=None, br=None):
        self.kind, self.X, self.r = kind, X, int(r)
        self.n = X.shape[0]
        self.W = W            # storage [F or 5r, ld]
        self.b = b            # storage [1, ld]
        self.Wr, self.br = Wr, br  # [F, ld5], [1, ld5]
        self.aux = 5 * self.r
        self.H = None
        alias = (kind == LINEAR and X.identity)
        self.E = W if alias else torch.zeros(self.n, pad4(r), dtype=torch.float32, device=W.device)
        self.dE = torch.zeros(self.n, pad4(r), dtype=torch.float32, device=W.device)
        self.grads = {}
        self._ws = None

    # -- helpers
    def _x_times(self, M, n_cols, out=None):
        X = self.X
        if X.dense is not None:  # genuinely dense features: X M on the tensor cores (embedding_graphs.py:38)
            return gemm(0, 0, self.n, n_cols, X.shape[1], X.dense, M, out=out)
        if X.identity:
            if out is None:
                return M
            out.copy_(M)
            return out
        return spmm(self.n, X.ptr, X.nnz, X.idx, None, X.val, M, n_cols, out=out)

    def _xt_times(self, D, n_cols):
        X = self.X
        if X.dense is not None:  # X^T D: the stored [n, F] matrix read transposed
            return gemm(1, 0, X.shape[1], n_cols, self.n, X.dense, D)
        if X.identity:
            return D
        ptr_t, rows_t, perm_t = X.transpose()
        return spmm(X.shape[1], ptr_t, X.nnz, rows_t, perm_t, X.val, D, n_cols)

    def forward(self):
        r = self.r
        if self.kind == LINEAR:
            if not self.X.identity:
                self._x_times(self.W, r, out=self.E)
        elif self.kind == BIASED:
            self._x_times(self.W, r, out=self.E)
            _abi.call("tmf_bias_add", _abi.ptr(self.E), self.n, r, self.E.shape[1], _abi.ptr(self.b), 0)
        else:
            if self.H is None:
                self.H = torch.zeros(self.n, pad4(self.aux), dtype=torch.float32, device=self.W.device)
            self._x_times(self.Wr, self.aux, out=self.H)
            _abi.call("tmf_bias_add", _abi.ptr(self.H), self.n, self.aux, self.H.shape[1], _abi.ptr(self.br), 1)
            gemm(0, 0, self.n, r, self.aux, self.H, self.W, out=self.E)
        return self.E

    def backward(self):
        """Gradients of every trainable from ``self.dE`` (SURVEY App. A.5)."""
        r, dE = self.r, self.dE
        if self.kind == LINEAR:
            self.grads = {"W": self._xt_times(dE, r)}
        elif self.kind == BIASED:
            self.grads = {"W": self._xt_times(dE, r), "b": col_sum(dE, r)}
        else:
            dW = gemm(1, 0, self.aux, r, self.n, self.H, dE)          # H^T dE
            dH = gemm(0, 1, self.n, self.aux, r, dE, self.W)          # dE W^T
            _abi.call("tmf_relu_mask", _abi.ptr(dH), _abi.ptr(self.H), dH.numel())
            self.grads = {"W": dW, "Wr": self._xt_times(dH, self.aux), "br": col_sum(dH, self.aux)}
        return self.grads

    def trainables(self):
        """Storage tensors in the order ``get_repr`` returns them."""
        if self.kind == LINEAR:
            return {"W": self.W}
        if self.kind == BIASED:
            return {"W": self.W, "b": self.b}
        return {"W": self.W, "Wr": self.Wr, "br": self.br}

    def update(self, lr, skip=(), state=None):
        """Reference behaviour (``state is None``): a brand-new Adam's first step (matrix_factorization.py:176).
        ``state``: dict of persistent moments + step count (the ``optimizer="adam"`` extension)."""
        if state is not None:
            state["t"] = state.get("t", 0) + 1
        for k, w in self.trainables().items():
            if k in skip:
                continue
            if state is None:
                adam1(w, self.grads[k], lr)
            else:
                if k not in state:
                    state[k] = (torch.zeros_like(w), torch.zeros_like(w))
                m, v = state[k]
                _abi.call("tmf_adam", _abi.ptr(w), _abi.ptr(self.grads[k]), _abi.ptr(m), _abi.ptr(v), w.numel(), float(lr), state["t"])


# ----------------------------------------------------------------------------- interaction structure


class InteractionPlan:
    """Everything derived from the (fixed) interactions and (fixed) negatives, built once per fit:
    CSR by user, the item-major list of (user, coefficient slot) over interactions ++ samples,
    heavy-first user order, coefficient / loss buffers."""

    def __init__(self, inter: SparseInteractions, loss, random_ind=None):
        self.inter, self.loss = inter, loss
        self.n_users, self.n_items = inter.dense_shape
        self.row_ptr, self.col_idx, self.vals, self.coo_rows, self.perm = inter.csr()
        dev = self.vals.device
        self.nnz = inter.nnz
        self.S = 0
        self.samp = None
        self.t_user = None
        self.comm = None        # set by TrainPlan under user sharding (KL needs the global moments)
        self.set_samples(random_ind)
        self._build_work_list()
        self.counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self.coef = torch.zeros(max(self.nnz + self.n_users * self.S, 1), dtype=torch.float32, device=dev)
        self.loss_k = torch.zeros(max(self.nnz, 1), dtype=torch.float32, device=dev)
        self.p = torch.zeros(max(self.nnz, 1), dtype=torch.float32, device=dev) if loss == KL else None
        self.kl_moments = torch.zeros(6, dtype=torch.float64, device=dev) if loss == KL else None
        self.kl_loss = torch.zeros(1, dtype=torch.float32, device=dev)
        self.red_ws = reduce_ws()
        self.red_out = torch.zeros(1, dtype=torch.float32, device=dev)
        self.spmm_ws = None
        self.n_pos = int((self.vals > 0).sum()) if loss == WMRB else self.nnz

    def set_samples(self, random_ind):
        """(Re)build everything that depends on the sampled negatives: the int32 sample table and the item-major
        list over interactions ++ samples.  Called once per fit (the reference samples once per model,
        matrix_factorization.py:72-73) and again by the ``resample_every`` extension."""
        dev = self.vals.device
        keys = self.col_idx
        if self.loss == WMRB:
            if random_ind is None:
                raise ValueError("WMRBLoss needs sampled items: construct the model with n_users, n_items and "
                                 "generate_sample=True (or set model.random_ind)")
            ri = to_device(random_ind, torch.int64)
            if ri.dim() != 2 or ri.shape[0] != self.n_users:
                raise ValueError(f"random_ind must be [n_users={self.n_users}, n_samples], got {tuple(ri.shape)}")
            if ri.numel():
                lo_hi = torch.stack(torch.aminmax(ri)).tolist()  # one synchronisation
                if lo_hi[0] < 0 or lo_hi[1] >= self.n_items:
                    raise ValueError("random_ind holds item ids outside [0, n_items)")
            if self.S and int(ri.shape[1]) != self.S:
                raise ValueError("the number of samples per user cannot change between resamplings")
            self.S = int(ri.shape[1])
            if self.n_users * self.S + self.nnz >= 2 ** 31:
                raise ValueError("nnz + n_users*n_samples must be < 2^31")
            self.samp = ri.to(torch.int32).contiguous()
            keys = torch.cat([self.col_idx, self.samp.reshape(-1)])
        self.T = int(keys.numel())
        self.t_ptr, self.t_src = build_transpose(keys, self.n_items)
        # Coefficients in item-major order: when the gathered table E_u fits the L2 (the item pass is then bound by the latency of
        # its 4-byte coefficient gathers, one 32-byte DRAM sector each) the user pass stores c_k / G_uj straight into the slot the
        # item pass will read (coef_pos = inverse of the transpose permutation) and the item pass streams them.  On HBM-bound
        # problems (E_u far larger than L2) the scattered partial-sector writes cost more DRAM traffic than the gathers: keep the
        # natural order there.
        self.coef_pos = None
        if self.loss in (MSE, WMRB) and self.DIRECT_COEF and self.n_users * 4 * 64 <= self.DIRECT_COEF_MAX_TABLE_BYTES and self.T:
            self.coef_pos = torch.empty(self.T, dtype=torch.int32, device=dev)
            self.coef_pos[self.t_src.long()] = torch.arange(self.T, dtype=torch.int32, device=dev)
        if self.t_user is None or self.t_user.numel() < max(self.T, 1):
            self.t_user = torch.empty(max(self.T, 1), dtype=torch.int32, device=dev)
        _abi.call("tmf_tlist_users", _abi.ptr(self.t_src), self.T, self.nnz, _abi.ptr(self.coo_rows), max(self.S, 1),
                  _abi.ptr(self.t_user))

    # users with more interactions than the slice length are processed as several slices (load balance: tmf_user_pass gives
    # a work item to ONE warp).  1024 on large problems; shorter -- down to 32 -- when the whole problem would otherwise
    # not fill the machine's ~9.5k resident warp slots (a 943-user problem's heaviest user must not be one warp's tail).
    DIRECT_COEF = os.environ.get("TMF_DIRECT_COEF", "1") != "0"   # development switch (A/B of the two coefficient layouts)
    DIRECT_COEF_MAX_TABLE_BYTES = 64 << 20                        # n_users x 256 B (a rank-64 row) must fit comfortably in the 126 MB L2
    SPLIT = 1024
    SPLIT_MIN = 32
    TARGET_ITEMS = 148 * 32 * 2

    def slice_len(self):
        return int(min(self.SPLIT, max(self.SPLIT_MIN, self.nnz // self.TARGET_ITEMS)))

    def _build_work_list(self):
        """Work items of the user pass: whole users, or slice_len()-sized slices of very heavy users, heaviest first."""
        dev = self.vals.device
        SPLIT = self.slice_len()
        rp = self.row_ptr.to(torch.int64)
        lens = rp[1:] - rp[:-1]
        nseg = torch.clamp((lens + SPLIT - 1) // SPLIT, min=1)
        first_seg = torch.cumsum(nseg, 0) - nseg
        w_user = torch.repeat_interleave(torch.arange(self.n_users, device=dev), nseg)
        seg = torch.arange(w_user.numel(), device=dev) - first_seg[w_user]
        w_a = rp[w_user] + seg * SPLIT
        w_b = torch.minimum(w_a + SPLIT, rp[w_user + 1])
        split = nseg[w_user] > 1
        slot = torch.cumsum(split.to(torch.int64), 0) - 1
        w_slot = torch.where(split, slot, torch.full_like(slot, -1))
        order = torch.argsort(w_b - w_a, descending=True, stable=True)
        i32 = lambda t: t.to(torch.int32).contiguous()  # noqa: E731
        self.n_work = int(w_user.numel())
        self.w_user, self.w_a, self.w_b, self.w_slot = i32(w_user[order]), i32(w_a[order]), i32(w_b[order]), i32(w_slot[order])
        su = torch.nonzero(nseg > 1).reshape(-1)
        self.n_split = int(su.numel())
        self.n_slots = int(split.sum())
        self.split_user = i32(su)
        self.split_first = i32(slot[first_seg[su]]) if self.n_split else i32(su)
        self.split_nseg = i32(nseg[su])
        self.part_G = self.part_E = None

    def _partials(self, ld):
        if self.n_slots and (self.part_E is None or self.part_E.shape[1] != ld):
            dev = self.vals.device
            self.part_E = torch.zeros(self.n_slots, ld, dtype=torch.float32, device=dev)
            self.part_G = torch.zeros(self.n_slots, max((self.S + 3) // 4 * 4, 4), dtype=torch.float32, device=dev)

    def user_pass(self, Eu, Ei, r, dEu):
        """scores + loss + coefficients + dE_u."""
        if self.loss in (MSE, WMRB):
            self._partials(Eu.shape[1])
            _abi.call("tmf_user_pass", _LOSS_CODE[self.loss], self.n_users, self.n_items, self.nnz,
                      _abi.ptr(self.row_ptr), _abi.ptr(self.col_idx), _abi.ptr(self.vals), _abi.ptr(Eu), _abi.ptr(Ei),
                      Eu.shape[1], r, _abi.ptr(self.samp), self.S, self.n_work, _abi.ptr(self.w_user), _abi.ptr(self.w_a),
                      _abi.ptr(self.w_b), _abi.ptr(self.w_slot), _abi.ptr(self.part_G), _abi.ptr(self.part_E),
                      _abi.ptr(self.counter), _abi.ptr(self.loss_k), _abi.ptr(self.coef), _abi.ptr(self.coef_pos), _abi.ptr(dEu))
            if self.n_split:
                _abi.call("tmf_user_pass_fixup", _LOSS_CODE[self.loss], self.n_split, _abi.ptr(self.split_user),
                          _abi.ptr(self.split_first), _abi.ptr(self.split_nseg), _abi.ptr(Ei), Eu.shape[1], _abi.ptr(self.samp),
                          self.S, self.nnz, _abi.ptr(self.part_G), _abi.ptr(self.part_E), _abi.ptr(self.coef), _abi.ptr(self.coef_pos),
                          _abi.ptr(dEu))
        else:
            _abi.call("tmf_pair_dots", self.nnz, _abi.ptr(self.coo_rows), _abi.ptr(self.col_idx), _abi.ptr(Eu),
                      _abi.ptr(Ei), Eu.shape[1], _abi.ptr(self.p))
            _abi.call("tmf_kl_moments", self.nnz, _abi.ptr(self.p), _abi.ptr(self.vals), _abi.ptr(self.kl_moments),
                      _abi.ptr(self.red_ws))
            if self.comm is not None:  # user-sharded: the two groups' moments are global (loss_graphs.py:116,118)
                self.comm.allreduce_kl_moments(self.kl_moments)
            _abi.call("tmf_kl_coef_from_moments", self.nnz, _abi.ptr(self.p), _abi.ptr(self.vals), _abi.ptr(self.kl_moments),
                      _abi.ptr(self.kl_loss), _abi.ptr(self.coef), _abi.ptr(self.red_ws))
            self.spmm_ws = self._spmm_ws(dEu.shape[1])
            spmm(self.n_users, self.row_ptr, self.nnz, self.col_idx, None, self.coef, Ei, r, out=dEu, ws=self.spmm_ws)

    def _spmm_ws(self, ld):
        need = max(_abi.query("tmf_spmm_ws_bytes", self.T, ld), _abi.query("tmf_spmm_ws_bytes", self.nnz, ld))
        if self.spmm_ws is None or self.spmm_ws.numel() < need:
            self.spmm_ws = _ws(need)
        return self.spmm_ws

    def item_pass(self, Eu, r, dEi):
        """dE_i[i] = sum over the item-major list of coef * E_u[user]  (deterministic)."""
        ws = self._spmm_ws(dEi.shape[1])
        cpos = None if self.coef_pos is not None else self.t_src  # coefficients already in list order: streamed, not gathered
        spmm(self.n_items, self.t_ptr, self.T, self.t_user, cpos, self.coef, Eu, r, out=dEi, ws=ws)

    # -- loss reporting (matrix_factorization.py:165-167, :179)
    def loss_vector(self):
        """The reference's ``loss_fn`` tensor in stored order."""
        if self.loss == KL:
            return self.kl_loss.reshape(())
        lk = self.loss_k[:self.nnz]
        vals = self.vals
        if self.perm is not None:  # back to the caller's stored order
            out = torch.empty_like(lk)
            out[self.perm] = lk
            v = torch.empty_like(vals)
            v[self.perm] = vals
            lk, vals = out, v
        return lk[vals > 0] if self.loss == WMRB else lk

    def mean_loss(self):
        """``tf.reduce_mean(loss_fn)`` (:179); fixed-order fp64 accumulation on the device."""
        if self.loss == KL:
            return float(self.kl_loss.item())
        if self.n_pos == 0:
            return float("nan")
        _abi.call("tmf_reduce_sum", _abi.ptr(self.loss_k), self.nnz, _abi.ptr(self.red_out), _abi.ptr(self.red_ws))
        return float(self.red_out.item()) / self.n_pos


def capture_graph(fn):
    """Capture ``fn()`` (a sequence of stream-ordered launches on the current torch stream) into a CUDA graph.

    Done by hand instead of ``with torch.cuda.graph(g)``: that context manager runs ``gc.collect()`` and
    ``torch.cuda.empty_cache()`` on entry, which hands every cached block back to the driver -- inside ``fit()`` that
    cost 0.1-0.5 s of cudaFree / cudaMalloc per call (measured: fit(20) 0.21-0.63 s where the 20 epochs take 0.062 s)."""
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        g.capture_begin()
        try:
            fn()
        except BaseException:
            try:
                g.capture_end()
            except Exception:  # noqa: BLE001 -- the capture is already invalid
                pass
            raise
        g.capture_end()
    torch.cuda.current_stream().wait_stream(side)
    return g


class BatchedInteractions:
    """Mini-batch mode (extension, SURVEY 8f-2; the reference is full-batch, matrix_factorization.py:128): the users are cut
    into contiguous blocks of ``batch_size`` users, each with its own ``InteractionPlan`` (CSR slab, item-major list of
    its interactions ++ its users' negatives) built once per fit.  One epoch = one optimizer step per block, in order;
    a block's step sees only its users' interactions, so every other user's gradient row is exactly zero."""

    def __init__(self, inter: SparseInteractions, loss, random_ind, batch_size):
        if loss == KL:
            raise NotImplementedError("mini-batch mode is defined for the per-interaction losses (MSE, WMRB)")
        self.loss = loss
        self.n_users, self.n_items = inter.dense_shape
        B = int(batch_size)
        if B < 1:
            raise ValueError("batch_size must be >= 1 (users per mini-batch)")
        row_ptr, col_idx, vals, coo_rows, perm = inter.csr()
        self.perm = perm
        self.nnz = inter.nnz
        self.vals_sorted = vals
        rp = row_ptr.cpu().numpy()
        ri = None if random_ind is None else to_device(random_ind, torch.int64)
        self.bounds, self.plans = [], []
        for lo in range(0, self.n_users, B):
            hi = min(lo + B, self.n_users)
            a, b = int(rp[lo]), int(rp[hi])
            idx = torch.stack([coo_rows[a:b].to(torch.int64) - lo, col_idx[a:b].to(torch.int64)], 1)
            sub = SparseInteractions(idx, vals[a:b], (hi - lo, self.n_items))
            self.plans.append(InteractionPlan(sub, loss, None if ri is None else ri[lo:hi]))
            self.bounds.append((lo, hi, a, b))
        self.S = self.plans[0].S if self.plans else 0
        self.n_pos = sum(p.n_pos for p in self.plans)
        self.vals = vals

    def set_samples(self, random_ind):
        ri = to_device(random_ind, torch.int64)
        for (lo, hi, _, _), p in zip(self.bounds, self.plans):
            p.set_samples(ri[lo:hi])

    def loss_vector(self):
        """Per-interaction losses in stored order, each taken at the step of its own mini-batch."""
        lk = torch.cat([p.loss_k[:p.nnz] for p in self.plans]) if self.plans else torch.zeros(0, device=self.vals.device)
        vals = self.vals_sorted
        if self.perm is not None:
            out = torch.empty_like(lk); out[self.perm] = lk
            v = torch.empty_like(vals); v[self.perm] = vals
            lk, vals = out, v
        return lk[vals > 0] if self.loss == WMRB else lk

    def mean_loss(self):
        if self.n_pos == 0:
            return float("nan")
        tot = 0.0
        for p in self.plans:
            if p.n_pos:
                tot += p.mean_loss() * p.n_pos
        return tot / self.n_pos


class TrainPlan:
    def __init__(self, user_tower: Tower, item_tower: Tower, inter_plan, r, comm=None):
        self.u, self.i, self.ip, self.r = user_tower, item_tower, inter_plan, int(r)
        self.batched = isinstance(inter_plan, BatchedInteractions)
        if self.batched and comm is not None and comm.world_size > 1:
            import torch.distributed as dist
            nb = torch.tensor([len(inter_plan.plans), -len(inter_plan.plans)], device=inter_plan.vals.device)
            dist.all_reduce(nb, op=dist.ReduceOp.MAX, group=comm.group)
            if int(nb[0]) != -int(nb[1]):
                raise ValueError("mini-batch mode under user sharding needs the same number of mini-batches on every rank "
                                 "(every step is a collective): choose batch_size so that ceil(n_local_users / batch_size) agrees")
        self.comm = comm  # optional teamoflow_b200.mf.dist.GradientSync
        self.opt_state = None  # ({}, {}) = persistent Adam moments per tower (extension; None = the reference's fresh Adam per step)
        if not self.batched:
            inter_plan.comm = comm if (comm is not None and comm.world_size > 1) else None  # KL: global moments
        if comm is not None:
            comm.attach(self)  # item-side gradient (and fusable weights) move into NVLink peer memory

    def forward_backward(self, lr=None, batch=None):
        """One forward + backward.  With ``lr`` (training step) the multi-GPU exchange may fuse the Adam update of the
        item weights into its reduction kernel; returns True when it did.  ``batch``: index of the mini-batch (mini-batch
        mode only): gradients of that block of users' interactions alone."""
        Eu = self.u.forward()
        Ei = self.i.forward()
        if self.batched:
            lo, hi, _, _ = self.ip.bounds[batch]
            bp = self.ip.plans[batch]
            self.u.dE.zero_()  # users outside the block: zero gradient rows (a fresh Adam step of g = 0 moves nothing)
            bp.user_pass(Eu[lo:hi], Ei, self.r, self.u.dE[lo:hi])
            bp.item_pass(Eu[lo:hi], self.r, self.i.dE)
        else:
            self.ip.user_pass(Eu, Ei, self.r, self.u.dE)
            self.ip.item_pass(Eu, self.r, self.i.dE)
        self.u.backward()  # local (needs dE_u only): its shared slices join the item-gradient exchange below
        fused = False
        if self.comm is not None:
            fused = self.comm.sync_grads(self, lr=lr)
        self.i.backward()
        return fused

    # ---- epoch loop.  One step is ~15-25 short launches; on small problems (and on every multi-GPU step, where the
    # exchange adds barrier / reduce / NCCL launches) the host's launch path, not the GPU, sets the pace.  The loop
    # therefore runs its first step eagerly (allocates every workspace, warms NCCL up) and replays ONE captured CUDA graph
    # of a step for the rest.  Everything a step launches is stream-ordered with fixed arguments (the peer barrier takes
    # its epoch from a device-side counter), so a replay is bit-identical to an eager step.
    USE_CUDA_GRAPH = os.environ.get("TMF_CUDA_GRAPH", "1") != "0"   # TMF_CUDA_GRAPH=0: eager epoch loop

    def run(self, n_steps, lr, graph=None):
        """``n_steps`` training steps (the body of the reference's epoch loop, matrix_factorization.py:129-180)."""
        n_steps = int(n_steps)
        use = self.USE_CUDA_GRAPH if graph is None else bool(graph)
        if self.batched:  # one epoch = len(plans) different steps: eager
            use = False
        if getattr(self, "_graph_failed", False):  # a capture of THIS plan's step was refused: stay eager (other plans may still capture)
            use = False
        if not use or self.opt_state is not None or n_steps < 3:
            for _ in range(n_steps):
                self.step(lr)
            return
        self.step(lr)
        g = self._captured_step(lr)
        if g is None:
            for _ in range(n_steps - 1):
                self.step(lr)
            return
        for _ in range(n_steps - 1):
            g.replay()
        _abi.launch_count += self._graph_launches * (n_steps - 1)
        self.graph_replays = getattr(self, "graph_replays", 0) + n_steps - 1

    def invalidate_graph(self):
        """Drop the captured step (its buffers changed: new negatives, new optimizer state)."""
        self._graph = None

    def _captured_step(self, lr):
        if getattr(self, "_graph", None) is not None and self._graph_lr == float(lr):
            return self._graph
        l0, c0 = _abi.launch_count, _abi.call_count
        try:
            torch.cuda.synchronize()
            g = capture_graph(lambda: self.step(lr))
        except Exception as e:  # capture refused (e.g. a collective that cannot be captured): eager loop, say so once
            import sys
            print(f"[teamoflow_b200] CUDA graph capture of the training step failed ({type(e).__name__}: {e}); "
                  "running the epoch loop eagerly", file=sys.stderr)
            torch.cuda.synchronize()
            self._graph_failed = True
            self._graph = None
            return None
        self._graph_launches = _abi.launch_count - l0
        _abi.launch_count, _abi.call_count = l0, c0  # captured, not launched
        self._graph, self._graph_lr = g, float(lr)
        return g

    def step(self, lr):
        """One epoch: a single full-batch step (the reference), or one step per mini-batch in mini-batch mode."""
        for batch in (range(len(self.ip.plans)) if self.batched else (None,)):
            if self.opt_state is not None:  # stateful Adam (extension): the exchange kernel's fused fresh-Adam step does not apply
                self.forward_backward(batch=batch)
                self.u.update(lr, state=self.opt_state[0])
                self.i.update(lr, state=self.opt_state[1])
                continue
            fused = self.forward_backward(lr, batch=batch)
            self.u.update(lr)
            self.i.update(lr, skip=("W",) if fused else ())
