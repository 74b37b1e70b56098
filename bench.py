#!/usr/bin/env python
"""Benchmark of the matrix-factorization hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2|c1|c4|c4mini] [--dump-outputs DIR]

Primary line (one JSON object on stdout, rank 0):
  metric  = training interactions/s, WMRB rank-64 on the ML-20M-shaped synthetic workload (BASELINE.json
            configs[2] -- the single-GPU configuration north_star's target is quoted on), one "step" = one
            full-batch epoch (embed -> fused score/loss/backward -> item-major gradient -> Adam step-1).
  value   = device-resident whole-job throughput (CUDA events, max over ranks);
  e2e     = the same metric through MatrixFactorization.fit() from pinned HOST buffers (H2D of interactions
            and features, structure build, K epochs, D2H of the loss) -- one fit call of K epochs;
  roofline= dominant training kernel vs measured HBM peak; step_roofline = whole step vs SURVEY 8(d) B_alg;
  parity_check = sampled oracle checks of the very state the timed loops left behind: c3 (and c4) -- losses and dE_u of
            512 users and complete dE_i rows of 16 items against oracle.train_step_sparse restricted to those users;
            c5 -- 64 rows of the top-k result bit for bit against the canonical score + (score desc, id asc);
  c4      = BASELINE.json configs[3]: ONE 10M x 2M, 500M-interaction rank-128 problem, user-sharded over the N ranks
            (strong scaling; the same dataset at every N, split by balanced user ranges);
  topk    = secondary metric of BASELINE.json: scored user-item pairs/s of the fused tcgen05 top-100
            (1M x 1M rank-128 by default, item-sharded over the N ranks) with its tensor roofline;
  cpu_baseline = the reference-faithful dense CPU step (oracle/autograd_twin, torch-CPU) on bounded user samples of the
            same workload, item-side fixed cost separated and extrapolated to the full user count (stated as such).
N > 1 (torchrun): users are sharded, every rank holds its own C3-sized user shard ("weak" scaling), the item gradient is
summed over NVLink peer memory each epoch (NCCL all-reduce as the fallback).
"""
import argparse
import json
import math
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: n_users, n_items, nnz, r, S, side features (user cols/nnz per row, item cols/nnz per row)
    "c3": dict(n_u=138_000, n_i=27_000, nnz=20_000_000, r=64, S=128, mu=(64, 4), mi=(1024, 16),
               desc="ML-20M-shaped synthetic: 138k x 27k, 20M interactions, rank 64, WMRB S=128, sparse [I|M] side features"),
    "c2": dict(n_u=943, n_i=1682, nnz=100_000, r=32, S=336, mu=None, mi=None,
               desc="ML-100K-shaped synthetic: 943 x 1682, 100k interactions (ratings>=4 positive), rank 32, WMRB S=336"),
    "c1": dict(n_u=1000, n_i=1000, nnz=10_000, r=10, S=0, mu=None, mi=None,
               desc="toy 1k x 1k, density 0.01, rank 10, MSE"),
    # BASELINE.json configs[3]: ONE 10M x 2M problem, user-sharded over the ranks (strong scaling: the SAME dataset at every N)
    "c4": dict(n_u=10_000_000, n_i=2_000_000, nnz=500_000_000, r=128, S=32, mu=None, mi=None, strong=True,
               desc="10M users x 2M items, 500M interactions, rank 128, WMRB S=32, identity features, user-sharded data parallel"),
    "c4mini": dict(n_u=1_250_000, n_i=2_000_000, nnz=62_500_000, r=128, S=32, mu=None, mi=None,
                   desc="1/8 user shard of the 10M x 2M, 500M-interaction rank-128 WMRB S=32 problem"),
}
PARITY_TOL = 1e-5  # north_star: losses, gradients and scores within 1e-5 relative in fp32


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------- clocks


class ClockSampler:
    """Samples SM clock / throttle reasons during the timed region (pynvml; falls back to nvidia-smi)."""

    def __init__(self, index=0):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            log("clock sampler unavailable:", e)

    def _run(self):
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for b, n in names.items():
                    if bits & b:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self.h is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d["bf16_tflops_sustained"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------- synthetic data


def gen_interactions(n_u, n_i, nnz, seed, dev):
    """Zipf(1.0)-weighted users and items, deduplicated, row-major sorted (SURVEY 8d).  Ids are seeded uniforms looked up in
    a cumulative distribution summed on the host in fp64, so a seed gives the same table on every run (torch.multinomial
    sums its distribution on the device, where the last bits are not reproducible and draws near a bin edge move).  Figures
    stored before this generator (profiles/, BASELINE) were measured on other draws of the same law and sizes."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)

    def zipf_cdf(n):
        c = np.cumsum(1.0 / np.arange(1, n + 1, dtype=np.float64))
        return torch.as_tensor(c / c[-1], device=dev)

    cu, ci = zipf_cdf(n_u), zipf_cdf(n_i)

    def draw(cdf, m):
        return torch.searchsorted(cdf, torch.rand(m, generator=g, device=dev, dtype=torch.float64), right=True)

    keys = torch.empty(0, dtype=torch.int64, device=dev)
    for _ in range(40):
        if keys.numel() >= nnz:
            break
        m = int((nnz - keys.numel()) * 1.5) + 4096
        u = draw(cu, m)
        i = draw(ci, m)
        keys = torch.unique(torch.cat([keys, u * n_i + i]))
        del u, i
    if keys.numel() > nnz:
        sel = torch.randperm(keys.numel(), generator=g, device=dev)[:nnz]
        keys = keys[sel].sort().values
    return keys // n_i, keys % n_i


def side_features(n, ident_cols, extra, seed):
    """CSR of [I | M] with M in {0,1}^{n x cols}, `per` ones per row (values 1.0)."""
    from scipy import sparse
    if extra is None:
        return None
    cols, per = extra
    rng = np.random.default_rng(seed)
    m_idx = np.argpartition(rng.random((n, cols), dtype=np.float32), per, axis=1)[:, :per]
    m_idx.sort(axis=1)
    idx = np.concatenate([np.arange(n, dtype=np.int64)[:, None], ident_cols + m_idx.astype(np.int64)], axis=1)
    ptr = np.arange(n + 1, dtype=np.int64) * (per + 1)
    return sparse.csr_matrix((np.ones(idx.size, np.float32), idx.ravel(), ptr), shape=(n, ident_cols + cols))


def alg_bytes(w, nnz, n_pos, Fu, Fi, nnz_xu, nnz_xi):
    """SURVEY 8(d) algorithmic-bytes model, split by phase (bytes per epoch)."""
    n_u, n_i, r, S = w["n_u"], w["n_i"], w["r"], w["S"]
    row = 4 * r
    user = 8 * nnz + 4 * (n_u + 1) + 4 * nnz + 4 * n_pos + row * (n_u + nnz + n_u)
    item = 8 * nnz + 4 * (n_i + 1) + row * (nnz + n_i)
    if S:
        user += 4 * n_u * S + 4 * n_u * S + row * n_u * S
        item += 8 * n_u * S + row * n_u * S
    feat = 0
    if w["mu"] is not None:
        feat = 2 * (nnz_xu + nnz_xi) * (8 + row) + (n_u + n_i) * row + (Fu + Fi) * row
    opt = 3 * (Fu + Fi) * row
    return {"user_pass": user, "item_pass": item, "features": feat, "adam": opt, "total": user + item + feat + opt}


class Workload:
    """Synthetic inputs of one configuration.  Weak-scaling workloads (c3 ...): every rank draws its own shard.  Strong-scaling
    workloads (c4): every rank generates the SAME full dataset (same seed), then keeps the contiguous user range
    ``dist.balanced_user_bounds`` assigns to it (equal interactions + sampled negatives per rank), user ids re-based."""

    def __init__(self, name, rank, world, host_copy=True, bounds=None):
        from teamoflow_b200.mf import dist as tdist
        from teamoflow_b200.mf import initializer_graphs as I, loss_graphs as L
        from teamoflow_b200.mf.matrix_factorization import MatrixFactorization
        from teamoflow_b200.mf.utils import random_sampler
        self.w = w = dict(WORKLOADS[name])
        self.name, self.rank, self.world = name, rank, world
        dev = torch.device("cuda", torch.cuda.current_device())
        n_i, r, S = w["n_i"], w["r"], w["S"]
        seed = 20240 + {"c1": 1, "c2": 2, "c3": 3, "c4mini": 4, "c4": 4}[name]
        t0 = time.time()
        self.total_nnz = None
        if w.get("strong"):
            rows, cols = gen_interactions(w["n_u"], n_i, w["nnz"], seed * 1000, dev)  # identical on every rank
            self.total_nnz = int(rows.numel())
            lens = torch.bincount(rows, minlength=w["n_u"])
            self.row_weights = (lens + S).cpu().numpy()  # first split: a user costs its interactions + its S negatives
            if bounds is None:
                bounds = tdist.balanced_user_bounds(self.row_weights, world)
            self.bounds = list(bounds)
            lo, hi = bounds[rank], bounds[rank + 1]
            csum = torch.cumsum(lens, 0)
            a = int(csum[lo - 1]) if lo > 0 else 0
            b = int(csum[hi - 1]) if hi > 0 else 0
            rows, cols = (rows[a:b] - lo).clone(), cols[a:b].clone()
            del lens, csum
            torch.cuda.empty_cache()
            w["n_u_total"], w["n_u"], self.user_range = w["n_u"], hi - lo, (lo, hi)
        else:
            rows, cols = gen_interactions(w["n_u"], n_i, w["nnz"], seed * 1000 + rank, dev)
        n_u = w["n_u"]
        self.nnz = int(rows.numel())
        if name == "c2":  # ratings 1..5 with P=(.06,.11,.27,.34,.22); train on ratings >= 4 (benchmarking_ML.py:38,61)
            g = torch.Generator(device=dev); g.manual_seed(seed)
            rating = torch.multinomial(torch.tensor([.06, .11, .27, .34, .22], device=dev), self.nnz, True, generator=g) + 1
            keep = rating >= 4
            rows, cols = rows[keep], cols[keep]
            vals = rating[keep].float()
            self.nnz = int(rows.numel())
        else:
            vals = torch.ones(self.nnz, dtype=torch.float32, device=dev)
        self.n_pos = int((vals > 0).sum())
        idx32 = torch.stack([rows, cols], 1).to(torch.int32)
        del rows, cols
        if host_copy:
            # pinned host copies: the inputs a user of the plugin API holds (int32 ids: half the H2D bytes of tf's int64)
            self.h_indices = idx32.cpu().pin_memory()
            self.h_vals = vals.cpu().pin_memory()
            self.d_indices = self.d_vals = None
        else:
            self.h_indices = self.h_vals = None
            self.d_indices, self.d_vals = idx32, vals
        self.Xu = side_features(n_u, n_u, w["mu"], seed + 11) if w["mu"] else None
        self.Xi = side_features(n_i, n_i, w["mi"], seed + 12) if w["mi"] else None
        self.Fu = n_u + (w["mu"][0] if w["mu"] else 0)
        self.Fi = n_i + (w["mi"][0] if w["mi"] else 0)
        loss = L.MSELoss() if S == 0 else L.WMRBLoss()
        init_u = I.UniformInitializer(seed=seed + 100 + rank) if S else I.NormalInitializer(seed=seed + 100 + rank)
        init_i = I.UniformInitializer(seed=seed + 200) if S else I.NormalInitializer(seed=seed + 200)
        self.model = MatrixFactorization(r, loss_graph=loss, user_weight_graph=init_u, item_weight_graph=init_i,
                                         n_users=n_u, n_items=n_i, n_samples=S if S else None)
        if S:
            self.model.random_ind = random_sampler(n_i, n_u, S, seed=seed + 300 + rank)
        self.lr = 0.1 if S else 1e-2
        self.bytes = alg_bytes(w, self.nnz, self.n_pos, self.Fu, self.Fi,
                               self.Xu.nnz if self.Xu is not None else 0, self.Xi.nnz if self.Xi is not None else 0)
        log(f"[rank {rank}] workload {name}: n_users={n_u} nnz={self.nnz} n_pos={self.n_pos} built in {time.time() - t0:.1f}s; "
            f"B_alg/epoch={self.bytes['total'] / 1e9:.3f} GB")

    def feature_args(self):
        from teamoflow_b200.mf._tensors import FeatureMatrix
        xu = self.Xu if self.Xu is not None else FeatureMatrix.eye(self.w["n_u"])
        xi = self.Xi if self.Xi is not None else FeatureMatrix.eye(self.w["n_i"])
        return xu, xi

    def interactions(self):
        shape = (self.w["n_u"], self.w["n_i"])
        if self.h_indices is not None:
            return (self.h_indices, self.h_vals, shape)
        return (self.d_indices, self.d_vals, shape)

    def h2d_bytes(self):
        b = self.h_indices.numel() * self.h_indices.element_size() + self.h_vals.numel() * 4
        for X in (self.Xu, self.Xi):
            if X is not None:
                b += X.indptr.nbytes // 2 + X.indices.nbytes + X.data.nbytes  # indptr goes down as int32
        return b


# ------------------------------------------------------------------------------------------- training bench


def profile_phases(plan, lr, reps=3):
    """CUDA-event time of each phase of the step (a separate pass, not the timed region)."""
    names = ["embed_fwd", "user_pass", "item_pass", "user_bwd", "comm", "item_bwd", "adam"]
    acc = {n: 0.0 for n in names}
    for _ in range(reps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
        ev[0].record()
        Eu = plan.u.forward(); Ei = plan.i.forward(); ev[1].record()
        plan.ip.user_pass(Eu, Ei, plan.r, plan.u.dE); ev[2].record()
        plan.ip.item_pass(Eu, plan.r, plan.i.dE); ev[3].record()
        plan.u.backward(); ev[4].record()
        fused = False
        if plan.comm is not None:
            fused = plan.comm.sync_grads(plan, lr=lr)
        ev[5].record()
        plan.i.backward(); ev[6].record()
        plan.u.update(lr); plan.i.update(lr, skip=("W",) if fused else ()); ev[7].record()
        torch.cuda.synchronize()
        for j, n in enumerate(names):
            acc[n] += ev[j].elapsed_time(ev[j + 1]) / reps
    acc["embed_bwd"] = acc.pop("user_bwd") + acc.pop("item_bwd")
    return acc


def gather_rate_denominator(plan, kernel_gbs, reps=5):
    """The embedding-row gathers of the user pass, alone (tmf_gather_rate: the same item rows in the same order -- every
    interaction's row, then every user's sampled negatives -- read as float4 and summed in registers).  Where the item table fits
    the L2 the HBM peak is no bound of that kernel; this measured rate is."""
    from teamoflow_b200 import _abi
    ip = plan.ip
    Ei = plan.i.forward()
    idx = ip.col_idx.reshape(-1).to(torch.int32)
    if getattr(ip, "samp", None) is not None and ip.S:
        idx = torch.cat([idx, ip.samp.reshape(-1).to(torch.int32)])
    ld = Ei.shape[1]
    if ld not in (64, 128):
        return None
    outb = torch.empty(148 * 8 * 256, dtype=torch.float32, device=Ei.device)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for it in range(2):  # warm-up, then the timed repetitions
        ev[0].record()
        for _ in range(reps):
            _abi.call("tmf_gather_rate", _abi.ptr(Ei), Ei.shape[0], ld, _abi.ptr(idx), idx.numel(), _abi.ptr(outb), outb.numel())
        ev[1].record(); torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / reps
    gbs = idx.numel() * ld * 4 / (ms * 1e-3) / 1e9
    table_mb = Ei.shape[0] * ld * 4 / 1e6
    return {"rows_gathered": int(idx.numel()), "row_bytes": ld * 4, "table_MB": round(table_mb, 1), "ms": ms, "gather_GBps": gbs,
            "kernel_alg_GBps": kernel_gbs,
            "note": "rate of the bare item-row gathers of one user pass (same rows, same order); the user pass moves "
                    "alg_bytes_per_launch in ms_per_launch while also computing hinges, coefficients and dE_u"}


KERNEL_OF = {"user_pass": "user_pass_kernel", "item_pass": "spmm_seg_kernel (item-major)", "embed_fwd": "spmm_seg_kernel (X.W)",
             "embed_bwd": "spmm_seg_kernel (X^T.dE)", "adam": "adam1_kernel"}


DUMP_BYTES = 64 << 20  # all arrays of --dump-outputs together


def dump_outputs(wl, plan, out_dir, seed=0):
    """Writes what fit() hands its caller after the last step run on `plan` as <out_dir>/<name>.npy: the embeddings
    recomputed from the final weights, the trainables, the per-interaction losses of that step (the reference's loss_fn)
    and their mean.  An array over its share of DUMP_BYTES is cut to a sample of its rows drawn from `seed`, so the same
    workload dumps the same entries on every run and two builds can be compared output for output."""
    r = wl.model.n_components
    arrays = {"user_embedding": plan.u.forward()[:, :r], "item_embedding": plan.i.forward()[:, :r]}
    for side, tower in (("user", plan.u), ("item", plan.i)):
        for j, t in enumerate(wl.model._trainable_list(tower)):
            arrays[f"{side}_trainable_{j}"] = t
    arrays["loss"] = plan.ip.loss_vector().reshape(-1)  # KL's loss is a scalar
    cap = DUMP_BYTES // (len(arrays) + 1)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        row_bytes = t[:1].numel() * 4
        if t.shape[0] * row_bytes > cap:
            rows = np.sort(np.random.default_rng(seed).choice(t.shape[0], cap // row_bytes, replace=False))
            t = t[torch.as_tensor(rows, device=t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    np.save(os.path.join(out_dir, "mean_loss.npy"), np.array([plan.ip.mean_loss()], np.float64))


def train_bench(wl, comm, steps, warmup, local, world, hbm_peak, parity_kw=None, dump_dir=None):
    """Device-resident timing of `steps` epochs of `wl` (inputs and structures already in HBM): returns the plan and a dict.
    `parity_kw`: run the strict sampled oracle check at the initial weights first (result under "parity_init").
    `dump_dir`: write the outputs of the last timed step there (dump_outputs)."""
    from teamoflow_b200 import _abi
    dev = torch.device("cuda", local)
    xu, xi = wl.feature_args()
    plan = wl.model._prepare(xu, xi, wl.interactions(), comm=comm)
    if comm is not None:
        comm.broadcast_params(plan.u, plan.i)
    parity_init = None
    if parity_kw is not None:
        try:
            parity_init = parity_train_sample(plan, strict=True, **parity_kw)
        except Exception as e:
            import traceback
            log(traceback.format_exc())
            parity_init = {"ok": False, "error": f"{type(e).__name__}: {e}"}
    # warm-up through the same entry point as the timed loop (TrainPlan.run = the body of fit()'s epoch loop: first step
    # eager, the rest replayed from ONE captured CUDA graph of a step); the capture happens here
    plan.run(max(warmup, 3), wl.lr)
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    l0 = _abi.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        e0.record()
        plan.run(steps, wl.lr)
        e1.record()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
    launches = _abi.launch_count - l0
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        torch.distributed.all_reduce(ms_total, op=torch.distributed.ReduceOp.MAX)
    ms_step = float(ms_total) / steps
    loss_now = plan.ip.mean_loss() if comm is None else comm.mean_loss(plan.ip)
    if dump_dir is not None:  # before profile_phases, which trains the plan further
        dump_outputs(wl, plan, dump_dir)
    phases = profile_phases(plan, wl.lr)
    phase_bytes = {"user_pass": wl.bytes["user_pass"], "item_pass": wl.bytes["item_pass"],
                   "embed_fwd": wl.bytes["features"] / 2, "embed_bwd": wl.bytes["features"] / 2, "adam": wl.bytes["adam"]}
    dom = max(KERNEL_OF, key=lambda n: phases[n])
    dom_gbs = phase_bytes[dom] / (phases[dom] * 1e-3) / 1e9 if phases[dom] > 0 else 0.0
    step_gbs = wl.bytes["total"] / (ms_step * 1e-3) / 1e9
    return plan, dict(ms_step=ms_step, launches=launches, loss=loss_now, phases=phases, dom=dom, dom_gbs=dom_gbs, step_gbs=step_gbs,
                      phase_bytes=phase_bytes, clocks=clk.summary(), parity_init=parity_init)


# ------------------------------------------------------------------------------------------- sampled parity checks


def _rel_err(got, want):
    want = np.asarray(want, np.float64)
    scale = max(float(np.abs(want).max()) if want.size else 0.0, 1e-30)
    return float(np.abs(np.asarray(got, np.float64) - want).max() / scale) if want.size else 0.0


def parity_train_sample(plan, n_us=512, n_is=16, seed=1, max_len=200_000, strict=True, max_inter=400_000):
    """Checks the CUDA training step against the fp64 oracle on a sample of the FULL-SIZE problem (same plan object, same kernels,
    same structures as the timed loop: heavy-user slicing, int32 offsets, the persistent schedule).

    Called twice: before the timed loop at the configuration's initial weights (`strict`: plain north_star tolerance, errors <=
    1e-5 * max|x|), and after it at the weights the timed loop left behind.  Those are badly conditioned for fp32 -- 26 sign-like
    lr = 0.1 updates blow the scores up to |p| ~ 1e3 while hinges h = 1 - p + s stay O(1), so h carries an absolute fp32 rounding
    error of ~4e-6 (1 + sum|u_c v_c|) that no implementation in fp32 (the reference's TensorFlow included) can avoid -- so there the
    tolerance is 1e-5 * max|x| PLUS the first-order propagation of that dot-product rounding bound through m, w = (n/S)/(1+m), c_k,
    G_uj into each loss and each dE_u component (`bud_l`, `bud_E` below); the plain relative errors are reported beside it.

    Runs the step's kernels once more WITHOUT an update (embed -> user pass -> item-major pass; under user sharding this is
    the rank's LOCAL partial dE_i, before the exchange), then compares on the host:
      (A) `n_us` users (random, plus the heaviest one): per-interaction losses and their dE_u rows against
          oracle.train_step_sparse run on exactly those users (their interactions, their negatives, the item rows they touch);
      (B) `n_is` items: their COMPLETE dE_i rows against the same oracle run on ALL users whose interactions or negatives
          touch those items (so the oracle's rows are complete too).
    The WMRB indicator 1[h >= 0] is discontinuous: a hinge whose fp64 value is within the fp32 rounding of its two dot products
    of 0 (|h| < 4e-6 (1 + sum|u_c v_c|)) may legitimately fall on the other side in fp32, so users holding such a hinge are
    excluded from the dE_u comparison and items they touch from the dE_i comparison (counted in the result); losses are
    continuous and are compared for every sampled interaction.
      (C) any item, the most popular included: dE_i rows recomputed in fp64 from the kernels' own coefficients."""
    from oracle import mf_oracle as o
    from scipy import sparse
    from teamoflow_b200.mf import _engine as eng
    ip, r = plan.ip, plan.r
    wmrb = ip.loss == eng.WMRB
    Eu = plan.u.forward(); Ei = plan.i.forward()
    ip.user_pass(Eu, Ei, r, plan.u.dE)
    ip.item_pass(Eu, r, plan.i.dE)
    torch.cuda.synchronize()
    rng = np.random.default_rng(seed)
    row_ptr = ip.row_ptr
    lens = (row_ptr[1:] - row_ptr[:-1])
    n_users, n_items, S = ip.n_users, ip.n_items, ip.S

    def run(users):
        """oracle on the sub-problem of `users` (sorted, unique): returns losses per interaction position, dE_u rows,
        (item id -> dE_i row) for every touched item, ambiguous-user mask, ambiguous item set."""
        ut = torch.as_tensor(users, device=row_ptr.device, dtype=torch.int64)
        a, b = row_ptr[ut].long(), row_ptr[ut + 1].long()
        cnt = (b - a)
        pos = torch.repeat_interleave(a - (torch.cumsum(cnt, 0) - cnt), cnt) + torch.arange(int(cnt.sum()), device=ut.device)
        sub_rows = torch.repeat_interleave(torch.arange(ut.numel(), device=ut.device), cnt).cpu().numpy()
        cols = ip.col_idx[pos].long()
        vals = ip.vals[pos].cpu().numpy().astype(np.float64)
        samp = ip.samp[ut].long() if wmrb else None
        touched = torch.unique(torch.cat([cols, samp.reshape(-1)]) if wmrb else cols)
        remap = torch.full((n_items,), -1, dtype=torch.int64, device=ut.device)
        remap[touched] = torch.arange(touched.numel(), device=ut.device)
        Eu_s = Eu[ut, :r].double().cpu().numpy()
        Ei_s = Ei[touched, :r].double().cpu().numpy()
        cols_s = remap[cols].cpu().numpy()
        samp_s = remap[samp].cpu().numpy() if wmrb else None
        lvec, gu, gi, _, _ = o.train_step_sparse(ip.loss, sparse.identity(len(users), format="csr"),
                                                 sparse.identity(int(touched.numel()), format="csr"), "linear", "linear",
                                                 {"W": Eu_s}, {"W": Ei_s}, sub_rows, cols_s, vals, samp_s, n_items, S or None, update=False)
        amb_user = np.zeros(len(users), bool)
        amb_items = np.zeros(0, np.int64)
        bud_l = np.zeros(int((vals > 0).sum()) if wmrb else vals.size)  # first-order fp32 rounding budget of each loss
        bud_E = np.zeros((len(users), r))                               # ... and of each dE_u component
        abs_terms = None                                                # sum of |terms| of each dE_u component (WMRB)
        if wmrb:
            # a hinge is ambiguous when |h| is within the fp32 rounding of its two dot products: 4e-6 * (1 + sum|u_c v_c| of both)
            p = np.einsum("kc,kc->k", Eu_s[sub_rows], Ei_s[cols_s])
            pa = np.einsum("kc,kc->k", np.abs(Eu_s)[sub_rows], np.abs(Ei_s)[cols_s])
            Es = Ei_s[samp_s.ravel()].reshape(len(users), S, -1)
            ss = np.einsum("uc,usc->us", Eu_s, Es)
            sa = np.einsum("uc,usc->us", np.abs(Eu_s), np.abs(Es))
            del Es
            pk = np.nonzero(vals > 0)[0]
            amb_k, amb_j = [], []
            scale = n_items / S
            absEi = np.abs(Ei_s)
            gb = np.zeros((len(users), S))      # sum_k eps_k w_k 1_kj  (budget of G_uj)
            Gs = np.zeros((len(users), S))      # sum_k w_k 1_kj        (G_uj itself, for the accumulation slack)
            terms = np.zeros((len(users), r))   # sum |c_k| |E_i[i_k]|
            for c0 in range(0, pk.size, 1 << 15):
                kk = pk[c0:c0 + (1 << 15)]
                uk = sub_rows[kk]
                h = (1.0 - p[kk])[:, None] + ss[uk]
                dh = 4e-6 * (1.0 + pa[kk][:, None] + sa[uk])      # |fp32 h - h| <= gamma_r (1 + sum|u_c v_c| of both dot products)
                act = h >= 0
                m = scale * np.maximum(h, 0.0).sum(1)
                eps = scale * np.where(h > -dh, dh, 0.0).sum(1) / (1.0 + m) + 1e-6   # relative error of (1 + m_k), hence of w_k
                bud_l[c0:c0 + kk.size] = eps                         # d log(1 + m) = dm / (1 + m)
                w = scale / (1.0 + m)
                ck = w * act.sum(1)
                np.add.at(bud_E, uk, (eps * ck)[:, None] * absEi[cols_s[kk]])
                np.add.at(terms, uk, ck[:, None] * absEi[cols_s[kk]])
                np.add.at(gb, uk, (eps * w)[:, None] * act)
                np.add.at(Gs, uk, w[:, None] * act)
                ak, aj = np.nonzero(np.abs(h) < dh)
                amb_k.append(kk[ak]); amb_j.append(samp_s[sub_rows[kk[ak]], aj])
            absEs = absEi[samp_s.ravel()].reshape(len(users), S, -1)
            bud_E += np.einsum("us,usc->uc", gb, absEs)
            abs_terms = terms + np.einsum("us,usc->uc", Gs, absEs)
            bud_E += 2e-6 * abs_terms  # fp32 accumulation of the row sums themselves
            del absEs
            amb_k = np.concatenate(amb_k) if amb_k else np.zeros(0, np.int64)
            amb_user[sub_rows[amb_k]] = True
            amb_items = np.unique(np.concatenate([cols_s[amb_k], np.concatenate(amb_j) if amb_j else np.zeros(0, np.int64)]))
        return dict(pos=pos, lvec=lvec, vals=vals, dEu=gu["W"], dEi=gi["W"], touched=touched.cpu().numpy(), amb_user=amb_user,
                    amb_items=amb_items, ut=ut, bud_l=bud_l, bud_E=bud_E, abs_terms=abs_terms)

    out = {"tolerance": PARITY_TOL if strict else "1e-5 * max|x| + first-order fp32 dot-product rounding budget", "loss": ip.loss}

    def within(got, want, budget):
        want = np.asarray(want, np.float64)
        if not want.size:
            return True
        return bool(np.all(np.abs(np.asarray(got, np.float64) - want) <= PARITY_TOL * np.abs(want).max() + budget))
    # ---- (A) users
    cand = torch.nonzero((lens > 0) & (lens <= max_len)).reshape(-1).cpu().numpy()
    users = rng.choice(cand, size=min(n_us, cand.size), replace=False)
    # bound the host work: a rank of a strong-scaling split may hold only very heavy users (C4 at N = 8: 1,379 users, 74k interactions
    # each) -- keep a random prefix of the sample within `max_inter` interactions (at least 4 users), the heaviest user on top
    ulen = lens[torch.as_tensor(users, device=lens.device)].cpu().numpy()
    users = users[:max(4, int(np.searchsorted(np.cumsum(ulen), max_inter, side="right")))]
    heavy = int(torch.argmax(torch.where(lens <= max_len, lens, torch.zeros_like(lens))))
    users = np.unique(np.concatenate([users, [heavy]]))
    A = run(users)
    lk = ip.loss_k[A["pos"]].double().cpu().numpy()
    got_l = lk[A["vals"] > 0] if wmrb else lk
    out["users"] = int(users.size)
    out["interactions"] = int(A["pos"].numel())
    out["heaviest_user_interactions"] = int(lens[heavy])
    out["loss_max_rel_err"] = _rel_err(got_l, A["lvec"])
    keep = ~A["amb_user"]
    out["ambiguous_users_excluded"] = int(A["amb_user"].sum())
    got_dEu = plan.u.dE[A["ut"], :r].double().cpu().numpy()
    out["dEu_max_rel_err"] = _rel_err(got_dEu[keep], A["dEu"][keep])
    if A["abs_terms"] is not None and int(keep.sum()) > 0:
        # a dE_u component is a sum of up to n_items signed terms c_k E_i[i_k] - G_uj E_i[s_j]; the rounding of ANY fp32 summation order
        # (this kernel's, tf's) scales with the sum of their magnitudes, not with the result -- error relative to that sum, per component
        out["dEu_max_err_over_abs_terms"] = float((np.abs(got_dEu[keep] - A["dEu"][keep]) / np.maximum(A["abs_terms"][keep], 1e-30)).max())
    if not strict:
        out["loss_within_budget"] = within(got_l, A["lvec"], A["bud_l"])
        out["dEu_within_budget"] = within(got_dEu[keep], A["dEu"][keep], A["bud_E"][keep])
        out["loss_frac_within_plain_tol"] = float(np.mean(np.abs(got_l - A["lvec"]) <= PARITY_TOL * max(np.abs(A["lvec"]).max(), 1e-30))) if got_l.size else 1.0
    # ---- (B) items: complete rows need every user that touches the item (interactions and negatives)
    t_ptr = ip.t_ptr
    tl = (t_ptr[1:] - t_ptr[:-1])

    def entries_of(items):
        it = torch.as_tensor(items, device=t_ptr.device, dtype=torch.int64)
        a, b = t_ptr[it].long(), t_ptr[it + 1].long()
        cnt = b - a
        pos = torch.repeat_interleave(a - (torch.cumsum(cnt, 0) - cnt), cnt) + torch.arange(int(cnt.sum()), device=it.device)
        which = torch.repeat_interleave(torch.arange(it.numel(), device=it.device), cnt)
        return it, pos, which, cnt

    icand = torch.nonzero((tl > 0) & (tl <= 1000)).reshape(-1).cpu().numpy()
    items = np.sort(rng.choice(icand, size=min(2 * n_is, icand.size), replace=False)) if icand.size else np.zeros(0, np.int64)
    out["items"], out["dEi_max_rel_err"] = 0, None
    if items.size:
        it, pos, which, _ = entries_of(items)
        eu = ip.t_user[pos].long()
        heavy_items = torch.unique(which[lens[eu] > max_len]).cpu().numpy()  # a too-heavy user makes the row too costly for the host
        items = np.delete(items, heavy_items)[:n_is]
    if items.size:
        it, pos, which, _ = entries_of(items)
        users_b = torch.unique(ip.t_user[pos].long()).cpu().numpy()
        while items.size > 1 and int(lens[torch.as_tensor(users_b, device=lens.device)].sum()) > 4 * max_inter:  # bound the host work
            items = items[:items.size // 2]
            it, pos, which, _ = entries_of(items)
            users_b = torch.unique(ip.t_user[pos].long()).cpu().numpy()
        B = run(users_b)
        where = {int(g): j for j, g in enumerate(B["touched"])}
        amb = set(int(B["touched"][j]) for j in B["amb_items"])
        rows_ok = [int(i) for i in items if int(i) in where and int(i) not in amb]
        if rows_ok:
            got = plan.i.dE[torch.as_tensor(rows_ok, device=it.device, dtype=torch.int64), :r].double().cpu().numpy()
            want = np.stack([B["dEi"][where[i]] for i in rows_ok])
            out["dEi_max_rel_err"] = _rel_err(got, want)
        out["items"] = len(rows_ok)
        out["items_users_involved"] = int(users_b.size)
        out["ambiguous_items_excluded"] = int(items.size - len(rows_ok))
    # ---- (C) the item-major segment-sum alone, on ANY item (the most popular one included): dE_i rows recomputed on the host in
    # fp64 from the kernels' own coefficients (c_k / G_uj, whose producers (A) checks) and E_u rows, in list order
    icand = torch.nonzero(tl > 0).reshape(-1).cpu().numpy()
    out["segment_items"], out["dEi_segment_max_rel_err"] = 0, None
    if icand.size:
        pop = int(torch.argmax(tl))
        items_c = np.unique(np.concatenate([rng.choice(icand, size=min(63, icand.size), replace=False), [pop]]))
        it, pos, which, cnt = entries_of(items_c)
        coef = (ip.coef[pos] if ip.coef_pos is not None else ip.coef[ip.t_src[pos].long()]).double()  # list order when the user pass scatters
        rows_e = Eu[ip.t_user[pos].long(), :r].double() * coef[:, None]
        want = torch.zeros(it.numel(), r, dtype=torch.float64, device=it.device).index_add_(0, which, rows_e).cpu().numpy()
        got = plan.i.dE[it, :r].double().cpu().numpy()
        out["segment_items"] = int(it.numel())
        out["most_popular_item_entries"] = int(tl[pop])
        out["dEi_segment_max_rel_err"] = _rel_err(got, want)
    if strict:
        # dE_u: 1e-5 of the largest gradient entry, or -- for the rows whose sums run over 10^4 terms -- 1e-5 of the component's own
        # sum of term magnitudes (the forward-error form of the same tolerance; both numbers are reported)
        dEu_err = min(out["dEu_max_rel_err"], out.get("dEu_max_err_over_abs_terms", np.inf))
        errs = [out["loss_max_rel_err"], dEu_err] + [e for e in (out["dEi_max_rel_err"], out["dEi_segment_max_rel_err"]) if e is not None]
        out["ok"] = bool(all(e <= PARITY_TOL for e in errs) and out["users"] > 0 and int(keep.sum()) > 0)
    else:  # complete dE_i rows inherit the users' conditioning: here only the segment-sum form (C) is held to the plain tolerance
        out["ok"] = bool(out["loss_within_budget"] and out["dEu_within_budget"] and out["users"] > 0 and
                         (out["dEi_segment_max_rel_err"] is None or out["dEi_segment_max_rel_err"] <= PARITY_TOL))
    return out


def parity_topk_rows(idx, U, r, k, v_shards, n_rows=64, n_cand=2000, seed=5):
    """Bit-exact check of `n_rows` rows of a top-k result: the candidates are the top `n_cand` items per shard by fp64 score (a
    superset of the answer by a huge margin), ranked on the host by the oracle's canonical score, (score desc, id asc).
    `v_shards`: list of (item offset, V storage) covering all items."""
    from oracle import mf_oracle as o
    rng = np.random.default_rng(seed)
    n_u = U.shape[0]
    rows = np.unique(np.concatenate([[0, n_u // 2, n_u - 1], rng.choice(n_u, size=min(n_rows, n_u), replace=False)]))[:max(n_rows, 3)]
    rt = torch.as_tensor(rows, device=U.device)
    Ur = U[rt, :r].double()
    cands = []
    for off, V in v_shards:
        sc = Ur @ V[:, :r].double().T
        top = torch.topk(sc, min(n_cand, V.shape[0]), dim=1).indices + off
        cands.append(top)
    cand = torch.cat(cands, 1)
    cand_np = cand.cpu().numpy()
    U_np = U[rt, :r].cpu().numpy()
    # gather the candidates' item rows shard by shard
    Vrows = torch.empty(cand.shape[0], cand.shape[1], r, dtype=torch.float32, device=U.device)
    for off, V in v_shards:
        m = (cand >= off) & (cand < off + V.shape[0])
        Vrows[m] = V[(cand[m] - off), :r]
    Vrows = Vrows.cpu().numpy()
    bad = 0
    for j in range(rows.size):
        sc = o.canonical_pair_scores(np.repeat(U_np[j:j + 1], cand_np.shape[1], 0), Vrows[j], np.arange(cand_np.shape[1]), np.arange(cand_np.shape[1]))
        order = np.lexsort((cand_np[j], -sc.astype(np.float64)))[:k]
        want = cand_np[j][order]
        bad += int(not np.array_equal(want, idx[rows[j]].cpu().numpy()))
    return {"rows": int(rows.size), "mismatching_rows": bad, "ok": bad == 0,
            "method": f"top-{n_cand} fp64 candidates per shard -> oracle.canonical_pair_scores -> (score desc, id asc) -> first {k}"}


# ------------------------------------------------------------------------------------------- top-k bench


def _topk_traffic(n_u, n_i, world):
    """DRAM bytes per launch of the dominant top-k kernel from the committed ncu capture (only for the captured shape)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if world == 1 and n_u == 1_000_000 and n_i == 1_000_000 and os.path.exists(tpath):
            return json.load(open(tpath)).get("score_topk_kernel"), name
    return None, None


def bench_topk(n_u, n_i, r, k, steps, warmup, world, rank, hbm_peak, tf_peak, user_sharded_too=False):
    from teamoflow_b200 import _abi
    from teamoflow_b200.mf import dist as tdist
    from teamoflow_b200.mf._engine import new_storage
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev); g.manual_seed(20245)
    bounds = tdist.shard_bounds(n_i, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    U = new_storage(n_u, r); U[:, :r] = torch.randn(n_u, r, generator=g, device=dev) / math.sqrt(r)

    def item_slab(gr):
        gi = torch.Generator(device=dev); gi.manual_seed(30000 + gr)
        n = bounds[gr + 1] - bounds[gr]
        Vg = new_storage(n, r); Vg[:, :r] = torch.randn(n, r, generator=gi, device=dev) / math.sqrt(r)
        return Vg

    V = item_slab(rank)
    times = []
    l0 = _abi.launch_count
    for s in range(warmup + steps):
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        idx, sc = tdist.sharded_topk(U, V, r, k, False, lo)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        if s >= warmup:
            times.append(float(ms))
    launches = (_abi.launch_count - l0) // (warmup + steps)
    # phases of one rank's call (CUDA events on the launching stream; a separate pass, not the headline timing)
    phases = None
    if world > 1:
        torch.distributed.barrier(); torch.cuda.synchronize()
        evs = []
        tdist.sharded_topk(U, V, r, k, False, lo, events=evs)
        torch.cuda.synchronize()
        phases = {f"{name}_ms": evs[j][1].elapsed_time(e) for j, (name, e) in enumerate(evs[1:])}
        phases["bound_sample_items"] = tdist.bound_sample_size(hi - lo, n_i, k, world)
        phases["exchange"] = tdist.exchange_mode()
    # the alternative decomposition (users sharded, items replicated: no merge), only on request
    user_sharded = None
    if world > 1 and user_sharded_too:
        ub = tdist.shard_bounds(n_u, world)
        n_loc = ub[1] - ub[0]  # equal slices (the bench sizes divide evenly; a short last slice is padded)
        Uloc = new_storage(n_loc, r)
        Uloc[:ub[rank + 1] - ub[rank]] = U[ub[rank]:ub[rank + 1]]
        Vfull = torch.cat([item_slab(gr) for gr in range(world)])
        ts = []
        for s in range(warmup + steps):
            torch.distributed.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            tdist.user_sharded_topk(Uloc, Vfull, r, k, False)
            e1.record()
            torch.cuda.synchronize()
            ms_u = torch.tensor([e0.elapsed_time(e1)], device=dev)
            torch.distributed.all_reduce(ms_u, op=torch.distributed.ReduceOp.MAX)
            if s >= warmup:
                ts.append(float(ms_u))
        ms_us = float(np.mean(ts))
        user_sharded = {"ms_per_step": ms_us, "value": float(n_u) * float(n_i) / (ms_us * 1e-3), "unit": "pairs/s",
                        "note": "users sharded, items replicated on every GPU, result all-gathered; no merge needed"}
        del Uloc, Vfull
    # ---- parity: sampled rows of the (merged) result, bit for bit against the oracle's canonical score + tie order
    parity = None
    if rank == 0:
        try:
            shards = [(bounds[gr], V if gr == rank else item_slab(gr)) for gr in range(world)]
            parity = parity_topk_rows(idx, U, r, k, shards)
            del shards
        except Exception as e:
            parity = {"ok": False, "error": f"{type(e).__name__}: {e}"}
    if world > 1:
        # rank 0 checks rows of the merged result against the oracle; the other ranks check that they hold the same merged result
        # (position-weighted checksum of all n_users x k indices)
        wts = torch.arange(1, k + 1, device=dev, dtype=torch.int64)
        chk = torch.stack([idx.long().sum(), (idx.long() * wts).sum()])
        gl = [torch.empty_like(chk) for _ in range(world)]
        torch.distributed.all_gather(gl, chk)
        if rank != 0:
            same = bool(torch.equal(gl[rank], gl[0]))
            parity = {"ok": same, "method": "merged result identical to rank 0's (checksum over all rows); rank 0 checks rows against the oracle"}
    # the recall_at_k path at the same scale (clamped scores, CSR interaction table; single GPU only)
    recall = None
    if world == 1:
        try:
            from teamoflow_b200.mf.matrix_factorization import MatrixFactorization
            from teamoflow_b200.mf._tensors import SparseInteractions
            mdl = MatrixFactorization(r)
            mdl.user_embedding, mdl.item_embedding = U[:, :r], V[:, :r]
            ga = torch.Generator(device=dev); ga.manual_seed(777)
            npos = min(50 * n_u, 50_000_000)
            keys = torch.unique(torch.randint(0, n_u * n_i, (npos,), generator=ga, device=dev, dtype=torch.int64))
            A = SparseInteractions(torch.stack([keys // n_i, keys % n_i], 1), torch.ones(keys.numel(), device=dev), (n_u, n_i))
            A.csr()
            del keys
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rec = mdl.recall_at_k(A, k=k)
            e1.record()
            torch.cuda.synchronize()
            recall = {"ms": e0.elapsed_time(e1), "recall_at_k_mean": float(rec.mean()), "positives": int(A.nnz),
                      "note": "MatrixFactorization.recall_at_k(A, k): clamped fused top-k + CSR membership kernel"}
            del A, mdl
        except Exception as e:
            recall = {"error": f"{type(e).__name__}: {e}"}
    ms = float(np.mean(times))
    pairs = float(n_u) * float(n_i)
    flops = 2.0 * pairs * r
    # e2e: host fp32 embeddings -> device -> top-k -> indices back on the host
    hU, hV = U.cpu().pin_memory(), V.cpu().pin_memory()
    h_out = torch.empty(n_u, k, dtype=torch.int32).pin_memory()  # the caller's (pinned) result buffer
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dU, dV = hU.to(dev, non_blocking=True), hV.to(dev, non_blocking=True)
    idx2, _ = tdist.sharded_topk(dU, dV, r, k, False, lo)
    out = h_out.copy_(idx2, non_blocking=True)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    dt = torch.tensor([t1 - t0], device=dev, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(dt, op=torch.distributed.ReduceOp.MAX)
    traffic, traffic_src = _topk_traffic(n_u, n_i, world)
    return {"metric": "top-k scored user-item pairs/sec", "value": pairs / (ms * 1e-3), "unit": "pairs/s", "ms_per_step": ms,
            "step_ms": [round(t, 3) for t in times], "warmup": warmup,
            "config": {"workload": f"{n_u} users x {n_i} items rank-{r} top-{k} (raw scores), item-sharded x{world}", "k": k,
                       "exchange": (tdist.exchange_mode() + " (bounds all-gathered, lists merged over NVLink peer memory)") if world > 1 else "none"},
            "dtype": "16-bit tensor-core operands (fp16 or bf16, chosen from the data), fp32 accumulate in TMEM, fp64-accumulated rerank",
            "roofline": {"bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12 / world, "peak": tf_peak, "unit": "TFLOP/s",
                         "frac": flops / (ms * 1e-3) / 1e12 / world / tf_peak, "traffic": traffic,
                         "traffic_note": f"DRAM bytes of one score_topk_kernel launch from the committed ncu --set full capture (profiles/{traffic_src})"},
            "e2e": {"value": pairs / float(dt), "unit": "pairs/s", "h2d_bytes_per_step": hU.numel() * 4 + hV.numel() * 4,
                    "d2h_bytes_per_step": out.numel() * 4},
            "gpu_launches": launches, "parity_check": parity, "user_sharded": user_sharded, "recall_path": recall,
            "phases_ms": phases}


# ------------------------------------------------------------------------------------------- CPU baselines


def _cpu_threads():
    """All host cores, whatever OMP_NUM_THREADS says (torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, which
    starved the reference arm of round 1 at N > 1)."""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:  # pragma: no cover
        pass
    torch.set_num_threads(n)
    return n


def _cpu_sample(w, n_sub, rng):
    n_i, S = w["n_i"], w["S"]
    per_user = max(1, w["nnz"] // w["n_u"])
    rows = np.repeat(np.arange(n_sub), per_user)
    wi = 1.0 / np.arange(1, n_i + 1)
    cols = rng.choice(n_i, size=rows.size, p=wi / wi.sum())
    cells = np.unique(rows.astype(np.int64) * n_i + cols)
    rows, cols = cells // n_i, cells % n_i
    vals = np.ones(rows.size, np.float32)
    samp = np.stack([rng.choice(n_i, max(S, 1), replace=False) for _ in range(n_sub)]) if S else None
    return rows, cols, vals, samp


def _time_steps(fn, budget_s, max_steps=6):
    times = []
    t_all = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
        if len(times) >= 2 and (time.perf_counter() - t_all > budget_s or len(times) >= max_steps):
            break
    return float(np.median(times[1:])) if len(times) > 1 else times[0], len(times) - 1


def cpu_reference_step(wl_name, budget_s=20.0):
    """The reference's own algorithm (dense features, dense U V^T, gathers, autograd of the summed loss, Keras-Adam step 1)
    on host cores via oracle/autograd_twin (torch-CPU; TensorFlow is not installable here).

    The full configuration cannot run densely on a host (C3: a 14.9 GB score matrix and a 76 GB dense user-feature matrix), so
    the step is timed on TWO user samples (n and 2n users against ALL items).  Its cost is t(n) = t_item + n * t_user: the
    item-side work (dense X_i W_i forward/backward over all items) is a fixed cost per step that a sample must not be charged
    per interaction (ADVICE r1), so the two timings are solved for t_item and t_user and the full-configuration step is
    EXTRAPOLATED as t_item + n_users * t_user.  (Favourable to the reference: its dense n_users x n_users identity-feature matmul
    grows quadratically and is left out.)  Returns a dict; `value` = full-config interactions / extrapolated step time."""
    from oracle import autograd_twin as tw
    from oracle import mf_oracle as o
    cores = _cpu_threads()
    w = WORKLOADS[wl_name]
    n_i, r, S = w["n_i"], w["r"], w["S"]
    n1 = {"c3": 2048, "c2": 943, "c1": 1000, "c4mini": 32, "c4": 32}[wl_name]
    full = n1 >= w["n_u"]
    sizes = [w["n_u"]] if full else [n1, 4 * n1]
    loss = "wmrb" if S else "mse"
    meas = []
    for n_sub in sizes:
        rng = np.random.default_rng(7)
        rows, cols, vals, samp = _cpu_sample(w, n_sub, rng)
        # dense features exactly like the reference (tf.eye / dense [I|M]); user identity columns restricted to the sample
        Xu = np.eye(n_sub, dtype=np.float32)
        Xi = np.eye(n_i, dtype=np.float32)
        if w["mu"]:
            Xu = np.concatenate([Xu, (rng.random((n_sub, w["mu"][0])) < w["mu"][1] / w["mu"][0]).astype(np.float32)], 1)
            Xi = np.concatenate([Xi, (rng.random((n_i, w["mi"][0])) < w["mi"][1] / w["mi"][0]).astype(np.float32)], 1)
        state = {"pu": {"W": o.uniform_initializer(Xu.shape[1], r, rng)}, "pi": {"W": o.uniform_initializer(Xi.shape[1], r, rng)}}

        def step():
            _, _, _, state["pu"], state["pi"] = tw.train_step(loss, Xu, Xi, "linear", "linear", state["pu"], state["pi"], rows, cols, vals,
                                                              samp, n_i, S or None, lr=0.1 if S else 1e-2)
        t, n_t = _time_steps(step, budget_s / len(sizes))
        meas.append((n_sub, rows.size, t, n_t))
    if full:
        n_sub, nnz_s, t, n_t = meas[0]
        return {"value": nnz_s / t, "unit": "interactions/s", "cores": cores, "kind": "port", "same_config": True, "extrapolated": False,
                "sample": f"the full configuration ({n_sub} users x {n_i} items, {nnz_s} interactions), dense features + dense U.V^T + "
                          f"autograd + Adam step-1 (oracle/autograd_twin, torch-CPU), median of {n_t} steps"}
    (na, nnz_a, ta, _), (nb, nnz_b, tb, n_t) = meas
    t_user = (tb - ta) / (nb - na)
    if not t_user > 0.02 * tb / nb:  # the slope drowned in timing noise: charge the whole larger step to its users (upper bound on t_user)
        t_user = tb / nb
    t_item = max(ta - na * t_user, 0.0)
    t_full = t_item + w["n_u"] * t_user
    return {"value": w["nnz"] / t_full, "unit": "interactions/s", "cores": cores, "kind": "port", "same_config": False, "extrapolated": True,
            "measured": {"users": [na, nb], "interactions": [int(nnz_a), int(nnz_b)], "step_s": [ta, tb]},
            "t_item_fixed_s": t_item, "t_per_user_s": t_user, "step_s_full_config_extrapolated": t_full,
            "raw_sample_value": nnz_b / tb,
            "sample": f"dense features + dense U.V^T + autograd + Adam step-1 (oracle/autograd_twin, torch-CPU) timed on {na} and {nb} of "
                      f"{w['n_u']} users x all {n_i} items (median of {n_t} steps each); step(n) = t_item + n t_user solved from the two, "
                      f"full configuration EXTRAPOLATED as t_item + {w['n_u']} t_user = {t_full:.1f} s per epoch"}


def cpu_sparse_step(wl_name, budget_s=12.0, frac=64):
    """The oracle's SPARSE restatement (only the needed dot products, segment-sum gradients: the algorithm the CUDA path
    implements) in NumPy fp32 on a 1/`frac` user sample of the workload, all items; linear in users, so value = sample
    interactions / sample step time (single-threaded NumPy apart from BLAS)."""
    from oracle import mf_oracle as o
    from scipy import sparse
    w = WORKLOADS[wl_name]
    n_i, r, S = w["n_i"], w["r"], w["S"]
    n_sub = max(1, w["n_u"] // frac)
    rng = np.random.default_rng(11)
    rows, cols, vals, samp = _cpu_sample(w, n_sub, rng)
    Xu, Xi = sparse.identity(n_sub, format="csr", dtype=np.float32), sparse.identity(n_i, format="csr", dtype=np.float32)
    state = {"pu": {"W": o.uniform_initializer(n_sub, r, rng)}, "pi": {"W": o.uniform_initializer(n_i, r, rng)}}
    loss = "wmrb" if S else "mse"

    def step():
        _, _, _, state["pu"], state["pi"] = o.train_step_sparse(loss, Xu, Xi, "linear", "linear", state["pu"], state["pi"], rows, cols, vals,
                                                                samp, n_i, S or None, lr=0.1 if S else 1e-2)
    t, n_t = _time_steps(step, budget_s, max_steps=4)
    return {"value": rows.size / t, "unit": "interactions/s", "cores": 1, "kind": "port",
            "sample": f"oracle.train_step_sparse (NumPy fp32) on {n_sub} of {w['n_u']} users x all {n_i} items, {rows.size} interactions, "
                      f"identity features, median of {n_t} steps"}


def cpu_topk(n_i, r, k, n_sub=48, budget_s=12.0):
    """CPU baseline of the retrieval metric: blocked fp32 GEMM (torch-CPU, all cores) + per-block STABLE descending sort
    (ties -> lower item id, like tf.math.top_k) + merge of the per-block lists, on `n_sub` users against all items."""
    cores = _cpu_threads()
    rng = np.random.default_rng(3)
    U = torch.from_numpy((rng.standard_normal((n_sub, r)) / math.sqrt(r)).astype(np.float32))
    V = torch.from_numpy((rng.standard_normal((n_i, r)) / math.sqrt(r)).astype(np.float32))
    blk = 65536

    def run():
        best_s = np.full((n_sub, 0), 0, np.float32); best_i = np.zeros((n_sub, 0), np.int64)
        for b0 in range(0, n_i, blk):
            P = (U @ V[b0:b0 + blk].T).numpy()
            kk = min(k, P.shape[1])
            part = np.argpartition(-P, kk - 1, axis=1)[:, :kk]
            ids = np.concatenate([best_i, part + b0], 1)
            scs = np.concatenate([best_s, np.take_along_axis(P, part, 1)], 1)
            order = np.lexsort((ids, -scs), axis=1)[:, :k]
            best_i, best_s = np.take_along_axis(ids, order, 1), np.take_along_axis(scs, order, 1)
        return best_i
    t, n_t = _time_steps(run, budget_s, max_steps=4)
    return {"value": n_sub * float(n_i) / t, "unit": "pairs/s", "cores": cores, "kind": "port",
            "sample": f"{n_sub} users x all {n_i} items, rank {r}, top-{k}: blocked torch-CPU GEMM ({blk}-item blocks) + per-block partition + "
                      f"(score desc, id asc) merge, median of {n_t} runs"}


# ------------------------------------------------------------------------------------------- main


def _claim_stdout():
    """Everything except the final JSON line goes to stderr: NCCL (and others) print banners on fd 1."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, "w")


def _teardown(world, plans, comm):
    """Leave a multi-rank run without hanging: drop the captured graphs, synchronise, barrier, then destroy the process group from
    a watchdog-guarded thread (round 1's graphs held NCCL work and destroy_process_group() never returned; with the peer-memory
    exchange a captured step holds none, but a stuck teardown must never burn the box's clock)."""
    if world <= 1:
        return
    import gc
    for pl in plans:
        if pl is not None:
            pl.invalidate_graph()
    gc.collect()
    torch.cuda.synchronize()
    torch.distributed.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    done = threading.Event()

    def _destroy():
        try:
            torch.distributed.destroy_process_group()
        finally:
            done.set()
    th = threading.Thread(target=_destroy, daemon=True)
    th.start()
    if not done.wait(20.0):
        log("[bench] destroy_process_group did not return within 20 s; leaving with os._exit(0) (results are already printed)")
        os._exit(0)


def main():
    out_stream = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--topk", default="1000000x1000000x128x100", help="users x items x rank x k of the secondary top-k bench; 'none' skips")
    ap.add_argument("--topk-steps", type=int, default=2)
    ap.add_argument("--c4", default="auto", choices=["auto", "on", "off"], help="also run BASELINE configs[3] (one 10M x 2M problem, strong scaling); "
                    "auto = on for the default c3 workload")
    ap.add_argument("--c4-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--topk-user-sharded", action="store_true", help="also time the user-sharded alternative of the top-k (N > 1)")
    ap.add_argument("--topk-only", action="store_true", help="run only the secondary top-k bench (profiling aid)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed training step (rank 0's shard) "
                    "as DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.topk_only):
        ap.error("--dump-outputs needs the timed training path (--impl ours, no --topk-only)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    w = WORKLOADS[args.workload]
    metric = "training interactions/sec"

    if args.impl == "reference":
        if rank != 0:
            return
        base = cpu_reference_step(args.workload, budget_s=max(20.0, 8.0 * args.steps))
        line = {"impl": "reference", "metric": metric, "value": base["value"], "unit": "interactions/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": w["desc"], "sample": base["sample"], "same_config": base["same_config"],
                           "extrapolated": base["extrapolated"]},
                "cpu_baseline": base,
                "e2e": {"value": base["value"], "unit": "interactions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        if args.topk != "none":
            try:
                tu, ti, tr, tk = (int(x) for x in args.topk.split("x"))
                line["topk"] = {"metric": "top-k scored user-item pairs/sec", "cpu_baseline": cpu_topk(ti, tr, tk)}
                line["topk"]["value"] = line["topk"]["cpu_baseline"]["value"]
                line["topk"]["unit"] = "pairs/s"
            except Exception as e:
                line["topk"] = {"error": f"{type(e).__name__}: {e}"}
        print(json.dumps(line), file=out_stream, flush=True)
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback on the product path)"
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    from teamoflow_b200.mf import dist as tdist
    dev = torch.device("cuda", local)
    hbm_peak, tf_peak, peak_src = peaks()
    t_start = time.time()

    if args.topk_only:
        tu, ti, tr, tk = (int(x) for x in args.topk.split("x"))
        res = bench_topk(tu, ti, tr, tk, args.topk_steps, 1, world, rank, hbm_peak, tf_peak, args.topk_user_sharded)
        if rank == 0:
            print(json.dumps(res), file=out_stream, flush=True)
        _teardown(world, [], None)
        return

    strong = bool(w.get("strong"))
    wl = Workload(args.workload, rank, world, host_copy=not strong)
    w = wl.w  # per-rank sizes (differs from WORKLOADS[...] for strong-scaling workloads)
    comm = None
    if world > 1:
        comm = tdist.GradientSync(shared_user_rows=w["n_u"] if w["mu"] else None)
    xu, xi = wl.feature_args()

    # ---- device-resident measurement: inputs and structures already in HBM
    model = wl.model
    plan, tb = train_bench(wl, comm, args.steps, args.warmup, local, world, hbm_peak, parity_kw=None if args.no_parity else {},
                           dump_dir=args.dump_outputs if rank == 0 else None)
    ms_step = tb["ms_step"]
    total_nnz = wl.total_nnz if strong else world * wl.nnz
    value = total_nnz / (ms_step * 1e-3)
    dom = tb["dom"]
    traffic = None  # DRAM bytes per launch of the dominant kernel, from the committed ncu capture (C3 only)
    traffic_src = None
    for name in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if args.workload == "c3" and os.path.exists(tpath) and traffic is None:
            traffic, traffic_src = json.load(open(tpath)).get(KERNEL_OF[dom]), name

    # ---- end to end through the plugin API from pinned host buffers (one fit call of K epochs)
    e2e = None
    if not args.no_e2e and not strong:
        dts = []
        for _ in range(3):  # three complete fit() calls from the host buffers; the median is reported
            if world > 1:
                torch.distributed.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            model.fit(args.steps, xu, xi, wl.interactions(), lr=wl.lr, comm=comm, verbose=False)
            final_loss = model._plan.ip.mean_loss() if comm is None else comm.mean_loss(model._plan.ip)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            dti = torch.tensor([t1 - t0], device=dev, dtype=torch.float64)
            if world > 1:
                torch.distributed.all_reduce(dti, op=torch.distributed.ReduceOp.MAX)
            dts.append(float(dti))
        dt = sorted(dts)[1]
        e2e = {"value": world * wl.nnz * args.steps / float(dt), "unit": "interactions/s",
               "h2d_bytes_per_step": wl.h2d_bytes() / args.steps, "d2h_bytes_per_step": 4.0 / args.steps,
               "note": f"one MatrixFactorization.fit({args.steps} epochs) from pinned host COO (int32 ids) + host CSR features, incl. H2D, "
                       f"CSR/item-major structure build, weight init, {args.steps} epochs, D2H of the mean loss; "
                       f"median of 3 calls ({', '.join('%.3f' % x for x in dts)} s), final loss {final_loss:.5f}"}

    parity = {}

    def both_stages(init, final):
        return {"ok": bool((init or {}).get("ok") and (final or {}).get("ok")), "init_state_strict": init, "final_state_fp32_budget": final}

    if not args.no_parity:
        try:
            final = parity_train_sample(plan, strict=False)
        except Exception as e:
            import traceback
            log(traceback.format_exc())
            final = {"ok": False, "error": f"{type(e).__name__}: {e}"}
        parity[args.workload] = both_stages(tb["parity_init"], final)
        log(f"[rank {rank}] parity {args.workload}: {parity[args.workload]}")
    out = {"metric": metric, "value": value, "unit": "interactions/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic",
           "config": {"workload": w["desc"], "n_users_per_gpu": w["n_u"], "n_items": w["n_i"], "nnz_per_gpu": wl.nnz, "rank": w["r"],
                      "n_samples": w["S"], "parallelism": f"user-sharded dp{world}" if world > 1 else "single GPU",
                      "grad_exchange": ("tmf_peer_reduce_push over NVLink peer memory (item gradient + staged shared user-side gradients; "
                                        "no NCCL inside the captured step)" if comm.peer else "NCCL all-reduce") if comm is not None else "none",
                      "l2_policy": "working set per step (interactions + lists + embeddings, ~%.1f GB) exceeds the 126 MB L2; no flush" % (
                          (wl.nnz * 28 + w["n_u"] * max(w["S"], 1) * 16) / 1e9),
                      "loss_after": tb["loss"]},
           "roofline": {"bound": "hbm", "kernel": KERNEL_OF[dom], "achieved": tb["dom_gbs"], "peak": hbm_peak, "unit": "GB/s",
                        "frac": tb["dom_gbs"] / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                        "alg_bytes_per_launch": tb["phase_bytes"][dom], "ms_per_launch": tb["phases"][dom],
                        "note": "achieved = SURVEY-8d ALGORITHMIC bytes (every embedding-row gather counted as HBM bytes) / "
                                f"CUDA-event time; `traffic` = DRAM bytes of one launch from the committed ncu capture (profiles/{traffic_src}). "
                                "Where the gathered table fits the 126 MB L2 (C3: 6.9 MB item table) traffic << algorithmic bytes, the "
                                "fraction can exceed 1 and the kernel's real bound is instruction issue + L1/L2 gather latency"},
           "step_roofline": {"alg_bytes_per_step": wl.bytes["total"], "achieved": tb["step_gbs"], "peak": hbm_peak, "unit": "GB/s",
                             "frac": tb["step_gbs"] / hbm_peak},
           "phases_ms": tb["phases"], "clocks": tb["clocks"], "e2e": e2e, "gpu_launches": tb["launches"]}

    if dom == "user_pass":
        try:
            out["roofline"]["gather_rate"] = gather_rate_denominator(plan, tb["dom_gbs"])
        except Exception as e:  # a measurement aid must not take the line down
            out["roofline"]["gather_rate"] = {"error": f"{type(e).__name__}: {e}"}
    plans = [plan, getattr(model, "_plan", None)]
    # ---- BASELINE configs[3]: one 10M x 2M problem, strong scaling over the ranks
    run_c4 = args.c4 == "on" or (args.c4 == "auto" and args.workload == "c3")
    if run_c4:
        try:
            # free the C3 state first (the arena of the gradient exchange is re-sized collectively by attach)
            for pl in plans:
                if pl is not None:
                    pl.invalidate_graph()
            if comm is not None:
                comm.detach(plan)
            del plan, tb
            model._plan = None
            plans = []
            wl.model = None
            torch.cuda.empty_cache()
            t0 = time.time()
            wl4 = Workload("c4", rank, world, host_copy=False)
            balance = None
            if world > 1:
                # measure-and-rebalance: time the rank-local part of a step on the first split, move the boundaries to equal shares
                # of the measured cost (dist.rebalanced_user_bounds), rebuild; at most two passes
                balance = {"rank_ms": []}
                for _ in range(2):
                    xu4, xi4 = wl4.feature_args()
                    pl = wl4.model._prepare(xu4, xi4, wl4.interactions(), comm=None)
                    for _ in range(2):
                        pl.step(wl4.lr)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(3):
                        pl.step(wl4.lr)
                    e1.record(); torch.cuda.synchronize()
                    tl = torch.tensor([e0.elapsed_time(e1) / 3], device=dev, dtype=torch.float64)
                    gl = [torch.zeros_like(tl) for _ in range(world)]
                    torch.distributed.all_gather(gl, tl)
                    times = [float(g) for g in gl]
                    balance["rank_ms"].append([round(x, 3) for x in times])
                    pl.invalidate_graph()
                    del pl
                    wl4.model._plan = None
                    if max(times) <= 1.03 * (sum(times) / world):
                        break
                    nb = tdist.rebalanced_user_bounds(wl4.row_weights, wl4.bounds, times)
                    del wl4
                    torch.cuda.empty_cache()
                    wl4 = Workload("c4", rank, world, host_copy=False, bounds=nb)
                torch.cuda.empty_cache()
            comm4 = tdist.GradientSync() if world > 1 else None
            kw4 = dict(n_us=256, n_is=8, max_len=50_000)
            plan4, t4 = train_bench(wl4, comm4, args.c4_steps, 3, local, world, hbm_peak, parity_kw=None if args.no_parity else kw4)
            plans = [plan4]
            if not args.no_parity:
                try:
                    fin4 = parity_train_sample(plan4, strict=False, **kw4)
                except Exception as e:
                    fin4 = {"ok": False, "error": f"{type(e).__name__}: {e}"}
                parity["c4"] = both_stages(t4["parity_init"], fin4)
                log(f"[rank {rank}] parity c4: {parity['c4']}")
            nnz_r = torch.tensor([wl4.nnz, wl4.w["n_u"]], device=dev, dtype=torch.int64)
            per_rank = [nnz_r.tolist()]
            if world > 1:
                gl = [torch.zeros_like(nnz_r) for _ in range(world)]
                torch.distributed.all_gather(gl, nnz_r)
                per_rank = [g.tolist() for g in gl]
            w4 = WORKLOADS["c4"]
            bytes_total = alg_bytes(w4, wl4.total_nnz, wl4.total_nnz, w4["n_u"], w4["n_i"], 0, 0)["total"]
            out["c4"] = {"metric": metric, "value": wl4.total_nnz / (t4["ms_step"] * 1e-3), "unit": "interactions/s", "ms_per_step": t4["ms_step"],
                         "steps": args.c4_steps, "scaling": "strong", "n_gpus": world,
                         "config": {"workload": w4["desc"], "one_problem": "the same dataset (seed) at every N; contiguous user ranges: first equal "
                                    "(interactions + sampled negatives) per rank (dist.balanced_user_bounds), then boundaries moved to equal shares "
                                    "of the MEASURED rank-local step time (dist.rebalanced_user_bounds, <= 2 passes)",
                                    "balance_passes_rank_ms": balance["rank_ms"] if balance else None,
                                    "users_interactions_per_rank": [{"nnz": a, "users": b} for a, b in per_rank],
                                    "grad_exchange": ("tmf_peer_reduce_push (1.02 GB dE_i: reduce-scatter + Adam + all-gather in one kernel)"
                                                      if comm4.peer else "NCCL all-reduce") if comm4 is not None else "none",
                                    "loss_after": t4["loss"]},
                         "phases_ms": t4["phases"], "gpu_launches": t4["launches"], "clocks": t4["clocks"],
                         "step_roofline": {"bound": "hbm", "alg_bytes_per_step_whole_problem": bytes_total,
                                           "achieved": bytes_total / (t4["ms_step"] * 1e-3) / 1e9 / world, "peak": hbm_peak, "unit": "GB/s per GPU",
                                           "frac": bytes_total / (t4["ms_step"] * 1e-3) / 1e9 / world / hbm_peak,
                                           "note": "SURVEY-8d algorithmic bytes of the WHOLE problem / step time / N, against the measured HBM peak; "
                                                   "the 1 GB item table does not fit L2, so HBM is the real bound here"},
                         "roofline": {"bound": "hbm", "kernel": KERNEL_OF[t4["dom"]], "achieved": t4["dom_gbs"], "peak": hbm_peak, "unit": "GB/s",
                                      "frac": t4["dom_gbs"] / hbm_peak, "alg_bytes_per_launch": t4["phase_bytes"][t4["dom"]],
                                      "ms_per_launch": t4["phases"][t4["dom"]]},
                         "setup_s": time.time() - t0}
            for pl in plans:
                pl.invalidate_graph()
            if comm4 is not None:
                comm4.detach(plan4)
            del plan4, wl4
            plans = []
            torch.cuda.empty_cache()
        except Exception as e:  # keep the primary line alive
            import traceback
            log(traceback.format_exc())
            out["c4"] = {"error": f"{type(e).__name__}: {e}"}

    if args.topk != "none":
        try:
            tu, ti, tr, tk = (int(x) for x in args.topk.split("x"))
            out["topk"] = bench_topk(tu, ti, tr, tk, args.topk_steps, 3, world, rank, hbm_peak, tf_peak, args.topk_user_sharded)
            parity["c5"] = out["topk"].get("parity_check")
        except Exception as e:  # keep the primary line alive
            import traceback
            log(traceback.format_exc())
            out["topk"] = {"error": f"{type(e).__name__}: {e}"}
    # every rank checks its own shard: the reported flag is the AND over the ranks (rank 0's detail is printed, failing ranks are named)
    keys = [args.workload, "c4", "c5"]  # the same on every rank; 2 = this rank did not run that check (skipped, or its section raised)
    flags = torch.tensor([2 if k not in parity else (1 if (parity[k] or {}).get("ok") else 0) for k in keys], dtype=torch.int32, device="cuda")
    allf = flags.reshape(1, -1)
    if world > 1:
        gl = [torch.empty_like(flags) for _ in range(world)]
        torch.distributed.all_gather(gl, flags)
        allf = torch.stack(gl)
    allf = allf.cpu().numpy()
    out["parity_check"], failing = {}, {}
    for j, k in enumerate(keys):
        if (allf[:, j] == 2).all():
            continue  # not run anywhere
        out["parity_check"][k] = "ok" if (allf[:, j] == 1).all() else "FAILED"
        if not (allf[:, j] == 1).all():
            failing[k] = [int(rk) for rk in np.nonzero(allf[:, j] != 1)[0]]
    if failing:
        out["parity_check"]["failing_ranks"] = failing
    out["parity_detail"] = parity

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            out["cpu_baseline"] = cpu_reference_step(args.workload, budget_s=14.0)
        except Exception as e:
            out["cpu_baseline"] = {"error": f"{type(e).__name__}: {e}"}
        try:
            out["cpu_baseline_sparse"] = cpu_sparse_step(args.workload, budget_s=8.0)
        except Exception as e:
            out["cpu_baseline_sparse"] = {"error": f"{type(e).__name__}: {e}"}
        if args.topk != "none" and isinstance(out.get("topk"), dict) and "error" not in out["topk"]:
            try:
                tu, ti, tr, tk = (int(x) for x in args.topk.split("x"))
                out["topk"]["cpu_baseline"] = cpu_topk(ti, tr, tk, budget_s=8.0)
            except Exception as e:
                out["topk"]["cpu_baseline"] = {"error": f"{type(e).__name__}: {e}"}
    out["bench_wall_s"] = time.time() - t_start
    if rank == 0:
        print(json.dumps(out), file=out_stream, flush=True)
        out_stream.flush()
    _teardown(world, plans, comm)


if __name__ == "__main__":
    main()
