"""Cost of the masked fused top-k ("the best k items each user has not seen") against the over-fetch it replaces.

    python scripts/masked_topk_bench.py [--out FILE.json] [--reps N]

Cases (k in {10, 100, 1000} each):
  * ML-20M shape: 138,493 x 26,744, r = 64, a 20M-entry seen table with Zipf row lengths (min 20), in two variants:
    random seen items, and trained-like seen sets (each user's own top-min(len, 1024) items by score, random items for the
    rest), which is what training makes of a user's positives;
  * C5 shape: 1M x 1M, r = 128, with the 50M random positives bench.py uses for recall_at_k.
Per case: the time of score_topk_masked; of score_topk at the same k (the masking overhead); of score_topk at the kc the
earlier recommend() over-fetched (kc = min(n_items, 128 or 1024, k + heaviest row)) together with the number of rows whose
top-kc list held fewer than k unseen items -- rows it sent to its dense canonical fallback (not timed here).  64 sampled rows
of each masked result are checked bit for bit against oracle.canonical_scores with the seen cells at -inf.  Inputs are seeded
N(0, 1/r) embeddings generated on the device; every call is warmed up once, then timed --reps times between CUDA events
(median reported).  Prints one JSON line per case and writes them all, with the GPU's name and power limit, to --out.
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ML20M = (138_493, 26_744, 64)
C5 = (1_000_000, 1_000_000, 128)
KS = (10, 100, 1000)
PAD = 2 ** 31 - 1


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:  # the card's name is still recorded
        info["power_limit"] = f"unavailable ({e})"
    return info


def timed(fn, reps):
    fn()  # warm-up (module load, workspace allocation)
    torch.cuda.synchronize()
    ts, out = [], None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), [round(t, 2) for t in ts], out


def csr_of_keys(keys, n_u, n_i):
    """sorted distinct row-major cell keys u * n_i + i -> (row_ptr int32, col_idx int32) on the device"""
    keys = torch.unique(keys)
    rows = keys // n_i
    ptr = torch.zeros(n_u + 1, dtype=torch.int64, device=keys.device)
    ptr[1:] = torch.cumsum(torch.bincount(rows, minlength=n_u), 0)
    return ptr.to(torch.int32), (keys % n_i).to(torch.int32)


def zipf_lengths(n_u, n_i, total, g):
    rank = torch.randperm(n_u, generator=g, device="cuda").double() + 1.0
    w = rank ** -0.9
    lens = (w / w.sum() * (total - 20 * n_u)).floor().long() + 20
    return lens.clamp(max=n_i)


def random_keys(lens, n_i, g):
    users = torch.repeat_interleave(torch.arange(lens.numel(), device="cuda"), lens)
    return users * n_i + torch.randint(0, n_i, (users.numel(),), generator=g, device="cuda")


def masked_scores(U, V, r, rows, ptr, idx):
    """canonical scores of the sampled rows, seen cells at -inf"""
    from oracle import mf_oracle as o
    P = o.canonical_scores(U[torch.as_tensor(rows, device="cuda"), :r].cpu().numpy(), V[:, :r].cpu().numpy()).astype(np.float32)
    p, ix = ptr.cpu().numpy(), idx.cpu().numpy()
    for j, u in enumerate(rows):
        P[j, ix[p[u]:p[u + 1]]] = -np.inf
    return P


def oracle_rows(P, k):
    """oracle.topk_stable of each row of P restricted to the entries at or above its k-th largest score (the same answer; a
    full stable sort of 1M-item rows would dominate the run), padded past the row's finite entries"""
    from oracle import mf_oracle as o
    widx = np.full((P.shape[0], k), PAD, np.int32)
    wsc = np.full((P.shape[0], k), -np.inf, np.float32)
    for j in range(P.shape[0]):
        n_unseen = int(np.isfinite(P[j]).sum())
        kk = min(k, n_unseen)
        if kk == 0:
            continue
        kth = -np.partition(-P[j], kk - 1)[kk - 1]
        cand = np.nonzero(P[j] >= kth)[0]  # ascending ids
        sel = cand[o.topk_stable(P[j, cand], kk)]
        widx[j, :kk], wsc[j, :kk] = sel, P[j, sel]
    return widx, wsc


def run_case(name, U, V, r, ptr, idx, reps, results):
    from teamoflow_b200 import _abi
    from teamoflow_b200.mf.evaluation import score_topk_masked
    from teamoflow_b200.mf.matrix_factorization import score_topk
    n_u, n_i = U.shape[0], V.shape[0]
    row_nnz = ptr[1:] - ptr[:-1]
    heaviest = int(row_nnz.max())
    rows = np.sort(np.random.default_rng(7).choice(n_u, 64, replace=False))
    P_rows = masked_scores(U, V, r, rows, ptr, idx)
    ones = torch.ones(idx.numel(), dtype=torch.float32, device="cuda")
    for k in KS:
        t_m, ts_m, (mi, ms) = timed(lambda: score_topk_masked(U, V, r, k, False, ptr, idx), reps)
        widx, wsc = oracle_rows(P_rows, k)
        ok = bool(np.array_equal(mi[rows].cpu().numpy(), widx) and np.array_equal(ms[rows].cpu().numpy(), wsc))
        del mi, ms
        t_p, ts_p, _ = timed(lambda: score_topk(U, V, r, k, False), reps)
        kc = min(n_i, 128 if k <= 128 else 1024, k + heaviest)
        t_c, ts_c, (ci, _) = timed(lambda: score_topk(U, V, r, kc, False), reps)
        seen_in_list = torch.empty(n_u, dtype=torch.float32, device="cuda")
        relevant = torch.empty(n_u, dtype=torch.float32, device="cuda")
        _abi.call("tmf_metrics_hits", _abi.ptr(ci), n_u, kc, _abi.ptr(ptr), _abi.ptr(idx), _abi.ptr(ones), _abi.ptr(seen_in_list),
                  _abi.ptr(relevant))
        dense_rows = int((seen_in_list > kc - k).sum())
        del ci
        rec = {"case": name, "n_users": n_u, "n_items": n_i, "r": r, "k": k, "seen_entries": int(idx.numel()),
               "heaviest_row": heaviest, "masked_ms": round(t_m, 2), "masked_ms_all": ts_m, "plain_ms": round(t_p, 2),
               "plain_ms_all": ts_p, "masking_overhead": round(t_m / t_p - 1.0, 4), "overfetch_kc": kc,
               "overfetch_ms": round(t_c, 2), "overfetch_ms_all": ts_c, "overfetch_dense_rows": dense_rows,
               "oracle_rows_checked": int(rows.size), "bit_exact": ok}
        print(json.dumps(rec), flush=True)
        results.append(rec)
        torch.cuda.empty_cache()


def embeddings(n_u, n_i, r, seed):
    from teamoflow_b200.mf._engine import new_storage
    g = torch.Generator(device="cuda"); g.manual_seed(seed)
    U = new_storage(n_u, r); U[:, :r] = torch.randn(n_u, r, generator=g, device="cuda") / math.sqrt(r)
    V = new_storage(n_i, r); V[:, :r] = torch.randn(n_i, r, generator=g, device="cuda") / math.sqrt(r)
    return U, V


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None, help="JSON file for all results")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("masked_topk_bench.py needs a CUDA device")
    from teamoflow_b200.mf.matrix_factorization import score_topk
    info = gpu_info()
    print(json.dumps({"gpu": info}), flush=True)
    results = []

    n_u, n_i, r = ML20M
    U, V = embeddings(n_u, n_i, r, 20245)
    g = torch.Generator(device="cuda"); g.manual_seed(11)
    lens = zipf_lengths(n_u, n_i, 20_000_000, g)
    ptr, idx = csr_of_keys(random_keys(lens, n_i, g), n_u, n_i)
    run_case("ml20m_random_seen", U, V, r, ptr, idx, args.reps, results)
    top, _ = score_topk(U, V, r, 1024, False)  # each user's own best items
    n_top = lens.clamp(max=1024)
    keep = torch.arange(1024, device="cuda")[None, :] < n_top[:, None]
    users = torch.arange(n_u, device="cuda")[:, None].expand(-1, 1024)
    top_keys = users[keep] * n_i + top[keep].long()
    rest_keys = random_keys(lens - n_top, n_i, g)
    del top, keep, users
    ptr, idx = csr_of_keys(torch.cat([top_keys, rest_keys]), n_u, n_i)
    del top_keys, rest_keys
    run_case("ml20m_trained_like_seen", U, V, r, ptr, idx, args.reps, results)
    del U, V, ptr, idx
    torch.cuda.empty_cache()

    n_u, n_i, r = C5
    U, V = embeddings(n_u, n_i, r, 20245)
    ga = torch.Generator(device="cuda"); ga.manual_seed(777)
    keys = torch.randint(0, n_u * n_i, (min(50 * n_u, 50_000_000),), generator=ga, device="cuda", dtype=torch.int64)
    ptr, idx = csr_of_keys(keys, n_u, n_i)
    del keys
    run_case("c5_bench_positives", U, V, r, ptr, idx, args.reps, results)

    out = {"gpu": info, "reps": args.reps,
           "timing": "CUDA events around one call (pack + main + rerank + exact path); the dense fallback of the over-fetch is "
                     "not timed, only its rows counted",
           "cases": results, "all_bit_exact": all(c["bit_exact"] for c in results)}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    if not out["all_bit_exact"]:
        raise SystemExit("oracle mismatch")


if __name__ == "__main__":
    main()
