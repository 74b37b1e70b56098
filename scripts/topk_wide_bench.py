"""Cost of the fused top-k across k, including the wide configuration (128 < k <= 1024).

    python scripts/topk_wide_bench.py [--out FILE.json] [--reps N]

Times `score_topk` on the C5 shape (1M x 1M, r = 128, k in {100, 128, 256, 512, 1024}, raw and clamp) and the ML-20M shape
(138,493 x 26,744, r = 64, k in {100, 500, 1000}, raw).  Inputs are seeded N(0, 1/r) embeddings generated on the device; every
case is warmed up once, then timed `--reps` times between CUDA events (median reported).  Per case: time, pairs/s, the
tensor-pipe fraction 2 n_u n_i r / t / 1386.5e12 (the sustained bf16 peak DESIGN uses), and the rerank's compulsory item-row
bytes n_u k 4 r (its floor once the item table is larger than L2).  64 sampled rows of each case are checked bit for bit
against oracle.canonical_scores of those rows.  Prints one JSON line per case and writes them all, with the GPU's name and
power limit, to --out.
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

SUSTAINED_BF16 = 1386.5e12
C5 = (1_000_000, 1_000_000, 128, [100, 128, 256, 512, 1024], (False, True))
ML20M = (138_493, 26_744, 64, [100, 500, 1000], (False,))


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:  # the card's name is still recorded
        info["power_limit"] = f"unavailable ({e})"
    return info


def oracle_topk(P, k, clamp):
    """oracle.topk_stable of the canonical score rows P (ties -> lower id), restricted per row to the entries at or above the
    k-th largest score (the same answer; a full stable sort of 1M-item rows would dominate the run)"""
    from oracle import mf_oracle as o
    if clamp:
        P = np.where(P > 0, P, np.float32(0))
    idx = np.empty((P.shape[0], k), np.int32)
    for j in range(P.shape[0]):
        kth = -np.partition(-P[j], k - 1)[k - 1]
        cand = np.nonzero(P[j] >= kth)[0]  # ascending ids
        idx[j] = cand[o.topk_stable(P[j, cand], k)]
    return idx, np.take_along_axis(P, idx.astype(np.int64), 1)


def run_shape(n_u, n_i, r, ks, modes, reps, results):
    from teamoflow_b200.mf._engine import new_storage
    from teamoflow_b200.mf.matrix_factorization import score_topk
    g = torch.Generator(device="cuda"); g.manual_seed(20245)
    U = new_storage(n_u, r); U[:, :r] = torch.randn(n_u, r, generator=g, device="cuda") / math.sqrt(r)
    V = new_storage(n_i, r); V[:, :r] = torch.randn(n_i, r, generator=g, device="cuda") / math.sqrt(r)
    from oracle import mf_oracle as o
    rows = np.sort(np.random.default_rng(7).choice(n_u, 64, replace=False))
    P_rows = o.canonical_scores(U[torch.as_tensor(rows, device="cuda"), :r].cpu().numpy(), V[:, :r].cpu().numpy())
    for k in ks:
        for clamp in modes:
            score_topk(U, V, r, k, clamp)  # warm-up (module load, workspace allocation)
            torch.cuda.synchronize()
            ts = []
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                idx, sc = score_topk(U, V, r, k, clamp)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1) / 1e3)
            t = float(np.median(ts))
            widx, wsc = oracle_topk(P_rows, k, clamp)
            ok = bool(np.array_equal(idx[rows].cpu().numpy(), widx) and np.array_equal(sc[rows].cpu().numpy(), wsc))
            del idx, sc
            rec = {"n_users": n_u, "n_items": n_i, "r": r, "k": k, "clamp": clamp, "ms": round(t * 1e3, 2),
                   "ms_all": [round(x * 1e3, 2) for x in ts], "pairs_per_s": n_u * n_i / t,
                   "tensor_pipe_fraction": round(2.0 * n_u * n_i * r / t / SUSTAINED_BF16, 4),
                   "rerank_item_row_bytes": n_u * k * 4 * r, "oracle_rows_checked": int(rows.size), "bit_exact": ok}
            print(json.dumps(rec), flush=True)
            results.append(rec)
    del U, V
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None, help="JSON file for all results")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("topk_wide_bench.py needs a CUDA device")
    info = gpu_info()
    print(json.dumps({"gpu": info}), flush=True)
    results = []
    for shape in (C5, ML20M):
        run_shape(*shape, args.reps, results)
    out = {"gpu": info, "reps": args.reps, "timing": "CUDA events around one score_topk call (pack + main + rerank + exact path)",
           "cases": results, "all_bit_exact": all(c["bit_exact"] for c in results)}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    if not out["all_bit_exact"]:
        raise SystemExit("oracle mismatch")


if __name__ == "__main__":
    main()
