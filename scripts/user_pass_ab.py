"""A/B of the training user pass between two libtmf.so builds, on one GPU.

    python scripts/user_pass_ab.py LIB_A LIB_B [--workloads c3 c4mini] [--rounds 5] [--calls 10] [--no-variants] [--out F]

First, on every case of tests/test_gpu_train_variants.py (all 27 kernel instantiations, with and without split users
and a coefficient slot map) but with normally distributed embeddings, so that a changed summation order would change
bits, it compares the two builds' outputs byte for byte.  Then, for each bench.py workload, it builds the training plan
once (same inputs, same initial weights), runs tmf_user_pass (and the fix-up of split users) from each build, compares
loss_out, coef_out, dE_u, part_G and part_E byte for byte, and times the two builds alternately: each round is `--calls`
back-to-back calls of A, then of B, between CUDA events.  Prints one JSON line per check (and writes them to --out);
exits 1 if any output differs."""
import argparse
import ctypes
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from teamoflow_b200 import _abi  # noqa: E402


def load(path):
    """a ctypes handle of the build at `path`, with the signatures _abi gives its own"""
    h = ctypes.CDLL(os.path.abspath(path))
    for name, (res, args) in _abi.SIGNATURES.items():
        fn = getattr(h, name)
        fn.restype, fn.argtypes = res, args
    assert h.tmf_abi_version() == 1, path
    return h


def outputs(ip, dEu):
    ts = {"loss_out": ip.loss_k, "coef_out": ip.coef, "dEu": dEu}
    if ip.n_split:
        ts.update(part_G=ip.part_G, part_E=ip.part_E)
    return {k: t.detach().clone() for k, t in ts.items()}


def variants(libs):
    """(cases, runs, names of the cases whose outputs differ) over the user-pass cases of the variant tests"""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_gpu_train_variants as tv
    bad, runs = [], 0
    for case in tv.UP_CASES:
        pb = dict(tv.user_problem(*case))
        rng = np.random.default_rng(11)
        r = pb["r"]
        for k in ("Eu", "Ei"):
            x = np.zeros_like(pb[k])
            x[:, :r] = rng.standard_normal((x.shape[0], r)) / r ** 0.25
            pb[k] = x
        up = tv.UserPassRun(pb)
        perm = rng.permutation(up.T).astype(np.int32)
        for items in (None, up.items):
            for coef_pos in (None, perm):
                got = {}
                for which in ("a", "b"):
                    _abi._lib = libs[which]
                    got[which] = up.run(items, coef_pos)
                runs += 1
                if not all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(got["a"], got["b"])):
                    bad.append(f"{tv._up_id(case)} items={'split' if items is not None else 'none'} "
                               f"coef_pos={'perm' if coef_pos is not None else 'none'}")
    return len(tv.UP_CASES), runs, bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("lib_a")
    ap.add_argument("lib_b")
    ap.add_argument("--workloads", nargs="+", default=["c3", "c4mini"])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--out")
    args = ap.parse_args()
    libs = {"a": load(args.lib_a), "b": load(args.lib_b)}
    props = torch.cuda.get_device_properties(0)
    lines = []
    if not args.no_variants:
        n_cases, runs, bad = variants(libs)
        line = {"variants": n_cases, "runs": runs, "differ": bad, "all_same": not bad}
        print(json.dumps(line), flush=True)
        lines.append(line)
    for name in args.workloads:
        wl = bench.Workload(name, 0, 1, host_copy=False)
        _abi._lib = libs["a"]
        xu, xi = wl.feature_args()
        plan = wl.model._prepare(xu, xi, wl.interactions(), comm=None)
        Eu, Ei = plan.u.forward(), plan.i.forward()
        dEu = torch.empty_like(Eu)
        ip = plan.ip

        def run(which, n=1):
            _abi._lib = libs[which]
            for _ in range(n):
                ip.user_pass(Eu, Ei, plan.r, dEu)

        res = {}
        for which in ("a", "b"):
            for t in (ip.loss_k, ip.coef, dEu):
                t.fill_(float("nan"))
            run(which)
            torch.cuda.synchronize()
            res[which] = outputs(ip, dEu)
        same = {k: bool(torch.equal(res["a"][k].view(torch.int32), res["b"][k].view(torch.int32))) for k in res["a"]}
        run("a", 3)
        run("b", 3)
        ms = {"a": [], "b": []}
        for _ in range(args.rounds):
            for which in ("a", "b"):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(which, args.calls)
                e1.record()
                torch.cuda.synchronize()
                ms[which].append(e0.elapsed_time(e1) / args.calls)
        med = {k: statistics.median(v) for k, v in ms.items()}
        line = {"workload": name, "gpu": props.name, "same_bits": same, "all_same": all(same.values()),
                "ms_a": [round(x, 4) for x in ms["a"]], "ms_b": [round(x, 4) for x in ms["b"]],
                "median_a": round(med["a"], 4), "median_b": round(med["b"], 4),
                "b_over_a": round(med["b"] / med["a"], 4), "lib_a": args.lib_a, "lib_b": args.lib_b}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del plan, ip, Eu, Ei, dEu, res, wl
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")
    return 0 if all(x["all_same"] for x in lines) else 1


if __name__ == "__main__":
    sys.exit(main())
