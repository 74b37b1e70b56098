"""The fused top-k past its first user batch: plain, masked and bounded scoring at shapes that need several main-kernel
and rerank launches, every row against an fp64 reference, indices and scores bit for bit.

score_topk_impl ranks the users in batches of UB_BATCH (k <= 128) or UB_BATCH_W (128 < k <= 1024) blocks of 128 rows; inside
a batch the candidate lists, counts and thresholds use the batch-local row and everything else (U, the error bounds, the
exclusion cursors, the row bounds, the overflow rows, the outputs) the global row.  exact_rows_kernel runs once, after the
last batch, over the overflow rows of every batch.  test_topk_batches_cpu.py checks that the shapes here straddle the batches.

Special rows sit at the first rows of batch 1, its last row, the first row of batch 2, the middle of the last batch and the
very last row:
  zero rows      every score 0: the list cannot shrink and the main kernel hands the row to exact_rows_kernel;
  grid rows      scores a/64 and 0 only, with more items tied at the top than the rerank can rank: the exact path again;
  non-positive   every score < 0: in clamp mode the answer is the k lowest ids (the filler rule).
The reference is torch fp64 on the device, anchored to the NumPy oracle on a small shape.  The outputs are filled with -7 and
NaN before every call, so a row that no launch writes cannot keep a correct answer from an earlier call, and a 4 KB canary
after the workspace must survive every call.
"""
import collections
import functools

import numpy as np
import pytest
import torch

from oracle import mf_oracle as o
from test_topk_batches_cpu import (BATCH_USERS, BATCH_USERS_W, BOUNDED, FAMILIES, INVARIANCE, LAUNCHES, MASKED, PLAIN,
                                   n_batches, straddles)

pytestmark = pytest.mark.gpu

DEV = "cuda"
PAD = 2 ** 31 - 1
SEL_CAP, SEL_CAP_W = 512, 2048  # survivors per row the rerank ranks (score_topk.cu); more go to exact_rows_kernel
KINDS = ("zero", "grid", "nonpos", "random")
CANARY = 4096


def _abi():
    from teamoflow_b200 import _abi
    return _abi


# ------------------------------------------------------------------------------- fp64 reference


def reference_topk(U, V, k, clamp, ex=None):
    """Top-k of every row of U [n_u, r] against V [n_i, r] (fp32, on the device) by (canonical score desc, id asc).

    The canonical score is fp32(fma chain in fp64 over the components in order): a product of two fp32 values is exact in
    fp64, so acc + u * v per component equals the fused chain bit for bit.  Clamp mode ranks where(P > 0, P, 0).  ``ex``:
    CSR (ptr, idx) of the item ids excluded per row (sorted, distinct); they score -inf after the clamp and rows with fewer
    than k unseen items end in (PAD, -inf).  Calls no tmf_* entry point."""
    n_u, r = U.shape
    n_i = V.shape[0]
    V64T = V.double().t().contiguous()
    out_i = torch.empty(n_u, k, dtype=torch.int32, device=U.device)
    out_s = torch.empty(n_u, k, dtype=torch.float32, device=U.device)
    chunk = max(1, min(n_u, (1 << 26) // n_i))
    for a in range(0, n_u, chunk):
        b = min(n_u, a + chunk)
        U64 = U[a:b].double()
        acc = torch.zeros(b - a, n_i, dtype=torch.float64, device=U.device)
        for c in range(r):
            acc.addcmul_(U64[:, c:c + 1], V64T[c])
        P = acc.float()
        del acc
        if clamp:
            P = torch.where(P > 0, P, torch.zeros_like(P))
        if ex is not None:
            ptr, idx = ex
            lens = (ptr[a + 1:b + 1] - ptr[a:b]).long()
            rows = torch.repeat_interleave(torch.arange(b - a, device=U.device), lens)
            P[rows, idx[int(ptr[a]):int(ptr[b])].long()] = float("-inf")
        s, i = torch.sort(P, dim=1, descending=True, stable=True)
        s, i = s[:, :k], i[:, :k].int()
        if ex is not None:
            pad = torch.arange(k, device=U.device)[None, :] >= (n_i - lens)[:, None]
            i = torch.where(pad, torch.full_like(i, PAD), i)
            s = torch.where(pad, torch.full_like(s, float("-inf")), s)
        out_i[a:b], out_s[a:b] = i, s
    return out_i, out_s


# ------------------------------------------------------------------------------- data


def special_rows(n, starts, ends):
    """{row: kind}: KINDS in order from each start row, and in reverse order up to each end row (so the row before an end
    is a zero row)"""
    kind = {}
    for a in starts:
        for j, kd in enumerate(KINDS):
            if a + j < n:
                kind[a + j] = kd
    for e in ends:
        for j, kd in enumerate(KINDS):
            if 0 <= e - 1 - j < n:
                kind[e - 1 - j] = kd
    return kind


def make_data(n_u, n_i, r, kind, seed):
    """U, V (fp32 on the device).  V: column 0 is 0 or 1/8 (about half each), column 1 positive, the rest N(0, 1/r).
    Rows of U: N(0, 1/r) except the special rows of ``kind``: zero; grid (a/8, 0, ..., 0), whose scores are a/64 for about
    n_i / 2 items and 0 for the rest; non-positive (0, -c, 0, ..., 0), every score < 0."""
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    U = torch.randn(n_u, r, generator=g, device=DEV) / r ** 0.5
    V = torch.randn(n_i, r, generator=g, device=DEV) / r ** 0.5
    V[:, 0] = (torch.rand(n_i, generator=g, device=DEV) < 0.5).float() * 0.125
    V[:, 1] = V[:, 1].abs() + 0.05
    for kd in ("zero", "grid", "nonpos"):
        rows = torch.tensor([x for x, v in kind.items() if v == kd], dtype=torch.long, device=DEV)
        U[rows] = 0.0
        if kd == "grid":
            U[rows, 0] = (rows % 4 + 1).float() / 8
        elif kd == "nonpos":
            U[rows, 1] = -(0.5 + (rows % 5).float() / 10)
    return U.contiguous(), V.contiguous()


# family -> (start anchors, end anchors): the first rows of batch 1, the last row of batch 1, the first row of each later
# batch, the middle of the last batch, the very last row; the prefix cases' last rows are anchors too
B, BW = BATCH_USERS, BATCH_USERS_W
ANCHORS = {
    "narrow": ([0, B, B + 100], [B, FAMILIES["narrow"]["n_users"]]),
    "narrow3": ([0, B, 2 * B, 2 * B + 500], [B, 2 * B, FAMILIES["narrow3"]["n_users"]]),
    "wide": ([0, BW, BW + 2112], [BW, FAMILIES["wide"]["n_users"]]),
    "ml20m": ([0, BW, BW + 31358], [BW, FAMILIES["ml20m"]["n_users"]]),
}
# the reference is computed once per family, clamp mode and mask at this k and sliced for smaller k
REF_K = {"narrow": 128, "narrow3": 10, "wide": 300, "ml20m": 1024}


@functools.lru_cache(maxsize=None)
def family(name):
    shape = FAMILIES[name]
    starts, ends = ANCHORS[name]
    kind = special_rows(shape["n_users"], starts, ends)
    U, V = make_data(shape["n_users"], shape["n_items"], shape["r"], kind, seed=len(name) * 7919 + shape["n_items"])
    return U, V, kind


@functools.lru_cache(maxsize=None)
def reference(name, clamp, masked=False):
    U, V, _ = family(name)
    return reference_topk(U, V, REF_K[name], clamp, exclusion(name) if masked else None)


@pytest.fixture(scope="module", autouse=True)
def _release_cached_data():
    """the data sets and references are cached across the tests of this module and released after its last test"""
    yield
    for f in (family, reference, exclusion):
        f.cache_clear()
    torch.cuda.empty_cache()


# masked families: how many items the rows planted with "fewer than k unseen items" keep unseen (< every k used)
N_FEW = {"narrow": 37, "ml20m": 150}


@functools.lru_cache(maxsize=None)
def exclusion(name):
    """Per-row exclusion CSR (int32, on the device), random lengths 0..100, sorted and distinct.  Special rows: zero rows
    get a non-empty list (exact_rows_kernel reads ex_ptr[row]); grid rows all but N_FEW items (padding, and in clamp mode
    clamp_fill_kernel); non-positive rows an empty list; the random rows next to them their own best 400 items."""
    U, V, kind = family(name)
    n_u, n_i = U.shape[0], V.shape[0]
    g = torch.Generator(device=DEV)
    g.manual_seed(n_u)
    lens = torch.randint(0, 101, (n_u,), generator=g, device=DEV)
    special = torch.tensor(sorted(kind), dtype=torch.long, device=DEV)
    lens[special] = 0
    rows = torch.repeat_interleave(torch.arange(n_u, device=DEV), lens)
    keys = [rows * n_i + torch.randint(0, n_i, (rows.numel(),), generator=g, device=DEV)]
    by_kind = collections.defaultdict(list)
    for x, kd in kind.items():
        by_kind[kd].append(x)
    for x in by_kind["zero"]:
        keys.append(x * n_i + torch.randperm(n_i, generator=g, device=DEV)[:50])
    for x in by_kind["grid"]:
        keys.append(x * n_i + torch.randperm(n_i, generator=g, device=DEV)[N_FEW[name]:])
    top = reference_topk(U[by_kind["random"]], V, 400, False)[0].long()
    for j, x in enumerate(by_kind["random"]):
        keys.append(x * n_i + top[j])
    keys = torch.unique(torch.cat(keys))  # sorted: by row, then id; duplicates of the random lists merge
    counts = torch.bincount(keys // n_i, minlength=n_u)
    ptr = torch.zeros(n_u + 1, dtype=torch.int32, device=DEV)
    ptr[1:] = torch.cumsum(counts, 0).int()
    return ptr, (keys % n_i).int().contiguous()


def sub_csr(ex, a, b):
    """the CSR of rows [a, b)"""
    ptr, idx = ex
    return (ptr[a:b + 1] - ptr[a]).contiguous(), idx[int(ptr[a]):int(ptr[b])].contiguous()


# ------------------------------------------------------------------------------- calls through the C ABI


def run_topk(U, V, k, clamp, item_offset=0, ex=None, row_bound=None):
    """One tmf_score_topk / _masked / _bounded call on outputs filled with -7 / NaN and a workspace followed by a canary"""
    A = _abi()
    n_u, r = U.shape
    n_i = V.shape[0]
    need = A.query("tmf_score_topk_ws_bytes", n_u, n_i, r, k)
    ws = torch.empty(need + CANARY, dtype=torch.uint8, device=DEV)
    canary = torch.arange(CANARY, device=DEV).remainder(251).add(1).to(torch.uint8)
    ws[need:] = canary
    idx = torch.full((n_u, k), -7, dtype=torch.int32, device=DEV)
    sc = torch.full((n_u, k), float("nan"), dtype=torch.float32, device=DEV)
    head = (A.ptr(U), n_u, A.ptr(V), n_i, r, r, k, int(clamp), int(item_offset))
    tail = (A.ptr(idx), A.ptr(sc), A.ptr(ws), need)
    if ex is not None:
        A.call("tmf_score_topk_masked", *head, A.ptr(ex[0]), A.ptr(ex[1]), *tail)
    elif row_bound is not None:
        A.call("tmf_score_topk_bounded", *head, A.ptr(row_bound), *tail)
    else:
        A.call("tmf_score_topk", *head, *tail)
    torch.cuda.synchronize()
    assert torch.equal(ws[need:], canary), "tmf_score_topk wrote past its workspace"
    return idx, sc


def assert_same(got, want, what, clamp=False):
    """indices and score bits equal in every row; in clamp mode no -0 score"""
    gi, gs = got
    wi, ws = want
    assert gi.shape == wi.shape, f"{what}: shape {tuple(gi.shape)}, want {tuple(wi.shape)}"
    bad = (gi != wi).any(1) | (gs.view(torch.int32) != ws.view(torch.int32)).any(1)
    if bool(bad.any()):
        rows = bad.nonzero().flatten()
        r0 = int(rows[0])
        raise AssertionError(f"{what}: {rows.numel()} of {gi.shape[0]} rows differ, first {rows[:6].tolist()}, last "
                             f"{int(rows[-1])}; row {r0}: got {gi[r0, :4].tolist()} {gs[r0, :4].tolist()}, want "
                             f"{wi[r0, :4].tolist()} {ws[r0, :4].tolist()}")
    if clamp:
        assert not bool((torch.signbit(gs) & (gs == 0)).any()), f"{what}: a clamped zero score has its sign bit set"


def check_specials(got, name, n, k, clamp):
    """what the special rows must hold, independent of the reference"""
    _, V, kind = family(name)
    gi, gs = got
    n_top = int((V[:, 0] > 0).sum())
    for x, kd in kind.items():
        if x >= n:
            continue
        if kd == "zero":  # every score 0: the k lowest ids
            assert torch.equal(gi[x].cpu(), torch.arange(k, dtype=torch.int32)) and not bool(gs[x].any()), f"zero row {x}"
        elif kd == "nonpos" and clamp:
            assert torch.equal(gi[x].cpu(), torch.arange(k, dtype=torch.int32)) and not bool(gs[x].any()), f"row {x}"
        elif kd == "grid":
            assert bool((gs[x] > 0).all()), f"grid row {x}: the top group holds {n_top} items"


# ------------------------------------------------------------------------------- the reference against the oracle


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("clamp", [False, True])
def test_reference_matches_the_cpu_oracle(clamp, masked):
    from test_gpu_topk_masked import oracle_masked
    from test_gpu_score import oracle_topk
    n_u, n_i, r, k = 300, 5000, 24, 200
    kind = special_rows(n_u, [0, 128], [128, n_u])
    U, V = make_data(n_u, n_i, r, kind, seed=11)
    Un, Vn = U.cpu().numpy(), V.cpu().numpy()
    if masked:
        g = torch.Generator(device=DEV)
        g.manual_seed(5)
        mask = torch.rand(n_u, n_i, generator=g, device=DEV) < 0.05
        mask[1, 3:] = True   # a grid row with 3 unseen items
        mask[2] = False      # a non-positive row with nothing seen
        ptr = torch.zeros(n_u + 1, dtype=torch.int32, device=DEV)
        ptr[1:] = torch.cumsum(mask.sum(1), 0).int()
        idx = mask.nonzero()[:, 1].int().contiguous()
        got = reference_topk(U, V, k, clamp, (ptr, idx))
        want = oracle_masked(Un, Vn, k, clamp, ptr.cpu().numpy(), idx.cpu().numpy())
    else:
        got = reference_topk(U, V, k, clamp)
        want = oracle_topk(Un, Vn, k, clamp)
    assert np.array_equal(got[0].cpu().numpy(), want[0])
    assert np.array_equal(got[1].cpu().numpy().view(np.uint32), np.asarray(want[1], np.float32).view(np.uint32))
    assert (o.canonical_scores(Un[[1]], Vn) == Un[1, 0] * Vn[:, 0]).all()  # grid scores are exact


# ------------------------------------------------------------------------------- plain top-k


@pytest.mark.parametrize("name,n,k,clamp", PLAIN, ids=[f"{a}-{n}-k{k}-{'clamp' if c else 'raw'}" for a, n, k, c in PLAIN])
def test_plain_topk_across_batches(name, n, k, clamp):
    assert straddles(n, k)
    U, V, _ = family(name)
    n_top = int((V[:, 0] > 0).sum())
    if V.shape[0] >= 2000:  # the grid rows' top tie group is more than the rerank can rank
        assert n_top > (SEL_CAP if k <= 128 else SEL_CAP_W)
    got = run_topk(U[:n], V, k, clamp)
    ri, rs = reference(name, clamp)
    assert_same(got, (ri[:n, :k], rs[:n, :k]), f"{name} n={n} k={k} clamp={clamp}", clamp)
    check_specials(got, name, n, k, clamp)


# ------------------------------------------------------------------------------- masked top-k


@pytest.mark.parametrize("name,n,k,clamp", MASKED, ids=[f"{a}-{n}-k{k}-{'clamp' if c else 'raw'}" for a, n, k, c in MASKED])
def test_masked_topk_across_batches(name, n, k, clamp):
    assert straddles(n, k)
    U, V, kind = family(name)
    assert n == U.shape[0]
    got = run_topk(U, V, k, clamp, ex=exclusion(name))
    ri, rs = reference(name, clamp, masked=True)
    assert_same(got, (ri[:, :k], rs[:, :k]), f"masked {name} k={k} clamp={clamp}", clamp)
    gi = got[0]
    for x, kd in kind.items():
        if kd == "grid":  # N_FEW unseen items, then padding
            assert bool((gi[x, N_FEW[name]:] == PAD).all()) and bool((gi[x, :N_FEW[name]] != PAD).all()), f"row {x}"


# ------------------------------------------------------------------------------- bounded item slabs


@pytest.mark.parametrize("name,n,k,bounds,clamp", BOUNDED,
                         ids=[f"{a}-{n}-k{k}-{'clamp' if c else 'raw'}" for a, n, k, _, c in BOUNDED])
def test_bounded_slabs_across_batches(name, n, k, bounds, clamp):
    """The protocol of dist.sharded_topk with the ranks played one after the other: a bound pass per (user slice, slab), a
    bounded pass per slab with item_offset, tmf_topk_merge."""
    from teamoflow_b200.mf import dist as tdist
    assert straddles(n, k)
    A = _abi()
    U, V, _ = family(name)
    U = U[:n]
    r = U.shape[1]
    G = len(bounds) - 1
    ub = tdist.shard_bounds(n, G)
    slabs = [V[a:b] for a, b in zip(bounds[:-1], bounds[1:])]
    rb = torch.cat([tdist.topk_row_bounds(U, slabs[g], r, k, clamp, bounds[g], ub[g], ub[g + 1], slabs[g].shape[0])
                    for g in range(G)]).contiguous()
    lists = [run_topk(U, slabs[g], k, clamp, item_offset=bounds[g], row_bound=rb) for g in range(G)]
    idx_in = torch.stack([x[0] for x in lists]).contiguous()
    sc_in = torch.stack([x[1] for x in lists]).contiguous()
    out_i = torch.full((n, k), -7, dtype=torch.int32, device=DEV)
    out_s = torch.full((n, k), float("nan"), dtype=torch.float32, device=DEV)
    A.call("tmf_topk_merge", A.ptr(idx_in), A.ptr(sc_in), G, n, k, A.ptr(out_i), A.ptr(out_s))
    torch.cuda.synchronize()
    ri, rs = reference(name, clamp)
    want = (ri[:n, :k], rs[:n, :k])
    assert_same((out_i, out_s), want, f"bounded {name} n={n} k={k} clamp={clamp}", clamp)
    assert bool((rb <= want[1][:, k - 1]).all()), "a row bound exceeds the row's k-th best score"
    assert bool((rb > float("-inf")).all())


# ------------------------------------------------------------------------------- batch invariance, reruns, launches


@pytest.mark.parametrize("name,k,clamp,masked", INVARIANCE,
                         ids=[f"{a}-k{k}-{'clamp' if c else 'raw'}{'-masked' if m else ''}" for a, k, c, m in INVARIANCE])
def test_rows_do_not_depend_on_their_batch(name, k, clamp, masked):
    """Ranking U[1000:] moves every batch boundary by 1000 rows, and splitting at row 131,072 by another amount; every row
    must come out with the same bits as in the full call, and a rerun must repeat them."""
    U, V, _ = family(name)
    n = U.shape[0]
    assert n_batches(n, k) >= 2
    ex = exclusion(name) if masked else None
    part = lambda a, b: run_topk(U[a:b], V, k, clamp, ex=None if ex is None else sub_csr(ex, a, b))  # noqa: E731
    full = part(0, n)
    assert_same(part(0, n), full, "rerun")
    assert_same(part(1000, n), (full[0][1000:], full[1][1000:]), "U[1000:]")
    h = 131_072
    assert_same(part(0, h), (full[0][:h], full[1][:h]), "U[:131072]")
    assert_same(part(h, n), (full[0][h:], full[1][h:]), "U[131072:]")


@pytest.mark.parametrize("name,k,clamp,masked", LAUNCHES,
                         ids=[f"{a}-k{k}-{'clamp' if c else 'raw'}{'-masked' if m else ''}" for a, k, c, m in LAUNCHES])
def test_launch_counts(name, k, clamp, masked):
    """torch.profiler's kernel records: one main-kernel and one rerank launch per batch, exact_rows_kernel once, and
    clamp_fill_kernel once for masked clamp-mode calls only"""
    from torch.profiler import ProfilerActivity, profile
    U, V, _ = family(name)
    ex = exclusion(name) if masked else None
    run_topk(U, V, k, clamp, ex=ex)  # module loads and attribute setting outside the trace
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run_topk(U, V, k, clamp, ex=ex)
    counts = collections.Counter()
    for e in prof.key_averages():
        counts[e.key] += e.count
    launched = lambda s: sum(c for key, c in counts.items() if s in key)  # noqa: E731
    batches = n_batches(U.shape[0], k)
    assert batches >= 2
    print(f"\n{name} n_users={U.shape[0]} k={k} clamp={clamp} masked={masked}: " +
          "; ".join(f"{key} x{c}" for key, c in sorted(counts.items()) if "tmf::" in key or "kernel" in key))
    assert launched("score_topk_kernel") == batches
    assert launched("rerank_kernel") == batches
    assert launched("exact_rows_kernel") == 1
    assert launched("clamp_fill_kernel") == (1 if masked and clamp else 0)
    assert len([key for key in counts if "score_topk_kernel" in key]) == 1  # one instantiation


# ------------------------------------------------------------------------------- the dense fallback beyond k = 1024


@pytest.mark.parametrize("clamp", [False, True])
def test_masked_topk_dense_row_blocks(clamp):
    """evaluation.masked_topk ranks k > 1024 in dense row blocks of min(4096, 2^27 // n_items) rows, re-basing the
    exclusion CSR per block.  Rows with 7 unseen items and rows with an empty list sit on both sides of each block edge."""
    from teamoflow_b200.mf.evaluation import PAD_ID, masked_topk
    n_u, n_i, r, k = 10_000, 6_000, 32, 1500
    block = max(1, min(4096, (1 << 27) // n_i))
    edges = list(range(block, n_u, block))
    assert len(edges) == 2
    g = torch.Generator(device=DEV)
    g.manual_seed(17)
    U = (torch.randn(n_u, r, generator=g, device=DEV) / r ** 0.5).contiguous()
    V = (torch.randn(n_i, r, generator=g, device=DEV) / r ** 0.5).contiguous()
    lens = torch.randint(0, 101, (n_u,), generator=g, device=DEV)
    few, empty = [0], [n_u - 1]
    for e in edges:
        few += [e - 1, e]
        empty += [e - 2, e + 1]
    lens[few + empty] = 0
    rows = torch.repeat_interleave(torch.arange(n_u, device=DEV), lens)
    keys = [rows * n_i + torch.randint(0, n_i, (rows.numel(),), generator=g, device=DEV)]
    for x in few:  # every item but 7 seen
        keys.append(x * n_i + torch.randperm(n_i, generator=g, device=DEV)[7:])
    keys = torch.unique(torch.cat(keys))
    ptr = torch.zeros(n_u + 1, dtype=torch.int32, device=DEV)
    ptr[1:] = torch.cumsum(torch.bincount(keys // n_i, minlength=n_u), 0).int()
    idx = (keys % n_i).int().contiguous()
    got = masked_topk(U, V, r, k, clamp, ptr, idx)
    want, _ = reference_topk(U, V, k, clamp, (ptr, idx))
    assert PAD_ID == PAD
    bad = (got != want).any(1)
    assert not bool(bad.any()), f"{int(bad.sum())} rows differ, first {bad.nonzero().flatten()[:6].tolist()}"
    for x in few:
        assert bool((got[x, 7:] == PAD).all()) and bool((got[x, :7] != PAD).all())
