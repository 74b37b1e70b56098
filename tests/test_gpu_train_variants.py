"""Every compiled variant of the training user pass (tmf_user_pass + tmf_user_pass_fixup) and of the segment sum
(tmf_spmm_seg) against an fp64 reference, through the raw C ABI.

tmf_user_pass launches one of 27 instantiations of user_pass_kernel<LPR, VPL, JPL, LOSS>, chosen from ld and the number of
samples; tmf_spmm_seg picks its lanes per row from n_cols and its chunk from n_entries.  `user_pass_variant` and
`spmm_variant` restate those rules, so the case tables below provably reach every instantiation, the narrow sample gather,
every chunk size and the thresholds between them: a CPU test checks the tables against the mirrors, and a GPU test checks the
mirror against the kernel names the profiler records.

Every output element is compared with a bound built from its own terms, not from the tensor's largest value, so a wrong small
row cannot hide behind a large one.  Outputs and partial buffers are filled with NaN before every call, so a skipped store
cannot pass for a correct zero.  Reruns, the order of the work items and the coefficient slot map must not change a bit.
"""
import functools
import math
import re

import numpy as np
import pytest
import torch
from scipy import sparse

from oracle import mf_oracle as o

MSE, WMRB = 0, 1  # TMF_LOSS_MSE, TMF_LOSS_WMRB (include/tmf.h)
REL = 1e-5        # north_star: losses, gradients and scores agree within 1e-5 relative in fp32
L = 48            # slice length of split users: not a power of two, so slices do not line up with the row groups


# ------------------------------------------------------------------------------- dispatch mirrors


def user_pass_variant(loss, ld, S):
    """(LPR, VPL, JPL, LOSS) of the user_pass_kernel that tmf_user_pass launches, and whether its narrow sample gather runs
    (train.cu: tmf_user_pass, dispatch_user_pass_j and NARROW_OK)."""
    nv = ld // 4
    lpr = 4
    while lpr < nv and lpr < 32:
        lpr *= 2
    if loss == WMRB:
        while lpr < 32 and -(-S // lpr) > 16:
            lpr *= 2
    vpl = 2 if nv > 32 else 1
    jpl = 0 if loss == MSE else next((j for j in (2, 4, 8, 16) if -(-S // lpr) <= j), -1)
    sw = lpr
    if (jpl == 16 or jpl < 0) and vpl == 1 and lpr > 4:
        while sw > 4 and sw // 2 >= nv:
            sw //= 2
    return (lpr, vpl, jpl, loss), sw < lpr


def spmm_variant(n_cols, n_entries):
    """(LPR, chunk) of tmf_spmm_seg (train.cu: tmf_spmm_seg and spmm_chunk_for)."""
    nv = -(-n_cols // 4)
    lpr = next(w for w in (4, 8, 16, 32) if nv <= w or w == 32)
    chunk = 32
    while chunk < n_entries // 32768 and chunk < 256:
        chunk *= 2
    return lpr, chunk


ALL_USER_PASS = [  # (LPR, VPL, JPL, LOSS): every user_pass_kernel instantiation in train.cu
    (4, 1, 0, MSE), (8, 1, 0, MSE), (16, 1, 0, MSE), (32, 1, 0, MSE), (32, 2, 0, MSE),
    (4, 1, 2, WMRB), (4, 1, 4, WMRB), (4, 1, 8, WMRB), (4, 1, 16, WMRB),
    (8, 1, 2, WMRB), (8, 1, 4, WMRB), (8, 1, 8, WMRB), (8, 1, 16, WMRB),
    (16, 1, 2, WMRB), (16, 1, 4, WMRB), (16, 1, 8, WMRB), (16, 1, 16, WMRB),
    (32, 1, 2, WMRB), (32, 1, 4, WMRB), (32, 1, 8, WMRB), (32, 1, 16, WMRB), (32, 1, -1, WMRB),
    (32, 2, 2, WMRB), (32, 2, 4, WMRB), (32, 2, 8, WMRB), (32, 2, 16, WMRB), (32, 2, -1, WMRB),
]


def _case(loss, r, S=0, ld=None):
    return loss, r, S, ld or -(-r // 4) * 4


# (loss, r, S, ld); consecutive entries sit on both sides of a threshold of the dispatch rule
UP_CASES = [_case(MSE, r) for r in (3, 13, 32, 61, 128, 129, 256)] + [_case(WMRB, r, S) for r, S in (
    (7, 8), (16, 9), (8, 20), (15, 33), (15, 64),                           # LPR 4
    (17, 16), (32, 17), (30, 64), (31, 128), (12, 100), (15, 65),          # LPR 8; the last two narrow
    (33, 32), (64, 33), (50, 128), (64, 256), (32, 200),                    # LPR 16; (32, 200) narrow
    (65, 64), (100, 65), (128, 256), (97, 512), (128, 512), (40, 400),      # LPR 32; (40, 400) narrow
    (128, 513), (128, 1000), (20, 700),                                     # generic G in shared memory; (20, 700) narrow
    (129, 64), (200, 65), (256, 256), (160, 512), (140, 513), (256, 1100),  # two float4 columns per lane (ld > 128)
)] + [_case(MSE, 10, 0, 136), _case(WMRB, 10, 40, 136)]  # padded storage: the kernel dispatches on ld, so this is VPL 2


def _up_id(case):
    loss, r, S, ld = case
    return f"{'mse' if loss == MSE else 'wmrb'}-r{r}-S{S}-ld{ld}"


# (chunk, n_cols, n_entries): every chunk size with two widths; every width with a chunk above 32; n_entries a multiple of
# the chunk in the first case of each pair and not in the second
SPMM_CASES = [(32, 3, 300_000), (32, 200, 300_013), (64, 20, 1_200_000), (64, 60, 1_200_037),
              (128, 3, 2_300_032), (128, 200, 2_300_101), (256, 20, 4_400_128), (256, 60, 4_400_203)]


def test_case_tables_reach_every_variant():
    assert len(set(ALL_USER_PASS)) == 27
    got = [user_pass_variant(loss, ld, S) for loss, r, S, ld in UP_CASES]
    assert {v for v, _ in got} == set(ALL_USER_PASS)
    # the narrow sample gather at every width that has it, in the register and in the shared-memory G kernels
    assert {v[:3] for v, narrow in got if narrow} == {(8, 1, 16), (16, 1, 16), (32, 1, 16), (32, 1, -1)}
    assert all(ld > -(-r // 4) * 4 for _, r, _, ld in UP_CASES[-2:])
    pairs = [spmm_variant(n_cols, n) for _, n_cols, n in SPMM_CASES]
    assert [c for _, c in pairs] == [c for c, _, _ in SPMM_CASES]
    assert set(pairs) == {(4, 32), (32, 32), (8, 64), (16, 64), (4, 128), (32, 128), (8, 256), (16, 256)}
    for w in {n_cols for _, n_cols, _ in SPMM_CASES}:
        assert any(c > 32 for c, n_cols, _ in SPMM_CASES if n_cols == w)
    assert any(-(-n_cols // 4) > 32 for _, n_cols, _ in SPMM_CASES)  # two column blocks (grid.y = 2)
    for c in (32, 64, 128, 256):
        ns = [n for cc, _, n in SPMM_CASES if cc == c]
        assert any(n % c == 0 for n in ns) and any(n % c for n in ns)


# ------------------------------------------------------------------------------- helpers


def close(got, want, rel=REL, name=""):
    """max-abs error relative to the tensor's max-abs value"""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    scale = max(np.abs(want).max() if want.size else 0.0, 1e-30)
    err = np.abs(got - want).max() if want.size else 0.0
    assert err <= rel * scale, f"{name}: max abs err {err:.3e} > {rel} * {scale:.3e}"


def within(got, want, bound, name):
    """elementwise |got - want| <= bound (NaN fails)"""
    err = np.abs(np.asarray(got, np.float64) - want)
    bad = ~(err <= bound)
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError(f"{name}: {int(bad.sum())} of {bad.size} elements outside their bound; first at {i}: "
                             f"got {got[i]!r}, want {want[i]!r}, bound {bound[i] if np.ndim(bound) else bound:.3e}")


def same_bits(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _abi():
    from teamoflow_b200 import _abi
    return _abi


def dev(x):
    return None if x is None else torch.as_tensor(np.ascontiguousarray(x), device="cuda")


# ------------------------------------------------------------------------------- user pass


@functools.lru_cache(maxsize=None)
def user_problem(loss, r, S, ld):
    """96 users with 0, 1, L, L + 1, 2L + 3 and 5L interactions, two users whose values are all non-positive (one of them
    split), random counts for the rest; the fp64 reference of every output."""
    rng = np.random.default_rng(1000 * r + S + ld + loss)
    n_u, n_i = 96, max(3 * S, 400)
    special = [0, 0, 1, 1, L, L + 1, 2 * L + 3, 5 * L, 7, L + 2]
    counts = np.concatenate([special, rng.integers(2, 40, n_u - len(special))])
    nonpos = np.isin(np.arange(n_u), [len(special) - 2, len(special) - 1])  # the users with 7 and L + 2 interactions
    perm = rng.permutation(n_u)
    counts, nonpos = counts[perm], nonpos[perm]
    row_ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    rows = np.repeat(np.arange(n_u), counts)
    cols = np.concatenate([rng.choice(n_i, c, replace=False) for c in counts]).astype(np.int32)
    vals = np.where(nonpos[rows], rng.choice(np.array([0.0, -1.0], np.float32), rows.size),
                    rng.choice(np.array([1.0, 2.0, 3.0, 0.0, -1.0], np.float32), rows.size)).astype(np.float32)
    if loss == WMRB:
        # small integers times powers of two: every product and partial sum of a score is exact in fp32 in any order, so
        # each hinge 1 - p + s is exact and the kernel's indicator must be the fp64 one, hinges exactly at 0 included.
        # Scores ~ N(0, 0.5^2) on a lattice of 2^-e.
        e = math.ceil(math.log2(8 * math.sqrt(r)))
        Eu = rng.integers(-3, 4, (n_u, r)) * 2.0 ** -(e // 2)
        Ei = rng.integers(-3, 4, (n_i, r)) * 2.0 ** -(e - e // 2)
        samp = np.argsort(rng.random((n_u, n_i)), axis=1)[:, :S].astype(np.int32)  # distinct items per row
    else:
        Eu = rng.standard_normal((n_u, r)) / r ** 0.25
        Ei = rng.standard_normal((n_i, r)) / r ** 0.25
        samp = np.zeros((n_u, 0), np.int32)
    pad = lambda x: np.pad(x, ((0, 0), (0, ld - r))).astype(np.float32)  # noqa: E731  columns [r, ld) are zero (tmf.h)
    Eu, Ei = pad(Eu), pad(Ei)

    Eu64, Ei64 = Eu.astype(np.float64), Ei.astype(np.float64)
    P = Eu64 @ Ei64.T
    p = P[rows, cols]
    a = vals.astype(np.float64)
    nnz = rows.size
    if loss == WMRB:
        ss = np.take_along_axis(P, samp, 1)
        pos = a > 0
        h = 1.0 - p[pos][:, None] + ss[rows[pos]]
        hinges = ((h == 0).sum(), (h > 0).sum(), (h < 0).sum())
        loss_pos, c, G = o.wmrb_coefs(rows, a, p, ss, n_i, S)
        loss_k = np.zeros(nnz)
        loss_k[pos] = loss_pos
        c_mag = np.abs(c)
        tol_c, tol_loss = REL * np.abs(c), REL * np.abs(loss_k)
    else:
        hinges = None
        df = a - p
        loss_k, c, G = df * df, -2.0 * df, np.zeros((n_u, 0))
        M = np.abs(a) + (np.abs(Eu64[rows]) * np.abs(Ei64[cols])).sum(1)  # magnitude of a - p's terms: it cancels
        c_mag = 2 * M
        tol_c, tol_loss = REL * c_mag, REL * 2 * np.abs(df) * M + (REL * M) ** 2
    C = sparse.csr_matrix((c, cols, row_ptr), shape=(n_u, n_i))
    Cm = sparse.csr_matrix((c_mag, cols, row_ptr), shape=(n_u, n_i))
    s_ptr = np.arange(0, n_u * S + 1, S) if S else np.zeros(n_u + 1, np.int64)
    Gs = sparse.csr_matrix((G.ravel(), samp.ravel(), s_ptr), shape=(n_u, n_i))
    Gm = sparse.csr_matrix((np.abs(G).ravel(), samp.ravel(), s_ptr), shape=(n_u, n_i))
    dE = C @ Ei64 + Gs @ Ei64
    dE_bound = REL * (Cm @ np.abs(Ei64) + Gm @ np.abs(Ei64))  # sum_k |c_k||Ei[col_k]| + sum_j |G_uj||Ei[samp_uj]|
    return dict(loss=loss, r=r, S=S, ld=ld, n_u=n_u, n_i=n_i, nnz=nnz, counts=counts, row_ptr=row_ptr, cols=cols, vals=vals,
                Eu=Eu, Ei=Ei, samp=samp, hinges=hinges, want_loss=loss_k, want_c=c, want_G=G, want_dE=dE,
                tol_loss=tol_loss, tol_c=tol_c, tol_G=REL * np.abs(G), tol_dE=dE_bound)


def work_list(row_ptr):
    """tmf.h's work list: whole users (slot -1) and the L-long slices of heavier users (consecutive slot rows), heaviest
    first; plus the split users' (user, first slot, slice count) for the fix-up"""
    items, split = [], []
    n_slots = 0
    for u in range(row_ptr.size - 1):
        a, b = int(row_ptr[u]), int(row_ptr[u + 1])
        if b - a <= L:
            items.append((u, a, b, -1))
            continue
        nseg = -(-(b - a) // L)
        split.append((u, n_slots, nseg))
        for s in range(nseg):
            items.append((u, a + s * L, min(a + (s + 1) * L, b), n_slots))
            n_slots += 1
    items.sort(key=lambda t: t[1] - t[2])  # stable: heaviest first
    return np.array(items, np.int32), np.array(split, np.int32), n_slots


class UserPassRun:
    """device buffers of one case; run() makes one tmf_user_pass (+ fix-up) call and returns (loss_out, coef_out, dEu)"""
    TAIL = 4  # extra NaN elements after loss_out and coef_out: nothing may write there

    def __init__(self, pb):
        self.pb = pb
        self.T = pb["nnz"] + pb["n_u"] * pb["S"]
        self.inputs = {k: dev(pb[k]) for k in ("row_ptr", "cols", "vals", "Eu", "Ei")}
        self.samp = dev(pb["samp"]) if pb["loss"] == WMRB else None
        self.items, self.split, self.n_slots = work_list(pb["row_ptr"])
        self.counter = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.loss_out = torch.empty(pb["nnz"] + self.TAIL, device="cuda")
        self.coef_out = torch.empty(self.T + self.TAIL, device="cuda")
        self.dEu = torch.empty(pb["n_u"], pb["ld"], device="cuda")
        self.part_G = torch.empty(max(self.n_slots, 1), max(-(-pb["S"] // 4) * 4, 4), device="cuda")
        self.part_E = torch.empty(max(self.n_slots, 1), pb["ld"], device="cuda")
        self.split_d = [dev(self.split[:, i]) for i in range(3)]

    def run(self, items=None, coef_pos=None):
        pb, A = self.pb, _abi()
        for t in (self.loss_out, self.coef_out, self.dEu, self.part_G, self.part_E):
            t.fill_(float("nan"))
        wl = [None] * 4 if items is None else [dev(items[:, i]) for i in range(4)]
        cp = dev(coef_pos)
        x = self.inputs
        A.call("tmf_user_pass", pb["loss"], pb["n_u"], pb["n_i"], pb["nnz"], A.ptr(x["row_ptr"]), A.ptr(x["cols"]),
               A.ptr(x["vals"]), A.ptr(x["Eu"]), A.ptr(x["Ei"]), pb["ld"], pb["r"], A.ptr(self.samp), pb["S"],
               pb["n_u"] if items is None else len(items), *[A.ptr(t) for t in wl], A.ptr(self.part_G), A.ptr(self.part_E),
               A.ptr(self.counter), A.ptr(self.loss_out), A.ptr(self.coef_out), A.ptr(cp), A.ptr(self.dEu))
        if items is not None:
            A.call("tmf_user_pass_fixup", pb["loss"], len(self.split), *[A.ptr(t) for t in self.split_d], A.ptr(x["Ei"]),
                   pb["ld"], A.ptr(self.samp), pb["S"], pb["nnz"], A.ptr(self.part_G), A.ptr(self.part_E),
                   A.ptr(self.coef_out), A.ptr(cp), A.ptr(self.dEu))
        torch.cuda.synchronize()
        return tuple(t.cpu().numpy() for t in (self.loss_out, self.coef_out, self.dEu))


def check_user_pass(pb, out, coef_pos, what):
    loss_k, coef, dEu = out
    nnz, n_u, S, r = pb["nnz"], pb["n_u"], pb["S"], pb["r"]
    T = nnz + n_u * S
    assert np.isnan(loss_k[nnz:]).all() and np.isnan(coef[T:]).all(), f"{what}: store past the end of loss_out / coef_out"
    loss_k, coef = loss_k[:nnz], coef[:T]
    if coef_pos is not None:
        coef = coef[coef_pos]  # slot e lives at coef_pos[e]
    for name, x in (("loss_out", loss_k), ("coef_out", coef), ("dEu", dEu)):
        assert not np.isnan(x).any(), f"{what}: {int(np.isnan(x).sum())} elements of {name} never written"
    assert (dEu[:, r:] == 0).all(), f"{what}: dEu columns [r, ld) are not zero"
    c, G = coef[:nnz], coef[nnz:].reshape(n_u, S)
    if pb["loss"] == WMRB:
        assert (loss_k[pb["vals"] <= 0] == 0).all(), f"{what}: non-positive interactions have a loss"
        empty = pb["counts"] == 0
        assert (G[empty] == 0).all() and (dEu[empty] == 0).all(), f"{what}: users without interactions have gradients"
    within(loss_k, pb["want_loss"], pb["tol_loss"], f"{what}: loss")
    within(c, pb["want_c"], pb["tol_c"], f"{what}: c")
    within(G, pb["want_G"], pb["tol_G"], f"{what}: G")
    within(dEu, pb["want_dE"], pb["tol_dE"], f"{what}: dE_u")
    close(loss_k, pb["want_loss"], name=f"{what}: loss")
    close(c, pb["want_c"], name=f"{what}: c")
    close(G, pb["want_G"], name=f"{what}: G")
    close(dEu, pb["want_dE"], name=f"{what}: dE_u")
    return loss_k, coef, dEu


@pytest.mark.gpu
@pytest.mark.parametrize("case", UP_CASES, ids=_up_id)
def test_user_pass_variant_matches_fp64(case):
    """Four runs (work list NULL or with split users, times coef_pos NULL or a permutation), each checked against the fp64
    reference element by element, rerun and, with a work list, rerun with its items shuffled: every bit must repeat."""
    pb = user_problem(*case)
    if pb["loss"] == WMRB:  # the data must put hinges exactly at 0 (tf.maximum routes the gradient there) and on both sides
        at0, active, inactive = pb["hinges"]
        assert at0 > 0 and active > 0 and inactive > 0, f"hinges at 0 / > 0 / < 0: {pb['hinges']}"
    up = UserPassRun(pb)
    assert len(up.split) > 0 and up.n_slots > len(up.split)
    rng = np.random.default_rng(7)
    perm = rng.permutation(up.T).astype(np.int32)
    for items in (None, up.items):
        natural = None
        for coef_pos in (None, perm):
            what = ("work list" if items is not None else "one item per user") + \
                (", coef_pos set" if coef_pos is not None else ", coef_pos NULL")
            out = up.run(items, coef_pos)
            got = check_user_pass(pb, out, coef_pos, what)
            again = up.run(items, coef_pos)
            assert all(same_bits(x, y) for x, y in zip(out, again)), f"{what}: a rerun changed the outputs"
            if items is not None:
                shuffled = up.run(items[rng.permutation(len(items))], coef_pos)
                assert all(same_bits(x, y) for x, y in zip(out, shuffled)), f"{what}: the work-item order changed the outputs"
            if natural is None:
                natural = got
            else:
                assert all(same_bits(x, y) for x, y in zip(natural, got)), f"{what}: differs from the natural coefficient layout"


_KERNEL = re.compile(r"user_pass_kernel<([^>]*)>")


def launched_user_pass(names):
    """(LPR, VPL, JPL, LOSS) of every user_pass_kernel name: '<16, 1, 4, 1>' and '<(int)16, (int)1, (int)4, (int)1>'"""
    found = (_KERNEL.search(n) for n in names)
    return {tuple(int(v.replace("(int)", "")) for v in m.group(1).split(",")) for m in found if m}


@pytest.mark.gpu
def test_user_pass_cases_launch_the_predicted_instantiation():
    """The profiler's kernel names prove on the device that each case runs the instantiation the mirror predicts and that
    the table reaches all 27."""
    from torch.profiler import ProfilerActivity, profile
    seen = set()
    for case in UP_CASES:
        up = UserPassRun(user_problem(*case))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            up.run()
        got = launched_user_pass(e.key for e in prof.key_averages())
        want = user_pass_variant(case[0], case[3], case[2])[0]
        assert got == {want}, f"{_up_id(case)}: launched {got}, the mirror predicts {want}"
        seen |= got
    assert seen == set(ALL_USER_PASS)


# ------------------------------------------------------------------------------- segment sum


def segment_layout(n, C, rng):
    """seg_ptr over n entries for chunk C: random lengths (one in eight spanning several chunks, one in twenty empty), an
    empty first and last segment, and in chunks of their own: a segment ending exactly at a chunk boundary with the next
    starting there; one starting mid-chunk and spanning four chunks; empty segments just before, at and just after a
    boundary around a length-1 segment on that chunk's last entry; and a length-1 segment on a chunk's last entry between
    two non-empty ones."""
    m = 2 * n // C + 64
    lens = rng.geometric(2.0 / C, m)
    long = rng.random(m) < 0.125
    lens[long] = rng.integers(C, 6 * C, int(long.sum()))
    lens[rng.random(m) < 0.05] = 0
    cuts = np.cumsum(lens)
    cuts = cuts[cuts < n]
    keep = np.ones(cuts.size, bool)
    for lo, hi in ((2 * C, 4 * C), (9 * C, 15 * C), (19 * C, 21 * C), (29 * C, 31 * C)):
        keep &= (cuts <= lo) | (cuts >= hi)
    k = 3 * C
    edge = [k - C + C // 3, k, k + C // 2]
    k = 10
    edge += [k * C + C // 2 + 1, (k + 3) * C + C // 2 + 3]
    k = 20 * C
    edge += [k - 3, k - 1, k - 1, k - 1, k, k, k, k + 1, k + 1, k + 4]
    k = 30 * C
    edge += [k - 5, k - 1, k, k + 7]
    cuts = np.sort(np.concatenate([cuts[keep], edge]))
    return np.concatenate([[0, 0], cuts, [n, n]]).astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk,n_cols,n", SPMM_CASES)
def test_spmm_seg_chunk_matches_fp64(chunk, n_cols, n):
    """tmf_spmm_seg at every chunk size and lanes-per-row width, with coef NULL (c = 1), coef with cpos NULL and coef with a
    cpos permutation, against an fp64 scipy.sparse product, element by element."""
    A = _abi()
    rng = np.random.default_rng(chunk + n_cols + n)
    nv4 = -(-n_cols // 4) * 4
    ld_src, ld_out = nv4, nv4 + 8
    need = A.query("tmf_spmm_ws_bytes", n, ld_out)
    assert (need - 256) % (8 * ld_out) == 0
    n_chunks = (need - 256) // (8 * ld_out)  # 2 * ceil(n / chunk) * ld_out * 4 + 256
    assert [c for c in (32, 64, 128, 256) if -(-n // c) == n_chunks] == [chunk] == [spmm_variant(n_cols, n)[1]]

    seg_ptr = segment_layout(n, chunk, rng)
    n_seg = seg_ptr.size - 1
    lens = np.diff(seg_ptr)
    first, last = seg_ptr[:-1] // chunk, (seg_ptr[1:] - 1) // chunk
    assert lens[0] == 0 and lens[-1] == 0 and ((seg_ptr[:-1] % chunk > 0) & (lens > 0) & (last - first >= 3)).any()
    n_src = 50_000
    idx = rng.integers(0, n_src, n).astype(np.int32)
    src = np.zeros((n_src, ld_src), np.float32)
    src[:, :n_cols] = rng.standard_normal((n_src, n_cols))
    coef = rng.standard_normal(n).astype(np.float32)
    cpos = rng.permutation(n).astype(np.int32)
    src64 = src[:, :n_cols].astype(np.float64)
    abs_src = np.abs(src64)
    d_seg, d_idx, d_src, d_coef, d_cpos = dev(seg_ptr), dev(idx), dev(src), dev(coef), dev(cpos)
    out = torch.empty(n_seg, ld_out, device="cuda")
    ws = torch.empty(need + 4096, dtype=torch.uint8, device="cuda")
    canary = torch.arange(4096, device="cuda").remainder(251).add(1).to(torch.uint8)

    def run(c_dev, p_dev):
        out.fill_(float("nan"))
        ws[need:] = canary
        A.call("tmf_spmm_seg", n_seg, A.ptr(d_seg), n, A.ptr(d_idx), A.ptr(p_dev), A.ptr(c_dev), A.ptr(d_src), ld_src,
               A.ptr(out), ld_out, n_cols, A.ptr(ws), need)
        torch.cuda.synchronize()
        assert torch.equal(ws[need:], canary), "tmf_spmm_seg wrote past its workspace"
        return out.cpu().numpy()

    for mode, c_dev, p_dev, c in (("coef NULL", None, None, np.ones(n)), ("cpos NULL", d_coef, None, coef.astype(np.float64)),
                                  ("cpos set", d_coef, d_cpos, coef[cpos].astype(np.float64))):
        got = run(c_dev, p_dev)
        assert not np.isnan(got[:, :nv4]).any(), f"{mode}: {int(np.isnan(got[:, :nv4]).sum())} output elements never written"
        assert np.isnan(got[:, nv4:]).all(), f"{mode}: columns past 4 * ceil(n_cols / 4) were written"
        assert (got[lens == 0, :nv4] == 0).all(), f"{mode}: empty segments are not zero"
        assert (got[:, n_cols:nv4] == 0).all(), f"{mode}: pad columns are not zero"
        want = sparse.csr_matrix((c, idx, seg_ptr), shape=(n_seg, n_src)) @ src64
        bound = REL * (sparse.csr_matrix((np.abs(c), idx, seg_ptr), shape=(n_seg, n_src)) @ abs_src)  # sum |c||src|
        within(got[:, :n_cols], want, bound, mode)
        close(got[:, :n_cols], want, name=mode)
        assert same_bits(got, run(c_dev, p_dev)), f"{mode}: a rerun changed the result"
