"""The row kernel's candidate select (k_rows in csrc/cco_kernels.cuh: counts, LLR and top-k fused) under candidate-buffer
pressure, in every bin and every top_k range, against the oracle -- plus the packed-word, level-1-cut and minLLR edges, and
the kernel's LLR against a 50-digit evaluation of Mahout's formula that does not go through the project's own fp64 code.

The workloads are structured so that the row work and the number of strongly positive cells of each row are known in
advance: primary item a has `ra` users of its own, each of them holds `d` B-columns nobody else holds.  So a row's work is
w = ra * d, every one of its w cells has k11 == 1, and extra users without any event make N large enough that every cell
is strongly positive.  With every column marginal cb == 1 all cells of a row tie on LLR and the column alone decides the
top-k: the radix select has to resolve the column digits.  The `spread` variant adds cb in 1..8 (several LLR levels, the
k-th cell inside a tie group)."""
import decimal
import functools
import math

import numpy as np
import pytest

import universal_recommender_b200 as ur
from test_gpu_parity import assert_indicators_equal, oracle_train

B200_SMEM_OPTIN = 232448   # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200
MAX_TOP_K = 2048           # CCO_MAX_TOP_K (include/cco_b200.h)
K_SWEEP = [1, 32, 64, 65, 97, 128, 224, 225, 256, 257, 300, 384, 385, 512, 513, 640, 768, 769, 896, 1024, 1100, 1536, 1537,
           1900, 2048]
# top_k ranges in which keep_max would exceed cbuf - group without the cap in make_cfg (one k of each for m = 500)
RANGES = {128: [(257, 384), (513, 896), (1025, 1920)], 256: [(513, 768), (1025, 1792)], 512: [(1025, 1536)]}
K_DOWNSAMPLED = [50, 300, 640, 1100, 1537, 2048]


# ---- mirror of the row-kernel configuration (csrc/cco_api.cu) --------------------------------------------------------------
def _next_pow2(x):
    p = 1
    while p < x:
        p <<= 1
    return p


def make_cfg(group, want_slots, k, n_cols_b, optin, capped=True):
    """make_cfg (cco_api.cu, "Candidate-buffer invariant").  capped=False is the formula before keep_max was capped."""
    groups = 2 if group == 32 else 1
    final_max = _next_pow2(k)
    cbuf = _next_pow2(k + max(group, 128) + (64 if group == 32 else 0))
    if group == 32 and k + 32 <= 96:
        cbuf = 128
    keep_max = max(final_max, (cbuf - group) // 2)
    if capped:
        keep_max = min(keep_max, cbuf - group)
    caux = 0 if group == 32 else max(keep_max, final_max)
    fixed = (cbuf + caux) * 16 + 2 * 256 + 512 + 1024 + (group // 32) * 256
    slots = min(want_slots, ((optin - 1024) // groups - fixed) // 4 & ~1023)
    return dict(group=group, slots=slots, cap=slots // 2, cbuf=cbuf, caux=caux, keep_max=keep_max, final_max=final_max,
                prune_limit=cbuf - group, dense=n_cols_b <= slots)


def bins(k, n_cols_b, optin, capped=True):
    """enqueue_indicator's bins (cco_api.cu, "2. bins"): [(cfg, lo, hi)], bin b takes the rows with lo < w <= hi; the
    first entry is the multi-pass bin (absent when the large bin is dense)."""
    top = 2 ** 32 - 1
    spec = [(1024, 1 << 20, top), (1024, 1 << 20, top), (512, 16384, 8192), (256, 8192, 4096), (128, 4096, 2048)]
    if k + 32 <= 256:
        spec += [(32, 2048, 1024), (32, 1024, 512), (32, 512, 256)]
    cfgs = [make_cfg(g, s, k, n_cols_b, optin, capped) for g, s, _ in spec]
    thr = []
    for b in range(len(spec)):
        lim = spec[b + 1][2] if b + 1 < len(spec) else 0
        if b + 1 < len(spec) and not cfgs[b + 1]["dense"]:
            lim = min(lim, cfgs[b + 1]["cap"])
        thr.append(min(lim, thr[-1]) if thr else lim)
    return [(cfgs[b], thr[b], top if b == 0 else thr[b - 1]) for b in range(len(spec)) if not (b == 0 and cfgs[1]["dense"])]


def bin_of(w, k, n_cols_b, optin, capped=True):
    return next(c for c, lo, hi in bins(k, n_cols_b, optin, capped) if lo < w <= hi)


def invariant_ok(c, k):
    return (k <= c["keep_max"] <= c["cbuf"] - c["group"] and c["final_max"] <= c["cbuf"]
            and (c["group"] == 32 or c["caux"] >= max(c["keep_max"], c["final_max"])))


# ---- structured workloads --------------------------------------------------------------------------------------------------
def _csr(rows, nc):
    rp = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum([len(r) for r in rows], out=rp[1:])
    ci = np.concatenate([np.asarray(r, dtype=np.int32) for r in rows]) if rows else np.zeros(0, np.int32)
    return (len(rows), nc, rp, ci.astype(np.int32))


def structured(shapes, n_extra=200_000, spread=False, n_cols=None, seed=0):
    """shapes = [(ra, d)] per primary item -> mats [A, B].  Item a gets ra users of its own, each with d B-columns of its
    own (w = ra * d cells, all k11 == 1).  spread: column c gets 0..7 more holders among 8 users without primary events."""
    rng = np.random.default_rng(seed)
    a_rows, b_rows = [], []
    col = 0
    for a, (ra, d) in enumerate(shapes):
        for _ in range(ra):
            a_rows.append([a])
            b_rows.append(np.arange(col, col + d))
            col += d
    nc = n_cols or col
    assert nc >= col
    if spread:
        extra = rng.integers(0, 8, col)                       # cb = 1 + extra
        for f in range(8):
            a_rows.append([])
            b_rows.append(np.nonzero(extra > f)[0])
    a_rows += [[]] * n_extra
    b_rows += [np.zeros(0, np.int64)] * n_extra
    return [_csr(a_rows, len(shapes)), _csr(b_rows, nc)]


# row work at both edges of every bin's max_w, inside every bin, and one multi-pass row (w > cap of the 1024 bin)
HASHED_SHAPES = [(4, 25), (4, 64), (1, 257), (8, 64), (3, 171), (16, 64), (5, 205), (12, 125), (32, 64), (3, 683),
                 (10, 300), (64, 64), (17, 241), (20, 300), (64, 128), (3, 2731), (24, 500), (8, 3000)]
# every column inside the table of the 1024 bin (dense at every top_k: n_cols <= 30720 slots at k = 2048)
DENSE_SHAPES = [(4, 25), (5, 205), (3, 683), (17, 241), (3, 2731), (24, 500)]


def _row_works(mats):
    """k_row_work: products of each primary item's row = sum of its users' B-row lengths."""
    a, b = mats
    owner = np.repeat(np.arange(a[0]), np.diff(a[2]))
    w = np.zeros(a[1], dtype=np.int64)
    np.add.at(w, a[3], np.diff(b[2])[owner])
    return w


def _no_duplicate_columns(got):
    for rb, re_, nc, rp, ci, ll, cn in got:
        for r in range(len(rp) - 1):
            row = ci[rp[r]:rp[r + 1]]
            assert len(np.unique(row)) == len(row), f"row {r}: duplicate columns"


def _pressure_rows(mats, k, optin):
    """-> {group: max positive cells of a row in that bin} for the bins of this k."""
    w = _row_works(mats)
    out = {}
    for x in w[w > 0]:
        c = bin_of(int(x), k, mats[1][1], optin)
        out[c["group"]] = max(out.get(c["group"], 0), int(x))
    return out


# ---- CPU: the configuration invariant ------------------------------------------------------------------------------------------
def test_cfg_invariant_holds_for_every_top_k():
    for k in range(1, MAX_TOP_K + 1):
        for c, _, _ in bins(k, 10 ** 6, B200_SMEM_OPTIN):
            assert invariant_ok(c, k), (k, c)
            assert c["slots"] > 0 and c["cap"] > 0


def test_cfg_cap_changes_only_the_violating_configurations():
    # top_k <= 224 (every warp-owned configuration, the benchmark's k = 50): the cap leaves every byte as it was
    for k in range(1, MAX_TOP_K + 1):
        for (new, _, _), (old, _, _) in zip(bins(k, 10 ** 6, B200_SMEM_OPTIN), bins(k, 10 ** 6, B200_SMEM_OPTIN, False)):
            assert {**new, "keep_max": 0} == {**old, "keep_max": 0}, (k, new, old)   # same shared-memory layout
            if old["keep_max"] <= old["prune_limit"]:
                assert new == old, (k, new, old)
            else:
                assert k > 224 and new["group"] in RANGES
                assert any(lo <= k <= hi for lo, hi in RANGES[new["group"]]), (k, new["group"])
    # and the ranges listed are exactly the uncapped violations
    for g, rs in RANGES.items():
        old = [make_cfg(g, 1 << 20, k, 10 ** 6, B200_SMEM_OPTIN, False) for k in range(1, MAX_TOP_K + 1)]
        bad = [k for k, c in enumerate(old, 1) if c["keep_max"] > c["prune_limit"]]
        assert bad == [k for lo, hi in rs for k in range(lo, hi + 1)], g


def test_structured_shapes_reach_every_bin_and_overfill_the_candidate_buffer():
    """The sweep's rows hold more strongly positive cells than prune_limit + group in every bin whose uncapped
    configuration violated the invariant (at least two prunes in a row), except where the bin's own row-work limit
    makes that impossible: the 128-thread bin holds rows of <= 2048 products, so at 1025 <= k <= 1920 (cbuf 2048) it can
    never overflow."""
    mats = structured(HASHED_SHAPES)
    for k in K_SWEEP:
        groups_hit = _pressure_rows(mats, k, B200_SMEM_OPTIN)
        assert set(groups_hit) == {c["group"] for c, _, _ in bins(k, mats[1][1], B200_SMEM_OPTIN)}, k
        for g, rs in RANGES.items():
            if not any(lo <= k <= hi for lo, hi in rs):
                continue
            old = make_cfg(g, {512: 16384, 256: 8192, 128: 4096}[g], k, mats[1][1], B200_SMEM_OPTIN, False)
            if g == 128 and k > 1024:
                assert old["prune_limit"] + g >= 2048
                continue
            assert groups_hit[g] > old["prune_limit"] + g, (k, g, groups_hit[g], old)
    # the multi-pass bin is populated at every k, and the 1024 bin is dense in the dense workload at every k
    dm = structured(DENSE_SHAPES)
    assert _row_works(dm).max() > 8192
    for k in K_SWEEP:
        b = bins(k, mats[1][1], B200_SMEM_OPTIN)
        assert b[0][1] < int(_row_works(mats).max()), k
        assert make_cfg(1024, 1 << 20, k, dm[1][1], B200_SMEM_OPTIN)["dense"], k
    assert make_cfg(1024, 1 << 20, 300, 0, B200_SMEM_OPTIN)["slots"] == 45056
    assert make_cfg(1024, 1 << 20, 2048, 0, B200_SMEM_OPTIN)["slots"] == 30720


# ---- CPU: LLR against a 50-digit evaluation ----------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _xlogx_exact(x):
    if x == 0:
        return decimal.Decimal(0)
    with decimal.localcontext() as c:
        c.prec = 50
        d = decimal.Decimal(x)
        return d * d.ln()


def llr_exact(k11, k12, k21, k22):
    """Mahout's LogLikelihood.logLikelihoodRatio (SURVEY.md A.3) in 50-digit decimal arithmetic."""
    with decimal.localcontext() as c:
        c.prec = 50
        x = _xlogx_exact
        n = k11 + k12 + k21 + k22
        row = x(n) - x(k11 + k12) - x(k21 + k22)
        col = x(n) - x(k11 + k21) - x(k12 + k22)
        mat = x(n) - x(k11) - x(k12) - x(k21) - x(k22)
        return float(2 * (row + col - mat))


def llr_bound(n):
    """|fp64 LLR - exact| <= 32 ulp(1) * N ln N: the entropies are O(N ln N) and cancel."""
    return 32 * 2.0 ** -53 * n * math.log(max(n, 2))


def _random_tables(rng, count):
    out = []
    for _ in range(count):
        n = int(math.exp(rng.uniform(math.log(4), math.log(2 ** 31 - 1))))
        ra = int(rng.integers(1, n))
        cb = int(rng.integers(1, n))
        lo, hi = max(0, ra + cb - n), min(ra, cb)
        k11 = int(rng.integers(lo, hi + 1))
        out.append((k11, ra - k11, cb - k11, n - ra - cb + k11))
    return out


def test_oracle_llr_against_50_digit_reference(orc):
    from conftest import load_golden
    rng = np.random.default_rng(31)
    tables = [tuple(t[:4]) for t in load_golden("llr_kats.json")["kats"]] + _random_tables(rng, 1500)
    # the recommender's side of the table: tiny k11 next to a huge N, where the cancellation is worst
    for _ in range(500):
        n = int(rng.integers(2 ** 20, 2 ** 31 - 1))
        ra, cb = int(rng.integers(1, 5000)), int(rng.integers(1, 5000))
        k11 = int(rng.integers(1, min(ra, cb) + 1))
        tables.append((k11, ra - k11, cb - k11, n - ra - cb + k11))
    for t in tables:
        n = sum(t)
        exact = llr_exact(*t)
        assert exact >= -llr_bound(n), t
        for flags in (0, orc.FLAG_ENTROPY_VARARGS):
            got = orc.llr(*t, flags)
            assert abs(got - exact) <= llr_bound(n), (t, flags, got, exact)


# ---- GPU ------------------------------------------------------------------------------------------------------------------------
def _optin():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def _check(orc, ctx, mats, params, seed, tag):
    ref = oracle_train(orc, mats, params, seed)
    got = ctx.train_csr(mats, params, seed=seed)
    assert_indicators_equal(ref, got, tag)
    _no_duplicate_columns(got)
    return got


@functools.lru_cache(maxsize=1)
def _workloads():
    return {"hashed": structured(HASHED_SHAPES), "hashed-spread": structured(HASHED_SHAPES, spread=True, seed=3),
            "dense": structured(DENSE_SHAPES)}


@pytest.mark.gpu
@pytest.mark.parametrize("k", K_SWEEP)
def test_top_k_sweep_under_candidate_pressure(orc, ctx, k):
    loads = _workloads()
    for c, _, _ in bins(k, loads["hashed"][1][1], _optin()):
        assert invariant_ok(c, k), c
    for name, mats in loads.items():
        _check(orc, ctx, mats, [(10 ** 6, k, None)] * 2, 5, f"{name} k={k}")


@pytest.mark.gpu
@pytest.mark.parametrize("k", K_DOWNSAMPLED)
def test_top_k_sweep_downsampled(orc, ctx, k):
    for name, mats in _workloads().items():
        _check(orc, ctx, mats, [(500, k, None)] * 2, 6, f"{name} m=500 k={k}")


@pytest.mark.gpu
def test_kept_llr_against_50_digit_reference(ctx):
    loads = _workloads()
    for name, k in (("hashed-spread", 300), ("hashed-spread", 2048), ("hashed", 64)):
        mats = loads[name]
        n = mats[0][0]
        got = ctx.train_csr(mats, [(10 ** 6, k, None)] * 2, seed=1)
        a, b = mats
        ra = np.bincount(a[3], minlength=a[1])
        cb = np.bincount(b[3], minlength=b[1])
        rb, re_, nc, rp, ci, ll, cn = got[1]
        tol = llr_bound(n)
        checked = 0
        for r in range(len(rp) - 1):
            exact = []
            for j in range(rp[r], rp[r + 1]):
                k11, colb = int(cn[j]), int(cb[ci[j]])
                e = llr_exact(k11, int(ra[r]) - k11, colb - k11, n - int(ra[r]) - colb + k11)
                assert abs(ll[j] - e) <= tol, (name, k, r, j, ll[j], e)
                exact.append(e)
            # a cell ranked below another never has a true LLR larger by more than twice the bound
            if exact:
                assert (np.array(exact) <= np.minimum.accumulate(exact) + 2 * tol).all(), (name, k, r)
            checked += len(exact)
        assert checked > 1000


@pytest.mark.gpu
def test_min_llr_exact_boundary(orc, ctx):
    mats = structured(HASHED_SHAPES, spread=True, seed=3)
    k = 50
    base = ctx.train_csr(mats, [(10 ** 6, k, None)] * 2, seed=2)
    ref = oracle_train(orc, mats, [(10 ** 6, k, None)] * 2, 2)
    rp, ci, ll = base[1][3], base[1][4], base[1][5]
    r = int(np.argmax(_row_works(mats)[:len(rp) - 1] == 4096))     # a 64 x 64 row: threshold and dominance filter active
    j = int(rp[r]) + k // 2
    v = float(ll[j])
    assert ref[1].llr[j] == v and ref[1].col_idx[j] == ci[j]          # the device value is the oracle's, bit for bit
    for thr, kept in ((v, True), (float(np.nextafter(v, np.inf)), False)):
        params = [(10 ** 6, k, None), (10 ** 6, k, thr)]
        got = _check(orc, ctx, mats, params, 2, f"minLLR={thr!r}")
        row = got[1][4][got[1][3][r]:got[1][3][r + 1]]
        assert (int(ci[j]) in row) == kept, (thr, kept)
        assert (got[1][5] >= thr).all()


@pytest.mark.gpu
def test_packed_word_count_edges(orc, ctx):
    # hashed tables, 3M columns: 22 key bits + 10 count bits.  A pair that co-occurs 1023 times fills the count field
    # without carrying into the key; 1024 co-occurrences cannot be represented and are refused.
    for hot, ok in ((1023, True), (1024, False)):
        nu, ib = 6000, 3_000_000
        rng = np.random.default_rng(hot)
        a_rows = [[0] if u < hot else [1 + int(u % 7)] for u in range(nu)]
        b_rows = [sorted({ib - 1} | set(rng.integers(0, ib - 1, 4).tolist())) if u < hot
                  else sorted(set(rng.integers(0, ib - 1, 4).tolist())) for u in range(nu)]
        mats = [_csr(a_rows, 8), _csr(b_rows, ib)]
        params = [(10 ** 6, 50, None)] * 2
        if ok:
            got = _check(orc, ctx, mats, params, 1, f"3M columns, k11={hot}")
            rp, ci, cn = got[1][3], got[1][4], got[1][6]
            assert ci[rp[0]] == ib - 1 and cn[rp[0]] == hot
        else:
            with pytest.raises(ur.CcoError) as e:
                ctx.train_csr(mats, params, seed=1)
            assert e.value.status == -6
    # dense 1024-bin table, 40000 columns: 16 key bits + 16 count bits -> 65535 co-occurrences of one pair
    for hot, ok in ((65535, True), (65536, False)):
        nu, ib = hot + 3000, 40_000
        rng = np.random.default_rng(hot)
        a_rows = [[0] if u < hot else [1] for u in range(nu)]
        b_rows = [sorted({ib - 1} | set(rng.integers(0, 2000, 2).tolist())) if u < hot
                  else sorted(set(rng.integers(0, ib - 1, 3).tolist())) for u in range(nu)]
        mats = [_csr(a_rows, 2), _csr(b_rows, ib)]
        params = [(10 ** 6, 50, None)] * 2
        if ok:
            got = _check(orc, ctx, mats, params, 1, f"40000 columns, k11={hot}")
            rp, ci, cn = got[1][3], got[1][4], got[1][6]
            assert ci[rp[0]] == ib - 1 and cn[rp[0]] == hot
        else:
            with pytest.raises(ur.CcoError) as e:
                ctx.train_csr(mats, params, seed=1)
            assert e.value.status == -6


@pytest.mark.gpu
def test_level1_cut_histogram_edge(orc, ctx):
    # The level-1 cut runs on rows of work < 65536, which bounds its u16 bins.  Every cell here has k11 == 1 and cb == 1,
    # so all of a pass's cells land in one bin: 40000 cells in one dense pass (the fullest a bin gets in one pass),
    # work 65535 (the largest row with the cut on, hashed, multi-pass) and 65536 (cut off).
    for ra, d in ((160, 250), (255, 257), (256, 256)):
        mats = structured([(ra, d), (2, 30)], n_extra=2_000_000)
        assert _row_works(mats)[0] == ra * d
        for k in (50, 600):
            got = _check(orc, ctx, mats, [(10 ** 6, k, None)] * 2, 1, f"w={ra * d} k={k}")
            rp, ci = got[1][3], got[1][4]
            assert np.array_equal(ci[rp[0]:rp[1]], np.arange(k))        # exact LLR ties: the k lowest columns


@pytest.mark.gpu
def test_cooccurrence_counts_through_every_bin(ctx):
    # debug_cooccurrence runs k_rows with every cell emitted at k = 1, so the warp-owned bins are on
    import scipy.sparse as sp
    for name, mats in _workloads().items():
        a, b = mats
        A = sp.csr_matrix((np.ones(len(a[3]), np.int64), a[3], a[2]), shape=(a[0], a[1]))
        B = sp.csr_matrix((np.ones(len(b[3]), np.int64), b[3], b[2]), shape=(b[0], b[1]))
        want = (A.T @ B).tocsr()
        want.sort_indices()
        rp, ci, cn = ctx.debug_cooccurrence(a, b)
        got = sp.csr_matrix((cn.astype(np.int64), ci, rp), shape=want.shape)
        got.sort_indices()
        assert np.array_equal(got.indptr, want.indptr), name
        assert np.array_equal(got.indices, want.indices), name
        assert np.array_equal(got.data, want.data), name
