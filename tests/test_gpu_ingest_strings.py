"""SURVEY.md 8f-1 from raw id strings: cco_ingest_strings / preparator.prepare_on_device against the host mirror
preparator.prepare (dictionaries and binary CSR element for element), against cco_ingest on tokens computed with numpy,
end to end into the Elasticsearch bulk body, and against the oracle's train."""
import numpy as np
import pytest

import universal_recommender_b200 as ur
from conftest import load_golden, prepared_from_fixture
from universal_recommender_b200 import _native as N
from universal_recommender_b200 import preparator

HOSTILE = ["", "a", "ab", "abc", "\x00", "a\x00", "\x00a", "\x00\x00", '"', "\\", "\n", '\\"', 'x"y\\z\n', "\t\r\x01\x1f",
           "\u00e9", "e\u0301", "日本語", "日本", "😀", "😀😀", "\x7f", "\u0080", "￿", "a b"]
ALPHABET = list("abxyz019") + ['"', "\\", "\n", "\x00", "é", "ß", "日", "😀", "\x7f", "\x01", " "]


def id_pool(rng, n):
    out, seen = [], set()
    for s in HOSTILE:
        out.append(s)
        seen.add(s)
    while len(out) < n:
        s = "".join(rng.choice(ALPHABET, int(rng.integers(0, 41))))
        if s not in seen:
            seen.add(s)
            out.append(s)
    return out


def hostile_actions(seed=11, sizes=(20_000, 15_000, 10_000)):
    """3 event types with Zipf users and items over hostile ids.  Item strings are shared with the user space and across
    types; the secondary types also see users the primary type never has."""
    rng = np.random.default_rng(seed)
    base = id_pool(rng, 3000)
    actions = []
    for t, n in enumerate(sizes):
        users = base[:1500] if t == 0 else base[:1800]
        items = base[:24] + base[500 + 300 * t:1700 + 300 * t]
        u = (rng.zipf(1.3, n) - 1) % len(users)
        i = (rng.zipf(1.2, n) - 1) % len(items)
        actions.append((f"ev{t}", [(users[a], items[b]) for a, b in zip(u, i)]))
    return actions


def assert_same(host, dev):
    assert [n for n, _ in host] == [n for n, _ in dev]
    for (_, h), (_, d) in zip(host, dev):
        assert list(h.row_ids.inverse) == list(d.row_ids.inverse)
        assert list(h.column_ids.inverse) == list(d.column_ids.inverse)
        assert (h.n_rows, h.n_cols) == (d.n_rows, d.n_cols)
        assert np.array_equal(h.row_ptr, d.row_ptr) and np.array_equal(h.col_idx, d.col_idx)


def decimal_column(prefix: bytes, v: np.ndarray):
    """ids prefix + decimal(v) (no leading zeros) as (offsets, bytes), built in numpy"""
    v = np.asarray(v, dtype=np.int64)
    w = 19
    digits = (v[:, None] // (10 ** np.arange(w - 1, -1, -1, dtype=np.int64))) % 10
    nd = np.maximum(1, np.floor(np.log10(np.maximum(v, 1))).astype(np.int64) + 1)
    keep = np.arange(w)[None, :] >= (w - nd)[:, None]
    mat = np.concatenate([np.broadcast_to(np.frombuffer(prefix, np.uint8), (len(v), len(prefix))),
                          (digits + 48).astype(np.uint8)], axis=1)
    mask = np.concatenate([np.ones((len(v), len(prefix)), bool), keep], axis=1)
    off = np.zeros(len(v) + 1, dtype=np.int64)
    np.cumsum(len(prefix) + nd, out=off[1:])
    return off, mat[mask]


def test_encode_ids_round_trips_hostile_ids():
    """CPU: the vectorised (offsets, bytes) encoder of prepare_on_device"""
    ids = HOSTILE + id_pool(np.random.default_rng(3), 500) + ["x" * 5000, "\U0010ffff", "߿ࠀ"]
    off, data = preparator.encode_ids(ids)
    assert off.dtype == np.int64 and data.dtype == np.uint8 and off[0] == 0 and off[-1] == len(data)
    blob = data.tobytes()
    assert [blob[a:b].decode("utf-8") for a, b in zip(off[:-1], off[1:])] == ids
    off0, data0 = preparator.encode_ids([])
    assert list(off0) == [0] and len(data0) == 0


def test_decimal_column_helper():
    """CPU: the numpy id builder of the scale test"""
    v = np.array([0, 7, 10, 99, 123456789, 10 ** 12])
    off, data = decimal_column(b"u", v)
    blob = data.tobytes()
    assert [blob[a:b].decode() for a, b in zip(off[:-1], off[1:])] == [f"u{x}" for x in v]


@pytest.mark.gpu
@pytest.mark.parametrize("short_hash", [False, True])
@pytest.mark.parametrize("min_ev", [None, 1, 3])
def test_matches_host_mirror(ctx, min_ev, short_hash, monkeypatch):
    actions = hostile_actions()
    host = preparator.prepare(actions, min_ev)
    if short_hash:   # every grouping goes through the exact (collision) pass
        orig = ctx.ingest_strings
        monkeypatch.setattr(ctx, "ingest_strings", lambda types, m=0, flags=0: orig(types, m, flags | N.FLAG_INGEST_SHORT_HASH))
    dev, ds = preparator.prepare_on_device(ctx, actions, min_ev)
    try:
        assert_same(host, dev)
        assert len(host[0][1].row_ids) > 100 and all(d.nnz > 0 for _, d in host)
    finally:
        ctx.free_dataset(ds)


@pytest.mark.gpu
@pytest.mark.parametrize("short_hash", [False, True])
def test_one_long_id_among_many_short(ctx, short_hash):
    """a 1 MiB id among 200K short ones (a warp hashes, compares and copies it), plus a second long id that differs only
    in its last byte"""
    rng = np.random.default_rng(4)
    big = "L" * (1 << 20)
    big2 = big[:-1] + "M"
    n = 200_000
    users = [f"u{x}" for x in (rng.zipf(1.3, n) - 1) % 30_000]
    items = [f"i{x}" for x in (rng.zipf(1.2, n) - 1) % 8_000]
    users[777] = big
    users[150_000] = big
    items[5] = big2
    items[6] = big
    items[100_000] = big
    actions = [("buy", list(zip(users, items))), ("view", list(zip(users[::-1], items)))]
    host = preparator.prepare(actions, None)
    flags = N.FLAG_INGEST_SHORT_HASH if short_hash else 0
    types = [(*preparator.encode_ids(u), *preparator.encode_ids(i)) for u, i in ((users, items), (users[::-1], items))]
    ds, user_ids, item_ids = ctx.ingest_strings(types, 0, flags)
    try:
        assert user_ids == list(host[0][1].row_ids.inverse)
        for t in range(2):
            assert item_ids[t] == list(host[t][1].column_ids.inverse)
            nr, nc, rp, ci = ctx.dataset_matrix(ds, t)
            assert np.array_equal(rp, host[t][1].row_ptr) and np.array_equal(ci, host[t][1].col_idx)
    finally:
        ctx.free_dataset(ds)


def _first_rank(values):
    """distinct values ranked by first appearance: (distinct in that order, rank of each element)"""
    uq, first, inv = np.unique(values, return_index=True, return_inverse=True)
    order = np.argsort(first, kind="stable")
    rank = np.empty(len(uq), dtype=np.int64)
    rank[order] = np.arange(len(uq))
    return uq[order], rank[inv.ravel()]


@pytest.mark.gpu
@pytest.mark.parametrize("min_ev", [0, 3])
def test_scale_against_integer_ingest(ctx, min_ev):
    """5M events over 2 types: the matrices equal cco_ingest on tokens numpy computes, the dictionaries follow the
    contract's order"""
    rng = np.random.default_rng(8)
    n_users, n_items = 300_000, 60_000
    ev = [((rng.zipf(1.3, n) - 1) % n_users, (rng.zipf(1.2, n) - 1) % n_items) for n in (3_000_000, 2_000_000)]
    # users: first appearance among type 0, kept by primary event count
    u0 = ev[0][0]
    uq, urank = _first_rank(u0)
    cnt = np.bincount(urank, minlength=len(uq))
    kept = cnt >= max(min_ev, 1)
    want_users = uq[kept]
    P = len(uq)
    tokens, want_items = [], []
    for t, (u, i) in enumerate(ev):
        if t == 0:
            raw_u = urank
        else:   # secondary users: first-appearance rank of the same primary user, P for users type 0 never has
            srt = np.argsort(uq)
            pos = np.minimum(np.searchsorted(uq[srt], u), P - 1)
            raw_u = np.where(uq[srt][pos] == u, srt[pos], P)
        surv = (raw_u < P) & kept[np.minimum(raw_u, P - 1)]
        iq, irank = _first_rank(i[surv])
        raw_i = np.zeros(len(i), dtype=np.int32)
        raw_i[surv] = irank
        want_items.append(iq)
        tokens.append((raw_u.astype(np.int64), raw_i, len(iq)))
    ref_ds, _, _ = ctx.ingest(tokens, P + 1, min_ev)
    types = [(*decimal_column(b"user-", u), *decimal_column(f"item{t}-".encode(), i)) for t, (u, i) in enumerate(ev)]
    ds, user_ids, item_ids = ctx.ingest_strings(types, min_ev)
    try:
        assert user_ids == [f"user-{x}" for x in want_users]
        for t in range(2):
            assert item_ids[t] == [f"item{t}-{x}" for x in want_items[t]]
            got, ref = ctx.dataset_matrix(ds, t), ctx.dataset_matrix(ref_ds, t)
            assert got[:2] == ref[:2] == (len(want_users), len(want_items[t]))
            assert np.array_equal(got[2], ref[2]) and np.array_equal(got[3], ref[3])
    finally:
        ctx.free_dataset(ds)
        ctx.free_dataset(ref_ds)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["handmade.json", "item_sets.json", "movielens_sample.json"])
def test_fixtures_end_to_end_bulk_body(ctx, name):
    fx = load_golden(name)
    host = prepared_from_fixture(fx)
    actions = [(n, [(u, i) for (u, e, i) in fx["events"] if e == n]) for n in fx["event_names"]]
    actions = [(n, p) for n, p in actions if p]
    params = fx["params"][:len(host)]
    names = [n for n, _ in host]
    mats = [(d.n_rows, d.n_cols, d.row_ptr, d.col_idx) for _, d in host]
    _, h = ctx.train_csr(mats, params, 1, keep=True)
    try:
        want = ctx.format_es_bulk(h, names, host[0][1].column_ids.inverse, [d.column_ids.inverse for _, d in host])
    finally:
        ctx.free_result(h)
    dev, ds = preparator.prepare_on_device(ctx, actions, fx.get("min_events_per_user"))
    try:
        assert_same(host, dev)
        _, h = ctx.train_dataset(ds, params, 1, keep=True)
        try:
            got = ctx.format_es_bulk(h, names, dev[0][1].column_ids.inverse, [d.column_ids.inverse for _, d in dev])
        finally:
            ctx.free_result(h)
    finally:
        ctx.free_dataset(ds)
    assert got == want and len(got) > 0


def _check_small_train(orc, ctx):
    """the context still ingests and trains correctly"""
    actions = hostile_actions(seed=5, sizes=(3000, 2000))
    host = preparator.prepare(actions, None)
    dev, ds = preparator.prepare_on_device(ctx, actions, None)
    try:
        assert_same(host, dev)
        params = [(500, 20, None)] * 2
        got = ctx.train_dataset(ds, params, 3)
        ref = orc.train([orc.Csr(d.n_rows, d.n_cols, d.row_ptr, d.col_idx) for _, d in host], [orc.Params(*p) for p in params], 3)
        for g, r in zip(got, ref):
            assert np.array_equal(g[3], r.row_ptr) and np.array_equal(g[4], r.col_idx) and np.array_equal(g[6], r.count)
    finally:
        ctx.free_dataset(ds)


@pytest.mark.gpu
def test_edges(orc, ctx):
    e = lambda: (np.zeros(1, np.int64), np.zeros(0, np.uint8))
    ds, users, items = ctx.ingest_strings([(*e(), *e()), (*e(), *e())])        # no events at all
    assert users == [] and items == [[], []] and ctx.dataset_matrix(ds, 1)[:2] == (0, 0)
    ctx.free_dataset(ds)
    base = hostile_actions(seed=2, sizes=(4000, 3000))
    cases = [([base[0], ("empty", [])], None),                                   # an empty secondary type
             (base, 10 ** 6),                                                     # every user filtered out
             ([base[0], ("strangers", [(f"nobody-{k}", f"x{k % 7}") for k in range(500)])], 2)]
    for actions, min_ev in cases:
        host = preparator.prepare(actions, min_ev)
        dev, ds = preparator.prepare_on_device(ctx, actions, min_ev)
        try:
            assert_same(host, dev)
            if actions[1][0] == "strangers":                                      # users all unknown: n_rows users, 0 columns
                assert dev[1][1].n_rows == len(host[0][1].row_ids) > 0 and dev[1][1].n_cols == 0
                got = ctx.train_dataset(ds, [(500, 20, None)] * 2, 1)
                ref = orc.train([orc.Csr(d.n_rows, d.n_cols, d.row_ptr, d.col_idx) for _, d in host],
                                [orc.Params(500, 20, None)] * 2, 1)
                for g, r in zip(got, ref):
                    assert np.array_equal(g[3], r.row_ptr) and np.array_equal(g[4], r.col_idx)
        finally:
            ctx.free_dataset(ds)


@pytest.mark.gpu
def test_errors_leave_the_context_usable(orc, ctx):
    good = (np.array([0, 1, 3], np.int64), np.frombuffer(b"abc", np.uint8))
    bad_inputs = [
        [(np.array([0, 2, 1, 3], np.int64), np.frombuffer(b"abc", np.uint8), np.array([0, 1, 2, 3], np.int64),
          np.frombuffer(b"xyz", np.uint8))],                                                        # user offsets decrease
        [(*good, np.array([0, 2, 1], np.int64), np.frombuffer(b"xy", np.uint8))],                    # item offsets decrease
        [(*good, *good), (*good, np.array([0, 3, 2], np.int64), np.frombuffer(b"xyz", np.uint8))],  # in a secondary type
        [(np.array([1, 2, 3], np.int64), np.frombuffer(b"abc", np.uint8), *good)],                  # offsets[0] != 0
        [(*good, np.array([0, 1], np.int64), np.frombuffer(b"x", np.uint8))],                        # user.n != item.n
    ]
    for types in bad_inputs:
        with pytest.raises(ur.CcoInvalidArgument):
            ctx.ingest_strings(types)
        _check_small_train(orc, ctx)
    g = ur.CcoContext(devices=[0])
    try:
        with pytest.raises(ur.CcoError) as e:
            g.ingest_strings([(*good, *good)])
        assert e.value.status == N.E_UNSUPPORTED
    finally:
        g.close()
    _check_small_train(orc, ctx)


@pytest.mark.gpu
def test_train_parity_small_workload(orc, ctx):
    """synth.py's `small` stream as id strings: ingested on the device and trained, equal to the oracle's train on the
    host mirror's matrices"""
    import synth
    w = synth.make("small")
    per_type = w.n_events // w.n_types
    utab = synth.user_tables(w.n_users)
    actions = []
    for t in range(w.n_types):
        u, i = synth.events_for_type(w.n_users, w.n_items, per_type, t, (utab, synth.item_tables(w.n_items, t)))
        actions.append((f"t{t}", [(f"user-{a:010d}", f"item-{b:08d}") for a, b in zip(u.tolist(), i.tolist())]))
    host = preparator.prepare(actions, None)
    dev, ds = preparator.prepare_on_device(ctx, actions, None)
    try:
        assert_same(host, dev)
        got = ctx.train_dataset(ds, w.params, 7)
    finally:
        ctx.free_dataset(ds)
    ref = orc.train([orc.Csr(d.n_rows, d.n_cols, d.row_ptr, d.col_idx) for _, d in host], [orc.Params(*p) for p in w.params], 7)
    for g, r in zip(got, ref):
        assert np.array_equal(g[3], r.row_ptr) and np.array_equal(g[4], r.col_idx) and np.array_equal(g[6], r.count)
        assert np.allclose(g[5], r.llr, rtol=1e-6, atol=0)
