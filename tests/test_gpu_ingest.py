"""SURVEY.md 8f-1 on the device: cco_ingest against the oracle's ingest restatement (dictionaries and binary CSR
bit-exact), and a train from the ingested, HBM-resident dataset against the oracle end to end."""
import numpy as np
import pytest

import universal_recommender_b200 as ur

pytestmark = pytest.mark.gpu


def random_events(rng, n_users, n_items, n_events, n_types):
    return [((rng.zipf(1.4, n_events) - 1) % n_users, ((rng.zipf(1.2, n_events) - 1) % n_items).astype(np.int32), n_items)
            for _ in range(n_types)]


@pytest.mark.parametrize("min_ev", [0, 3])
def test_ingest_matches_oracle(orc, ctx, min_ev):
    rng = np.random.default_rng(5)
    events = random_events(rng, 5000, 800, 60_000, 3)
    ds, user_map, item_maps = ctx.ingest(events, 5000, min_ev)
    o_user_map, o_res = orc.ingest(events, 5000, min_ev)
    assert np.array_equal(user_map, o_user_map)
    mats = []
    for t, (csr, imap) in enumerate(o_res):
        assert np.array_equal(item_maps[t], imap)
        nr, nc, rp, ci = ctx.dataset_matrix(ds, t)
        assert (nr, nc) == (csr.n_rows, csr.n_cols)
        assert np.array_equal(rp, csr.row_ptr) and np.array_equal(ci, csr.col_idx)
        mats.append(csr)
    params = [(500, 20, None)] * 3
    got = ctx.train_dataset(ds, params, seed=9, flags=ur.FLAG_ASSUME_CANONICAL)
    ref = orc.train(mats, [orc.Params(*p) for p in params], 9)
    for g, r in zip(got, ref):
        assert np.array_equal(g[3], r.row_ptr) and np.array_equal(g[4], r.col_idx) and np.array_equal(g[6], r.count)
        assert np.allclose(g[5], r.llr, rtol=1e-6, atol=0)
    ctx.free_dataset(ds)


def test_ingest_edge_cases(orc, ctx):
    e = lambda: (np.zeros(0, np.int64), np.zeros(0, np.int32), 4)
    ds, um, im = ctx.ingest([e(), e()], 6, 0)                      # no events at all
    assert (um == -1).all() and ctx.dataset_matrix(ds, 0)[0] == 0
    ctx.free_dataset(ds)
    with pytest.raises(ur.CcoInvalidArgument):
        ctx.ingest([(np.array([7]), np.array([0], dtype=np.int32), 1)], 3, 0)


@pytest.mark.parametrize("name", ["tiny", "small", "C3-tenth"])
def test_device_generator_matches_numpy_twin(ctx, name, monkeypatch):
    """cco_synth_ingest (events generated and ingested in HBM) and synth.py's numpy path give the same matrices bit for bit:
    same counter-based stream, same Preparator semantics (user dictionary from the primary events, dedup)."""
    import synth
    monkeypatch.setenv("CCO_SYNTH_CACHE", "0")     # a cached file from an earlier run is not the numpy path under test
    host = synth.make(name)
    dev = synth.make(name, ctx=ctx)
    assert host.n_users == dev.n_users
    for (nr, nc, rp, ci), (dnr, dnc, drp, dci) in zip(host.mats, dev.mats):
        assert (nr, nc) == (dnr, dnc)
        assert np.array_equal(rp, drp) and np.array_equal(ci, dci)


def test_device_generator_min_events_filter(ctx):
    import synth
    host = synth.make("small", min_events_per_user=12)
    dev = synth.make("small", ctx=ctx, min_events_per_user=12)
    assert host.n_users == dev.n_users < 20_000
    for h, d in zip(host.mats, dev.mats):
        assert np.array_equal(h[2], d[2]) and np.array_equal(h[3], d[3])
