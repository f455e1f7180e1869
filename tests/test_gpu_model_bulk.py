"""The whole model document (URModel.save with recsModel "all", URAlgorithm.scala:351-367, 537-560): correlators, rank fields
and item properties joined by id string.
CPU: Double.toString of the ranks, the restatement oracle/model_oracle.py against a plain-dict restatement of
`fieldsRDD fullOuterJoin ranks` + groupAll on the handmade fixture, the ranking-params resolver.
GPU: cco_format_model_bulk byte for byte against the restatement (fixtures, end to end from id strings, random logs over
hostile ids with and without the short hash, 5M Zipf events), its invariant against cco_format_es_bulk, its errors."""
import json
from collections import Counter

import numpy as np
import pytest

from conftest import load_golden, prepared_from_fixture

NOW = 1_700_000_000_000          # a fixed "now" in epoch milliseconds
DAY = 86_400_000


def _docs(body: bytes):
    lines = body.decode("utf-8").split("\n")
    assert lines[-1] == "" and len(lines) % 2 == 1
    return [(json.loads(lines[i]), json.loads(lines[i + 1])) for i in range(0, len(lines) - 1, 2)]


def set_fragments():
    """the $set properties of the handmade data aggregated per item (a later $set of a property replaces it), each item's
    as JSON object members without braces"""
    props: dict = {}
    for item, name, value in load_golden("handmade_set.json")["set"]:
        props.setdefault(item, {})[name] = value
    return {item: ",".join(json.dumps(k) + ":" + json.dumps(v) for k, v in p.items()) for item, p in props.items()}, props


def handmade_events():
    """the handmade events with times: one minute apart, the last one a minute before NOW"""
    ev = load_golden("handmade.json")["events"]
    return [(e, i, NOW - (len(ev) - k) * 60_000) for k, (u, e, i) in enumerate(ev)]


def handmade_model(orc):
    fx = load_golden("handmade.json")
    prepared = prepared_from_fixture(fx)
    ref = orc.train([orc.Csr(d.n_rows, d.n_cols, d.row_ptr, d.col_idx) for _, d in prepared], [orc.Params(*p) for p in fx["params"]], 1)
    names = [ev for ev, _ in prepared]
    return fx, prepared, names, [(r.row_ptr, r.col_idx) for r in ref]


def default_params():
    from universal_recommender_b200.ur_algorithm import IndicatorParams, URAlgorithmParams
    return URAlgorithmParams(indicators=[IndicatorParams("purchase"), IndicatorParams("view"), IndicatorParams("category-pref")])


def rankings_for(ap, events, now=NOW):
    from universal_recommender_b200.ur_algorithm import resolve_rankings
    out = []
    for r in resolve_rankings(ap, now):
        sel = [(i, t) for e, i, t in events if e in r.eventNames]
        out.append((r.name, r.type, [i for i, _ in sel], np.array([t for _, t in sel], np.int64), r.start_ms, r.end_ms))
    return out


# ---- CPU -----------------------------------------------------------------------------------------------------------
def test_java_double():
    from oracle.model_oracle import java_double
    want = {0: "0.0", -3: "-3.0", 9999999: "9999999.0", 10 ** 7: "1.0E7", 12345678: "1.2345678E7", -8589934592: "-8.589934592E9",
            10 ** 10: "1.0E10", -10 ** 7: "-1.0E7", 2 ** 34 - 1: "1.7179869183E10", 120000000: "1.2E8"}
    for v, s in want.items():
        assert java_double(float(v)) == s.encode() and float(s) == v


@pytest.mark.parametrize("with_props", [False, True])
def test_oracle_handmade_matches_the_join_of_fields_and_ranks(orc, with_props):
    from oracle.model_oracle import model_bulk
    fx, prepared, names, inds = handmade_model(orc)
    a = prepared[0][1]
    rows = list(a.column_ids.inverse)
    frags, props = set_fragments()
    events = handmade_events()
    body = model_bulk(inds, names, rows, [d.column_ids.inverse for _, d in prepared], rankings_for(default_params(), events),
                      frags if with_props else None)
    # plain restatement: fieldsRDD fullOuterJoin ranks (getRanksRDD), then groupAll with the correlators and "id"
    pop = Counter(i for e, i, _ in events if e == "purchase")
    fields = props if with_props else {}
    joined: dict = {}
    for i in list(pop) + list(fields):
        joined.setdefault(i, {})
    for i, n in pop.items():
        joined[i]["popRank"] = float(n)
    for i, p in fields.items():
        joined[i].update(p)
    want = []
    for r, item in enumerate(rows):
        doc = {"id": item}
        for ev in names:
            doc[ev] = [x[0] for x in fx["oracle"]["indicators"][ev][item]]
        doc.update(joined.get(item, {}))
        want.append(doc)
    want += [{"id": i, **p} for i, p in joined.items() if i not in rows]
    docs = _docs(body)
    assert [d for _, d in docs] == want
    assert all(act == {"index": {"_id": d["id"]}} for act, d in docs)
    by_id = {d["id"]: d for _, d in docs}
    assert by_id["Galaxy"]["popRank"] == 8.0 and all(by_id["Galaxy"][ev] == [] for ev in names)
    if with_props:
        assert by_id["Surface"]["categories"] == ["Tablets", "Electronics", "Microsoft"] and by_id["Surface"]["defaultRank"] == 1.0
        assert by_id["Iphone 4"]["countries"] == ["United States", "Canada", "Estados Unidos Mexicanos"]
        assert by_id["Surface"]["popRank"] == 2.0
    else:
        assert by_id["Surface"] == {"id": "Surface", "popRank": 2.0}
        assert b'{"index":{"_id":"Surface"}}\n{"id":"Surface","popRank":2.0}\n' in body


def test_ranking_resolver():
    from universal_recommender_b200.ur_algorithm import (RankingParams, URAlgorithmParams, duration_seconds, resolve_rankings)
    ap = default_params()
    (r,) = resolve_rankings(ap, NOW)
    assert (r.name, r.type, r.eventNames, r.start_ms, r.end_ms) == ("popRank", "popular", ["purchase"], NOW - 3650 * DAY, NOW)
    ap2 = URAlgorithmParams.from_engine_json({"eventNames": ["buy", "view"], "rankings": [
        {"name": "t1", "type": "trending", "duration": "3 days"},
        {"type": "popular", "eventNames": ["view"], "offsetDate": "2017-01-02T00:00:00Z", "duration": "12 hours"},
        {"name": "t2", "type": "trending", "duration": "5 days"},
        {"name": "u", "type": "userDefined"}, {"name": "rnd", "type": "random"},
        {"name": "h", "type": "hot", "offsetDate": "not a date", "duration": "1.5 hours"}]})
    got = [(x.name, x.type, x.eventNames, x.start_ms, x.end_ms) for x in resolve_rankings(ap2, NOW)]
    jan2 = 1_483_315_200_000
    assert got == [("t1", "trending", ["buy"], NOW - 3 * DAY, NOW), ("popRank", "popular", ["view"], jan2 - DAY // 2, jan2),
                   ("h", "hot", ["buy"], NOW - 5_400_000, NOW)]
    assert isinstance(ap2.rankings[0], RankingParams)
    assert [duration_seconds(s) for s in ["3650 days", "1 d", "90 min", "10s", " 2   hours ", "1500 millis", "999 ms", "7 day"]] == \
        [315_360_000, 86_400, 5_400, 10, 7_200, 1, 0, 604_800]
    assert duration_seconds("100000 days") == 8_640_000_000 - 2 ** 33     # .toInt wraps
    for bad in ["3 fortnights", "days", "Inf"]:
        with pytest.raises(ValueError):
            duration_seconds(bad)


# ---- GPU -----------------------------------------------------------------------------------------------------------
HOSTILE_ALPHABET = ['"', "\\", "\t", "\n", "\x01", "é", "☃", "\U0001f600", "a", "B", "7", " ", "-", "/", "\x00"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["handmade.json", "item_sets.json", "movielens_sample.json"])
def test_no_rankings_no_properties_is_es_bulk(ctx, name):
    fx = load_golden(name)
    prepared = prepared_from_fixture(fx)
    mats = [(d.n_rows, d.n_cols, d.row_ptr, d.col_idx) for _, d in prepared]
    names = [ev for ev, _ in prepared]
    rows, cols = prepared[0][1].column_ids.inverse, [d.column_ids.inverse for _, d in prepared]
    _, h = ctx.train_csr(mats, fx["params"], 1, keep=True)
    try:
        want = ctx.format_es_bulk(h, names, rows, cols)
        assert ctx.format_model_bulk(h, names, rows, cols) == want and len(want) > 0
    finally:
        ctx.free_result(h)


@pytest.mark.gpu
def test_no_rankings_no_properties_is_es_bulk_with_hostile_ids(ctx):
    import synth
    import universal_recommender_b200 as ur
    w = synth.make("small")
    rng = np.random.default_rng(3)

    def ids(n, salt):
        out = ["".join(HOSTILE_ALPHABET[int(x)] for x in rng.integers(0, len(HOSTILE_ALPHABET), int(rng.integers(0, 9)))) + f"{salt}{i}"
               for i in range(n)]
        out[0] = ""
        return out
    row_ids = ids(w.n_items, "i")
    col_ids = [row_ids] + [ids(w.n_items, f"t{t}_") for t in range(1, w.n_types)]
    names = ["purchase", 'vi"ew', "category-pref"]
    _, h = ctx.train_csr(w.mats, w.params, 5, flags=ur.FLAG_RESULT_NO_COUNT | ur.FLAG_RESULT_NO_LLR, keep=True)
    try:
        assert ctx.format_model_bulk(h, names, row_ids, col_ids) == ctx.format_es_bulk(h, names, row_ids, col_ids)
    finally:
        ctx.free_result(h)


def _check_handmade(orc, ctx):
    """handmade end to end from id strings: prepare_on_device -> train_dataset(keep) -> format_model_bulk, equal to the
    restatement on the host mirror's model"""
    from oracle.model_oracle import model_bulk
    from universal_recommender_b200 import preparator
    fx, prepared, names, inds = handmade_model(orc)
    actions = [(n, [(u, i) for (u, e, i) in fx["events"] if e == n]) for n in fx["event_names"]]
    dev, ds = preparator.prepare_on_device(ctx, actions, fx["min_events_per_user"])
    frags, _ = set_fragments()
    rk = rankings_for(default_params(), handmade_events())
    try:
        _, h = ctx.train_dataset(ds, fx["params"], 1, keep=True)
        try:
            got = ctx.format_model_bulk(h, names, dev[0][1].column_ids.inverse, [d.column_ids.inverse for _, d in dev], rk, frags)
        finally:
            ctx.free_result(h)
    finally:
        ctx.free_dataset(ds)
    want = model_bulk(inds, names, prepared[0][1].column_ids.inverse, [d.column_ids.inverse for _, d in prepared], rk, frags)
    assert got == want
    return got


@pytest.mark.gpu
def test_handmade_end_to_end(orc, ctx):
    got = _check_handmade(orc, ctx)
    docs = {d["id"]: d for _, d in _docs(got)}
    assert docs["Surface"]["popRank"] == 2.0 and docs["Galaxy"]["popRank"] == 8.0 and "purchase" not in docs["Surface"]


def random_model(ctx, rng, n_rows=400, n_other=300):
    """a trained `tiny`-shaped model whose primary items are hostile ids, and a pool of other ids (never rows)"""
    import synth
    w = synth.make("tiny", n_items=n_rows)
    seen: set = set()
    pool = []
    while len(pool) < n_rows + n_other:
        s = "".join(HOSTILE_ALPHABET[int(x)] for x in rng.integers(0, len(HOSTILE_ALPHABET), int(rng.integers(0, 7))))
        if s not in seen:
            seen.add(s)
            pool.append(s)
    pool[n_rows + 5] = "L" * (1 << 20)            # one 1 MiB id, not a row
    rows, others = pool[:n_rows], pool[n_rows:]
    res, h = ctx.train_csr(w.mats, w.params, 3, keep=True)
    return w, rows, others, [(r[3], r[4]) for r in res], h


@pytest.mark.gpu
@pytest.mark.parametrize("short_hash", [False, True])
def test_random_logs_all_modes(ctx, short_hash):
    """popular, trending and hot together over logs that hit rows, extras and ids that are never present, with empty
    buckets; properties on rows, on extras and on ids with no rank, some empty"""
    from oracle.model_oracle import model_bulk
    from universal_recommender_b200 import _native as N
    rng = np.random.default_rng(21 + short_hash)
    w, rows, others, inds, h = random_model(ctx, rng)
    names = ["purchase", "view", 'c"at']
    try:
        space = rows + others
        end = NOW
        for case in range(4):
            rk = []
            for r, (mode, nm) in enumerate([("popular", "popRank"), ("trending", "trendRank"), ("hot", "hotRank")]):
                n = int(rng.integers(0, 3000))
                items = [space[int(x)] for x in (rng.zipf(1.3, n) - 1) % len(space)]
                start = end - int(rng.integers(3, 30)) * DAY
                t = rng.integers(start - 2 * DAY, end + DAY, n)
                if case == 1 and mode != "popular":       # the older bucket empty: trending / hot have nothing
                    t = np.maximum(t, start + (end - start) // 2)
                if case == 2 and mode == "hot":           # the middle third empty
                    th = (end - start) // 3
                    t = np.where((t >= start + th) & (t < start + 2 * th), start, t)
                if case == 3 and r == 0:
                    items, t = [], np.zeros(0, np.int64)  # a ranking without events
                rk.append((nm, mode, items, t.astype(np.int64), start, end))
            pids = list(dict.fromkeys(space[int(x)] for x in rng.integers(0, len(space), 120)))
            frags = [("" if k % 7 == 0 else json.dumps("p") + ":" + json.dumps(k)) for k in range(len(pids))]
            want = model_bulk(inds, names, rows, [rows, rows, rows], rk, (pids, frags))
            got = ctx.format_model_bulk(h, names, rows, [rows, rows, rows], rk, (pids, frags),
                                        flags=N.FLAG_INGEST_SHORT_HASH if short_hash else 0)
            assert got == want, case
            assert len(_docs(got)) >= len(rows)
    finally:
        ctx.free_result(h)


@pytest.mark.gpu
def test_five_million_zipf_events(ctx):
    """a 5M-event popular ranking over Zipf items as decimal id strings: popRank = np.bincount of the tokens, extras =
    exactly the tokens outside the row space, in order of first appearance"""
    import synth
    import universal_recommender_b200 as ur
    from test_gpu_ingest_strings import decimal_column
    w = synth.make("small")
    n_rows = w.n_items
    n = 5_000_000
    _, tok = synth.events_for_type(w.n_users, 2 * n_rows, n, 0)
    tok = tok.astype(np.int64)
    t = np.full(n, NOW - DAY, np.int64)
    t[::97] = NOW + 1                                   # outside [start, end)
    rows = [str(j) for j in range(n_rows)]
    _, h = ctx.train_csr(w.mats, w.params, 5, flags=ur.FLAG_RESULT_NO_COUNT | ur.FLAG_RESULT_NO_LLR, keep=True)
    try:
        body = ctx.format_model_bulk(h, ["a", "b", "c"], rows, [rows, rows, rows],
                                     [("popRank", "popular", decimal_column(b"", tok), t, NOW - 30 * DAY, NOW)])
    finally:
        ctx.free_result(h)
    inside = tok[t < NOW]
    cnt = np.bincount(inside, minlength=2 * n_rows)
    docs = _docs(body)
    ids = [int(d["id"]) for _, d in docs]
    assert ids[:n_rows] == list(range(n_rows))
    uq, first = np.unique(tok, return_index=True)               # first appearance among all the ranking's events
    keep = (uq >= n_rows) & (cnt[uq] > 0)
    assert ids[n_rows:] == [int(x) for x in uq[keep][np.argsort(first[keep], kind="stable")]]
    assert all(d.get("popRank", 0.0) == float(cnt[int(d["id"])]) for _, d in docs)
    assert sum(d.get("popRank", 0.0) for _, d in docs) == len(inside)


@pytest.mark.gpu
def test_errors_leave_the_context_usable(orc, ctx):
    import universal_recommender_b200 as ur
    from universal_recommender_b200 import _native as N
    w, rows, others, inds, h = random_model(ctx, np.random.default_rng(5), n_rows=50, n_other=20)
    names = ["purchase", "view", "cat"]
    cols = [rows] * 3
    one = lambda name="popRank", mode="popular", start=NOW - DAY, end=NOW: (name, mode, others[:3], np.full(3, NOW - 1), start, end)
    bad_off = (np.array([0, 2, 1, 3], np.int64), np.frombuffer(b"abc", np.uint8))
    from universal_recommender_b200.preparator import encode_ids
    r_off, r_bytes = encode_ids(rows)
    r_off = r_off.copy()
    r_off[11] = r_off[10] - 1                                          # 50 row ids whose offsets decrease once
    bad_rows = (r_off, r_bytes)
    invalid = [
        dict(row_ids=rows[:-1]),                                        # row_ids.n != rows
        dict(row_ids=rows[:-1] + [rows[0]]),                            # two equal row ids
        dict(rankings=[one(name=None)]),
        dict(rankings=[one(name="id")]),
        dict(rankings=[one(name="view")]),                               # an indicator name
        dict(rankings=[one(), one(mode="hot")]),                         # repeated
        dict(rankings=[one(start=NOW, end=NOW - 1)]),
        dict(rankings=[one(mode=7)]),
        dict(rankings=[("popRank", "popular", bad_off, np.zeros(3, np.int64), 0, 1)]),      # offsets decrease
        dict(properties=([others[0], others[1], others[0]], ["", "", ""])),                 # two equal property ids
        dict(properties=([rows[0], rows[0]], ["", ""])),                                    # equal property ids that are a row
        dict(properties=(bad_off, ["", "", ""])),
        dict(properties=(others[:3], bad_off)),
        dict(col_ids=[rows, bad_rows, rows]),
        dict(row_ids=bad_rows),
    ]
    try:
        for kw in invalid:
            args = dict(row_ids=rows, col_ids=cols, rankings=(), properties=None)
            args.update(kw)
            with pytest.raises(ur.CcoInvalidArgument):
                ctx.format_model_bulk(h, names, **args)
            _check_handmade(orc, ctx)
        L = ctx._L
        out, ln = N.C.c_void_p(), N.C.c_int64()
        keep: list = []
        rd = ctx._raw_dictionary(rows, keep)
        cds = (N.DictionaryRawT * 3)(*[ctx._raw_dictionary(rows, keep) for _ in range(3)])
        nm = (N.C.c_char_p * 3)(*[x.encode() for x in names])
        assert L.cco_format_model_bulk(ctx._h, h, 3, nm, N.C.byref(rd), cds, 0, None, N.C.byref(rd), None, 0, N.C.byref(out),
                                       N.C.byref(ln)) == N.E_INVALID_ARG                  # only one of prop_ids / prop_json
        with pytest.raises(ur.CcoError) as e:
            ctx.format_model_bulk(h, names, rows, cols, [one(name=f"r{k}") for k in range(4)])
        assert e.value.status == N.E_UNSUPPORTED
    finally:
        ctx.free_result(h)
    _check_handmade(orc, ctx)


@pytest.mark.gpu
def test_write_model(orc, ctx):
    """recsModel "collabFiltering" writes exactly format_es_bulk's bytes; "all" adds the default popRank"""
    from oracle.model_oracle import model_bulk
    from universal_recommender_b200.ur_algorithm import URAlgorithmParams, write_model
    fx, prepared, names, inds = handmade_model(orc)
    mats = [(d.n_rows, d.n_cols, d.row_ptr, d.col_idx) for _, d in prepared]
    rows, cols = prepared[0][1].column_ids.inverse, [d.column_ids.inverse for _, d in prepared]
    events = handmade_events()
    frags, _ = set_fragments()
    _, h = ctx.train_csr(mats, fx["params"], 1, keep=True)
    try:
        cf = URAlgorithmParams.from_engine_json({"indicators": [{"name": n} for n in names], "recsModel": "collabFiltering"})
        assert write_model(ctx, h, names, rows, cols, cf, events, frags, NOW) == ctx.format_es_bulk(h, names, rows, cols)
        al = URAlgorithmParams.from_engine_json({"indicators": [{"name": n} for n in names]})
        got = write_model(ctx, h, names, rows, cols, al, events, frags, NOW)
    finally:
        ctx.free_result(h)
    assert got == model_bulk(inds, names, rows, cols, rankings_for(default_params(), events), frags)


@pytest.mark.gpu
def test_group_context_formats_like_one_gpu(orc, ctx):
    import torch
    import universal_recommender_b200 as ur
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    fx, prepared, names, inds = handmade_model(orc)
    import synth
    w = synth.make("small")
    rows = [f"item-{j}" for j in range(w.n_items)]
    rng = np.random.default_rng(9)
    items = [rows[int(x)] if x < w.n_items else f"x{x}" for x in (rng.zipf(1.2, 50_000) - 1) % (2 * w.n_items)]
    rk = [("popRank", "popular", items, np.full(len(items), NOW - 1), NOW - DAY, NOW)]
    props = {rows[3]: '"a":1', "x77": '"b":2'}
    out = []
    for c in (ctx, ur.CcoContext(devices=[0, 1])):
        _, h = c.train_csr(w.mats, w.params, 5, keep=True)
        try:
            out.append(c.format_model_bulk(h, names[:3], rows, [rows] * 3, rk, props))
        finally:
            c.free_result(h)
        if c is not ctx:
            c.close()
    assert out[0] == out[1]
