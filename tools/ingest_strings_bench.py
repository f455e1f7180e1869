"""Throughput of cco_ingest_strings (Preparator.prepare from raw id strings on the device) at a synth.py shape, next to
the integer-tokenised cco_ingest of the same events (the floor) and the host mirror preparator.prepare on a named slice.

Events are synth.py's integer stream turned into id strings, in two formats:
  fixed     user-%010d / item-%08d
  variable  2..64 bytes with multi-byte UTF-8 (an injective spelling of the integer id plus filler), and one 1 MiB item
            id per type
The id columns live in pinned host memory (what the JNI shim hands over); the time is a host clock around the C call,
which includes the host->device copy of the columns and ends in a stream synchronise.  Prints one JSON line.

usage: python tools/ingest_strings_bench.py [--shape C3] [--warmup 1] [--repeat 3] [--host-slice 500000]"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import synth  # noqa: E402
import universal_recommender_b200 as ur  # noqa: E402
from universal_recommender_b200 import _native as N  # noqa: E402
from universal_recommender_b200 import preparator  # noqa: E402

SYMBOLS = ["0", "1", "2", "3", "4", "é", "ß", "ж", "日", "\U0001f600"]   # 1, 2, 3 and 4 UTF-8 bytes


def fixed_table(prefix: str, n: int, width: int):
    """id k -> prefix + k zero-padded to `width` digits: ([n, L] uint8, lengths)"""
    k = np.arange(n, dtype=np.int64)
    pre = np.frombuffer(prefix.encode(), np.uint8)
    digits = (k[:, None] // (10 ** np.arange(width - 1, -1, -1, dtype=np.int64))) % 10 + 48
    tab = np.concatenate([np.broadcast_to(pre, (n, len(pre))), digits.astype(np.uint8)], axis=1)
    return np.ascontiguousarray(tab), np.full(n, tab.shape[1], np.int64)


def variable_table(n: int, seed: int):
    """id k -> its 7 decimal digits spelled with SYMBOLS, '_', then 0.. 'x' up to a length drawn in [body + 1, 64]"""
    k = np.arange(n, dtype=np.int64)
    sym = [s.encode() for s in SYMBOLS]
    sb = np.zeros((10, 4), np.uint8)
    sl = np.array([len(s) for s in sym], np.int64)
    for d, s in enumerate(sym):
        sb[d, :len(s)] = np.frombuffer(s, np.uint8)
    digits = (k[:, None] // (10 ** np.arange(6, -1, -1, dtype=np.int64))) % 10
    body = np.concatenate([sb[digits].reshape(n, 28), np.full((n, 1), ord("_"), np.uint8)], axis=1)
    body_mask = np.concatenate([(np.arange(4)[None, None, :] < sl[digits][:, :, None]).reshape(n, 28), np.ones((n, 1), bool)], axis=1)
    body_len = body_mask.sum(axis=1)
    total = np.random.default_rng(seed).integers(body_len, 65)
    tab = np.full((n, 64), ord("x"), np.uint8)
    pos = np.cumsum(body_mask, axis=1) - 1
    tab[np.nonzero(body_mask)[0], pos[body_mask]] = body[body_mask]
    return tab, total


def column(ctx, tab, lens, v, long_at=None):
    """events v -> (offsets, bytes) in pinned memory; long_at: event whose id becomes a 1 MiB id"""
    ev_len = lens[v].copy()
    if long_at is not None:
        ev_len[long_at] = 1 << 20
    off = ctx.host_array(len(v) + 1, np.int64)
    off[0] = 0
    np.cumsum(ev_len, out=off[1:])
    data = ctx.host_array(int(off[-1]), np.uint8)
    step = 1 << 21
    for s in range(0, len(v), step):
        vv = v[s:s + step]
        rows = tab[vv]
        mask = np.arange(tab.shape[1])[None, :] < lens[vv][:, None]
        if long_at is not None and s <= long_at < s + step:
            mask[long_at - s] = False
        chunk = rows[mask]
        if long_at is not None and s <= long_at < s + step:
            a = int(off[long_at] - off[s])
            chunk = np.concatenate([chunk[:a], np.full(1 << 20, ord("L"), np.uint8), chunk[a:]])
        data[off[s]:off[s] + len(chunk)] = chunk
    return off, data


def dict_t(off, data):
    return N.DictionaryRawT(len(off) - 1, off.ctypes.data_as(C.POINTER(C.c_int64)), data.ctypes.data if len(data) else None)


def time_string_ingest(ctx, cols, warmup, repeat):
    L = ctx._L
    n = len(cols)
    ev = (N.StringEventsT * n)(*[N.StringEventsT(dict_t(*u), dict_t(*i)) for u, i in cols])
    times, sizes = [], None
    for r in range(warmup + repeat):
        user, items = N.DictionaryRawT(), (N.DictionaryRawT * n)()
        ds = C.c_void_p()
        t0 = time.perf_counter()
        N.check(L.cco_ingest_strings(ctx._h, n, ev, 0, 0, C.byref(user), items, C.byref(ds)))
        dt = time.perf_counter() - t0
        if r >= warmup:
            times.append(dt * 1e3)
        sizes = (user.n, [items[t].n for t in range(n)])
        for d in [user] + [items[t] for t in range(n)]:
            L.cco_host_free(ctx._h, C.cast(d.offsets, C.c_void_p))
            L.cco_host_free(ctx._h, d.bytes)
        L.cco_dataset_free(ds)
    return times, sizes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="C3")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--host-slice", type=int, default=500_000, help="events per type for the host preparator.prepare run")
    a = ap.parse_args()
    cfg = synth.CONFIGS[a.shape]
    n_users, n_items, n_types = cfg["n_users"], cfg["n_items"], cfg["n_types"]
    per_type = cfg["n_events"] // n_types
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    gpu = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 and smi.stdout.strip() else "unknown"
    ctx = ur.CcoContext(device=0)
    utab = synth.user_tables(n_users)
    events = [synth.events_for_type(n_users, n_items, per_type, t, (utab, synth.item_tables(n_items, t))) for t in range(n_types)]
    out = dict(tool="ingest_strings_bench", shape=a.shape, n_users=n_users, n_items=n_items, n_events=per_type * n_types,
               n_types=n_types, gpu=gpu, warmup=a.warmup, repeat=a.repeat,
               timing="host clock around the C call, which includes the H2D of the pinned id columns and ends in a synchronise")
    formats = {"fixed": (fixed_table("user-", n_users, 10), [fixed_table("item-", n_items, 8)] * n_types, False),
               "variable": (variable_table(n_users, 1), [variable_table(n_items, 10 + t) for t in range(n_types)], True)}
    for fmt, (ut, its, long_id) in formats.items():
        cols = [(column(ctx, *ut, u), column(ctx, *its[t], i, per_type // 2 if long_id else None)) for t, (u, i) in enumerate(events)]
        id_bytes = int(sum(len(u[1]) + len(i[1]) for u, i in cols))
        times, sizes = time_string_ingest(ctx, cols, a.warmup, a.repeat)
        med = float(np.median(times))
        out[fmt] = dict(ms_median=round(med, 3), ms_all=[round(x, 3) for x in times], events_per_s=round(per_type * n_types / med * 1e3),
                        id_bytes_in=id_bytes, offset_bytes_in=16 * per_type * n_types, n_user_dict=sizes[0], n_item_dicts=sizes[1])
        for u, i in cols:
            for arr in (*u, *i):
                ctx.host_free(arr)
    # the floor: the same events already tokenised, through cco_ingest
    toks = []
    for u, i in events:
        pu, pi = ctx.host_array(len(u), np.int64), ctx.host_array(len(i), np.int32)
        pu[:], pi[:] = u, i
        toks.append((pu, pi, n_items))
    L = ctx._L
    ev = (N.EventsT * n_types)(*[N.EventsT(len(u), u.ctypes.data_as(C.POINTER(C.c_int64)), i.ctypes.data_as(C.POINTER(C.c_int32)), ni)
                                 for u, i, ni in toks])
    umap = np.zeros(n_users, np.int32)
    imaps = [np.zeros(n_items, np.int32) for _ in range(n_types)]
    mp = (C.POINTER(C.c_int32) * n_types)(*[m.ctypes.data_as(C.POINTER(C.c_int32)) for m in imaps])
    itimes = []
    for r in range(a.warmup + a.repeat):
        ds = C.c_void_p()
        t0 = time.perf_counter()
        N.check(L.cco_ingest(ctx._h, n_types, ev, n_users, 0, umap.ctypes.data_as(C.POINTER(C.c_int32)), mp, C.byref(ds)))
        dt = time.perf_counter() - t0
        if r >= a.warmup:
            itimes.append(dt * 1e3)
        L.cco_dataset_free(ds)
    out["integer_ingest"] = dict(ms_median=round(float(np.median(itimes)), 3), ms_all=[round(x, 3) for x in itimes],
                                 input="pinned int64 user / int32 item arrays (cco_ingest range-checks every id on the host)")
    # the host mirror on a slice: fixed-width ids, the first host_slice events of every type
    ns = min(a.host_slice, per_type)
    actions = [(f"t{t}", [(f"user-{x:010d}", f"item-{y:08d}") for x, y in zip(u[:ns].tolist(), i[:ns].tolist())])
               for t, (u, i) in enumerate(events)]
    t0 = time.perf_counter()
    preparator.prepare(actions, None)
    out["host_prepare"] = dict(slice=f"first {ns} events of each of the {n_types} types, fixed-width ids", events=ns * n_types,
                               ms=round((time.perf_counter() - t0) * 1e3, 1))
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
