"""Times the model document writers at the C3 shape (1M users, 100K items, 50M events over 4 types, k = 50).

The model comes from synth_dataset + train_dataset(keep=True); every id is a decimal string.  The rankings run over the
12.5M primary events (the synthetic stream's items, times spread over 30 days); 100K property fragments of about 100 bytes
go to the primary items.  Timed, each as the median of --reps calls after --warmup calls (host clock around the C call,
which ends in a stream synchronise; the id columns are encoded once, before the timer):
  1. cco_format_es_bulk
  2. cco_format_model_bulk, no rankings, no properties (its bytes must equal 1)
  3. the default ranking: popRank, popular over the primary events
  4. popular + trending + hot, and the properties
  5. the CPU restatement oracle/model_oracle.py on a named slice (first --oracle-rows rows, --oracle-events events), once
Prints one JSON line with the device name and power limit read in the same run.
usage: python tools/model_bulk_bench.py [--reps 5] [--warmup 1]"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DAY = 86_400_000


def decimal_ids(v: np.ndarray):
    """decimal(v) without leading zeros as (offsets int64[n + 1], bytes uint8[]), built in numpy"""
    v = np.asarray(v, dtype=np.int64)
    w = 19
    digits = (v[:, None] // (10 ** np.arange(w - 1, -1, -1, dtype=np.int64))) % 10
    nd = np.maximum(1, np.floor(np.log10(np.maximum(v, 1))).astype(np.int64) + 1)
    keep = np.arange(w)[None, :] >= (w - nd)[:, None]
    off = np.zeros(len(v) + 1, dtype=np.int64)
    np.cumsum(nd, out=off[1:])
    return off, (digits + 48).astype(np.uint8)[keep]


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:   # the numbers still stand with the device name from CUDA
        import torch
        return torch.cuda.get_device_name(0), f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--oracle-rows", type=int, default=2000)
    ap.add_argument("--oracle-events", type=int, default=200_000)
    a = ap.parse_args()

    import synth
    import universal_recommender_b200 as ur
    from universal_recommender_b200 import _native as N
    ctx = ur.CcoContext(device=0)
    L = ctx._L
    w = synth.make("C3", ctx=ctx, keep_dataset=True)
    res, h = ctx.train_dataset(w.dataset, w.params, 7, flags=ur.FLAG_RESULT_NO_COUNT | ur.FLAG_RESULT_NO_LLR, keep=True)
    ctx.free_dataset(w.dataset)
    n_items = w.n_items
    per_type = w.n_events // w.n_types
    _, prim = synth.events_for_type(w.n_users, n_items, per_type, 0)      # the primary stream's items, as on the device
    now = 1_700_000_000_000
    times = np.random.default_rng(1).integers(now - 30 * DAY, now, per_type).astype(np.int64)

    keep: list = []
    rows = decimal_ids(np.arange(n_items))
    names = [f"event{t}" for t in range(w.n_types)]
    d_rows = ctx._raw_dictionary(rows, keep)
    d_cols = (N.DictionaryRawT * w.n_types)(*[ctx._raw_dictionary(rows, keep) for _ in range(w.n_types)])
    d_names = (C.c_char_p * w.n_types)(*[x.encode() for x in names])
    d_prim = ctx._raw_dictionary(decimal_ids(prim), keep)
    frags = [f'"categories":["cat-{j % 50}","sub-{j % 7}"],"available":"2017-01-{1 + j % 28:02d}T00:00:00Z","defaultRank":{j}.0'
             for j in range(n_items)]
    d_pid, d_pjs = ctx._raw_dictionary(rows, keep), ctx._raw_dictionary(frags, keep)
    tp = times.ctypes.data_as(C.POINTER(C.c_int64))
    nb = [x.encode() for x in ("popRank", "trendRank", "hotRank")]
    rk = (N.RankingT * 3)(*[N.RankingT(nb[m], m, 0, now - 30 * DAY, now, d_prim, tp) for m in range(3)])

    def es_bulk():
        out, ln = C.c_void_p(), C.c_int64()
        N.check(L.cco_format_es_bulk(ctx._h, h, w.n_types, d_names, C.cast(C.pointer(d_rows), C.POINTER(N.DictionaryT)),
                                     C.cast(d_cols, C.POINTER(N.DictionaryT)), C.byref(out), C.byref(ln)))
        return out, ln.value

    def model(n_rank, props):
        out, ln = C.c_void_p(), C.c_int64()
        N.check(L.cco_format_model_bulk(ctx._h, h, w.n_types, d_names, C.byref(d_rows), d_cols, n_rank, rk,
                                        C.byref(d_pid) if props else None, C.byref(d_pjs) if props else None, 0,
                                        C.byref(out), C.byref(ln)))
        return out, ln.value

    cases = [("es_bulk", es_bulk), ("model_bulk_no_rankings", lambda: model(0, False)),
             ("model_bulk_popular", lambda: model(1, False)), ("model_bulk_3_rankings_props", lambda: model(3, True))]
    result = {"shape": "C3", "n_rows": n_items, "ranking_events": per_type, "n_properties": n_items,
              "fragment_bytes_mean": round(float(np.mean([len(f) for f in frags])), 1)}
    first_bytes = {}
    for name, fn in cases:
        ms = []
        for k in range(a.warmup + a.reps):
            t0 = time.perf_counter()
            out, ln = fn()
            t1 = time.perf_counter()
            if k == 0:
                first_bytes[name] = C.string_at(out.value, ln) if name in ("es_bulk", "model_bulk_no_rankings") else None
            L.cco_host_free(ctx._h, out)
            if k >= a.warmup:
                ms.append((t1 - t0) * 1e3)
        result[name] = {"median_ms": round(statistics.median(ms), 2), "min_ms": round(min(ms), 2), "max_ms": round(max(ms), 2),
                        "out_bytes": ln}
        print(f"[model_bulk_bench] {name}: median {statistics.median(ms):.2f} ms over {a.reps}, {ln} bytes", flush=True)
    result["no_rankings_equals_es_bulk"] = first_bytes["es_bulk"] == first_bytes["model_bulk_no_rankings"]

    # 5. the CPU restatement on a named slice: the first R rows and the first E primary events, popRank only
    from oracle.model_oracle import model_bulk
    R, E = a.oracle_rows, a.oracle_events
    row_ids = [str(j) for j in range(n_items)]
    inds = []
    for t in range(w.n_types):
        rp, ci = res[t][3], res[t][4]
        inds.append((rp[:R + 1].copy(), ci[:int(rp[R])].copy()))
    items = [str(int(x)) for x in prim[:E]]
    t0 = time.perf_counter()
    body = model_bulk(inds, names, row_ids[:R], [row_ids] * w.n_types,
                      [("popRank", "popular", items, times[:E], now - 30 * DAY, now)])
    result["oracle_slice"] = {"rows": R, "events": E, "ms": round((time.perf_counter() - t0) * 1e3, 1), "out_bytes": len(body)}
    ctx.free_result(h)
    ctx.close()
    result["device"], result["power_limit"] = device_info()
    print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()
