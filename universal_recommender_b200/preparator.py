"""Host-side mirror of Preparator.prepare + the two IndexedDatasetSpark.apply builders
(/root/reference/src/main/scala/Preparator.scala:44-87, 100-216): event (user, item) string pairs
per event name -> IndexedDatasets that share one user dictionary.

This is the INPUT side of the hot-path boundary (SURVEY.md 8a-H1).  `prepare` is the host logic;
`prepare_on_device` gives the same result from the same id strings through cco_ingest_strings (SURVEY.md 8f-1)."""
from __future__ import annotations

from typing import Sequence

import numpy as np

from .indexed_dataset import BiDictionary, IndexedDataset


def _build(pairs: Sequence[tuple[str, str]], row_ids: BiDictionary, freeze_rows: bool) -> IndexedDataset:
    """IndexedDatasetSpark.apply(elements, existingRowIDs) (Preparator.scala:160-214): events of
    unknown users are dropped when a dictionary is passed in; item ids always come from the events
    that survive; duplicates collapse (`setQuick(col, 1.0)`)."""
    col_ids = BiDictionary()
    rows: list[int] = []
    cols: list[int] = []
    for user, item in pairs:
        if freeze_rows:
            r = row_ids.get(user)
            if r < 0:
                continue
        else:
            r = row_ids.add(user)
        rows.append(r)
        cols.append(col_ids.add(item))
    n_rows = row_ids.size
    r = np.asarray(rows, dtype=np.int64)
    c = np.asarray(cols, dtype=np.int64)
    if len(r):
        keys = np.unique(r * max(col_ids.size, 1) + c)   # dedup + sort by (row, col)
        r, c = keys // max(col_ids.size, 1), keys % max(col_ids.size, 1)
    row_ptr = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(r, minlength=n_rows), out=row_ptr[1:])
    return IndexedDataset(row_ptr, c.astype(np.int32), row_ids, col_ids, n_rows=n_rows, n_cols=col_ids.size)


def indexed_dataset_min_events(pairs: Sequence[tuple[str, str]], min_events_per_user: int) -> BiDictionary:
    """IndexedDatasetSpark.apply(elements, minEventsPerUser) (Preparator.scala:102-158): the dictionary
    of users with >= minEventsPerUser events, counting duplicates (`items.size` over groupByKey, :129-132)."""
    counts: dict[str, int] = {}
    for user, _ in pairs:
        counts[user] = counts.get(user, 0) + 1
    return BiDictionary(u for u, n in counts.items() if n >= min_events_per_user)


def prepare(actions: Sequence[tuple[str, Sequence[tuple[str, str]]]],
            min_events_per_user: int | None = None) -> list[tuple[str, IndexedDataset]]:
    """Preparator.prepare (Preparator.scala:44-87).  `actions` = TrainingData.actions, first = primary.
    Every later event type is restricted to the users known so far and all share one row space."""
    user_dict: BiDictionary | None = None
    out: list[tuple[str, IndexedDataset]] = []
    for idx, (name, pairs) in enumerate(actions):
        if idx == 0 and min_events_per_user is not None:
            passing = indexed_dataset_min_events(pairs, min_events_per_user)
            ids = _build(pairs, passing, freeze_rows=True)            # :62 rebuilt on passing users only
        elif user_dict is None:
            ids = _build(pairs, BiDictionary(), freeze_rows=False)
        else:
            ids = _build(pairs, user_dict, freeze_rows=True)          # :69 IndexedDatasetSpark(eventRDD, userDictionary)
        user_dict = ids.row_ids
        out.append((name, ids))
    return out


def encode_ids(ids: Sequence[str]) -> tuple[np.ndarray, np.ndarray]:
    """id strings -> (offsets int64[n + 1], UTF-8 bytes uint8[]): id e = bytes[offsets[e]:offsets[e + 1]].  Vectorised:
    one join, one UTF-8 and one UTF-32 encode of the whole column; the UTF-8 length of every code point gives the offsets."""
    n = len(ids)
    joined = "".join(ids)
    data = np.frombuffer(joined.encode("utf-8"), dtype=np.uint8)
    cps = np.frombuffer(joined.encode("utf-32-le"), dtype=np.uint32)
    cp_bytes = np.zeros(len(cps) + 1, dtype=np.int64)
    np.cumsum(1 + (cps >= 0x80) + (cps >= 0x800) + (cps >= 0x10000), out=cp_bytes[1:])
    chars = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.fromiter(map(len, ids), dtype=np.int64, count=n), out=chars[1:])
    return cp_bytes[chars], data


def prepare_on_device(ctx, actions: Sequence[tuple[str, Sequence[tuple[str, str]]]],
                      min_events_per_user: int | None = None):
    """`prepare` on the B200 (cco_ingest_strings): same arguments and the same [(name, IndexedDataset)], plus the
    HBM-resident dataset the matrices came from, ready for ctx.train_dataset (release it with ctx.free_dataset)."""
    types = []
    for _, pairs in actions:
        users, items = zip(*pairs) if len(pairs) else ((), ())
        types.append((*encode_ids(users), *encode_ids(items)))
    ds, user_ids, item_ids = ctx.ingest_strings(types, min_events_per_user or 0)
    row_ids = BiDictionary(user_ids)
    out = []
    for t, (name, _) in enumerate(actions):
        nr, nc, rp, ci = ctx.dataset_matrix(ds, t)
        out.append((name, IndexedDataset(rp, ci, row_ids, BiDictionary(item_ids[t]), n_rows=nr, n_cols=nc)))
    return out, ds
