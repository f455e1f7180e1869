"""TEST INFRASTRUCTURE: CPU restatement of the whole model document (SURVEY.md 8f-2 + 8f-3 joined), the checker of
cco_format_model_bulk.  URModel.save writes groupAll(correlators ++ propertiesRDD) with recsModel "all"
(/root/reference/src/main/scala/URAlgorithm.scala:351-367, getRanksRDD :537-560, URModel.scala:57-102): the rows of
format_oracle.es_bulk, one rank field per ranking (pop_oracle.pop_model) and the item's property fragment, plus a document
of its own for every other id with a rank or a property entry.  Byte layout: this repo's definition, identical in the CUDA
path; rank values as Java's Double.toString writes them (elasticsearch-hadoop serialises a JDouble with it)."""
from __future__ import annotations

from oracle.format_oracle import es_bulk, json_escape
from oracle.pop_oracle import pop_model


def java_double(v: float) -> bytes:
    """Double.toString of an integral double with |v| < 2^34, as elasticsearch-hadoop writes a rank: "<int>.0" below 10^7,
    otherwise d.dddE<n> with the trailing zeros of the fraction stripped (at least one digit kept)."""
    x = int(v)
    assert x == v and abs(x) < 2 ** 34
    if abs(x) < 10 ** 7:
        return f"{x}.0".encode()
    d = str(abs(x))
    return f"{'-' if x < 0 else ''}{d[0]}.{d[1:].rstrip('0') or '0'}E{len(d) - 1}".encode()


def model_bulk(indicators, names, row_ids, col_ids, rankings=(), properties=None) -> bytes:
    """The checker of cco_format_model_bulk: URModel.save with recsModel "all" (URAlgorithm.scala:351-367, 537-560).
    indicators / names / row_ids / col_ids as es_bulk over the whole model; rankings: [(field name, mode, item id strings of
    the ranking's events, times_ms, start_ms, end_ms)]; properties: {id: fragment} or (ids, fragments), a fragment being JSON
    object members without braces, spliced in verbatim.
    Documents: the rows in row order, then every other id with a present rank or a property entry, in order of first
    appearance in (ranking 0's items, ranking 1's, ..., property ids).  Fields: "id", the indicators (rows only), the ranks
    (pop_oracle.pop_model over the ranking's events), the fragment if non-empty."""
    if properties is None:
        properties = ([], [])
    elif isinstance(properties, dict):
        properties = (list(properties.keys()), list(properties.values()))
    pids, frags = properties
    cls: dict[str, int] = {}
    for x in list(row_ids) + [x for _, _, items, _, _, _ in rankings for x in items] + list(pids):
        cls.setdefault(x, len(cls))
    ranks = [(name.encode("utf-8"), pop_model(mode, [cls[x] for x in items], times, start, end))
             for name, mode, items, times, start, end in rankings]
    frag_of = {cls[x]: f.encode("utf-8") if isinstance(f, str) else bytes(f) for x, f in zip(pids, frags)}

    def tail(c: int) -> bytes:
        out = b"".join(b',"' + json_escape(n.decode("utf-8")) + b'":' + java_double(r[c]) for n, r in ranks if c in r)
        if frag_of.get(c):
            out += b"," + frag_of[c]
        return out + b"}\n"

    lines = es_bulk(indicators, names, row_ids, col_ids).split(b"\n")
    out = bytearray()
    for r in range(len(row_ids)):
        out += lines[2 * r] + b"\n" + lines[2 * r + 1][:-1] + tail(r)
    ids = list(cls)
    for c in range(len(row_ids), len(ids)):
        if c in frag_of or any(c in r for _, r in ranks):
            e = json_escape(ids[c])
            out += b'{"index":{"_id":"' + e + b'"}}\n{"id":"' + e + b'"' + tail(c)
    return bytes(out)
