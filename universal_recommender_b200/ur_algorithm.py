"""Mirror of the train half of URAlgorithm that reaches the hot path
(/root/reference/src/main/scala/URAlgorithm.scala:130-171 params, :310-349 calcAll) and of the model document calcAll
hands to URModel.save (:351-367, getRanksRDD :537-560).  ES query building and calcPop (recsModel "backfill") are out of
scope."""
from __future__ import annotations

import re
import time
from datetime import datetime, timedelta, timezone
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np

from .indexed_dataset import IndexedDataset
from .similarity_analysis import CcoContext, DownsamplableCrossOccurrenceDataset, SimilarityAnalysis


class DefaultURAlgoParams:
    """URAlgorithm.scala:53-57"""
    MaxEventsPerEventType = 500
    MaxCorrelatorsPerEventType = 50


@dataclass
class IndicatorParams:
    """URAlgorithm.scala:136-140"""
    name: str
    maxItemsPerUser: Optional[int] = None
    maxCorrelatorsPerItem: Optional[int] = None
    minLLR: Optional[float] = None


@dataclass
class RankingParams:
    """URAlgorithm.scala:110-127; `type` is popular | trending | hot | userDefined | random (PopModel.scala:43-51)."""
    name: Optional[str] = None
    type: Optional[str] = None
    eventNames: Optional[Sequence[str]] = None
    offsetDate: Optional[str] = None
    endDate: Optional[str] = None     # parsed, unused by getRanksRDD (as in the reference)
    duration: Optional[str] = None


@dataclass
class URAlgorithmParams:
    """The subset of URAlgorithmParams (URAlgorithm.scala:142-171) that reaches the hot path."""
    eventNames: Optional[Sequence[str]] = None
    maxEventsPerEventType: Optional[int] = None
    maxCorrelatorsPerEventType: Optional[int] = None
    indicators: Optional[Sequence[IndicatorParams]] = None
    seed: Optional[int] = None
    recsModel: str = "all"
    # not an engine.json key of the reference: selects the literal Int/Int row sample rate recalled from Mahout 0.13.0's
    # sampleDownAndBinarize (SURVEY.md A.1; every interaction of a user above maxItemsPerUser is dropped) instead of the
    # real division min(m, d) / d this build defaults to (INTEGRATION.md "Deviation to know about")
    rowRateIntDiv: bool = False
    rankings: Optional[Sequence[RankingParams]] = None

    @staticmethod
    def from_engine_json(algo_params: dict) -> "URAlgorithmParams":
        ind = algo_params.get("indicators")
        return URAlgorithmParams(
            eventNames=algo_params.get("eventNames"),
            maxEventsPerEventType=algo_params.get("maxEventsPerEventType"),
            maxCorrelatorsPerEventType=algo_params.get("maxCorrelatorsPerEventType"),
            indicators=None if ind is None else [IndicatorParams(i["name"], i.get("maxItemsPerUser"),
                                                                 i.get("maxCorrelatorsPerItem"), i.get("minLLR")) for i in ind],
            seed=algo_params.get("seed"), recsModel=algo_params.get("recsModel", "all"),
            rowRateIntDiv=bool(algo_params.get("rowRateIntDiv", False)),
            rankings=None if algo_params.get("rankings") is None else [
                RankingParams(r.get("name"), r.get("type"), r.get("eventNames"), r.get("offsetDate"), r.get("endDate"),
                              r.get("duration")) for r in algo_params["rankings"]])


def calc_all(actions: Sequence[tuple[str, IndexedDataset]], ap: URAlgorithmParams,
             ctx: CcoContext | None = None, flags: int = 0) -> list[tuple[str, IndexedDataset]]:
    """URAlgorithm.calcAll up to `cooccurrenceCorrelators` (URAlgorithm.scala:310-349): picks the global-
    params call or the per-indicator call, then zips the event names back on positionally (:349).
    `indicators(i)` is indexed by POSITION in `actions` exactly like the reference (:334-340)."""
    if ap.recsModel not in ("all", "collabFiltering", "backfill"):
        raise ValueError(f"Bad algorithm param recsModel=[{ap.recsModel}] in engine definition params, possibly a bad json "
                         "value. Use one of the available parameter values (all, collabFiltering, backfill).")
    if ap.recsModel == "backfill":
        return []  # calcPop only: no CCO (URAlgorithm.scala:296)
    seed = ap.seed if ap.seed is not None else int(time.time() * 1000)   # System.currentTimeMillis() (:325,345)
    if ap.rowRateIntDiv:
        flags |= 1   # CCO_FLAG_ROWRATE_INTDIV
    ids = [d for _, d in actions]
    if not ap.indicators:
        out = SimilarityAnalysis.cooccurrencesIDSs(
            ids, randomSeed=seed,
            maxInterestingItemsPerThing=ap.maxCorrelatorsPerEventType or DefaultURAlgoParams.MaxCorrelatorsPerEventType,
            maxNumInteractions=ap.maxEventsPerEventType or DefaultURAlgoParams.MaxEventsPerEventType, ctx=ctx, flags=flags)
    else:
        inds = ap.indicators
        datasets = [DownsamplableCrossOccurrenceDataset(
            iD, inds[i].maxItemsPerUser or DefaultURAlgoParams.MaxEventsPerEventType,
            inds[i].maxCorrelatorsPerItem or DefaultURAlgoParams.MaxCorrelatorsPerEventType, inds[i].minLLR)
            for i, iD in enumerate(ids)]
        out = SimilarityAnalysis.crossOccurrenceDownsampled(datasets, seed, ctx=ctx, flags=flags)
    return [(name, o) for (name, _), o in zip(actions, out)]


# ---- the model document: correlators + rank fields + item properties (URAlgorithm.scala:351-367, 537-560) ---------------
BACKFILL_FIELD_NAME, BACKFILL_TYPE, BACKFILL_DURATION = "popRank", "popular", "3650 days"   # URAlgorithm.scala:64-66
RANK_FIELD_BY_TYPE = {"popular": "popRank", "trending": "trendRank", "hot": "hotRank"}      # PopModel.nameByType :205-210

# scala.concurrent.duration.Duration unit labels: the first of each line has no plural form
_UNIT_NANOS: dict[str, int] = {}
for _labels, _nanos in (("d day", 86_400 * 10 ** 9), ("h hour", 3_600 * 10 ** 9), ("min minute", 60 * 10 ** 9),
                        ("s sec second", 10 ** 9), ("ms milli millisecond", 10 ** 6), ("\u00b5s micro microsecond", 10 ** 3),
                        ("ns nano nanosecond", 1)):
    _hd, *_rest = _labels.split()
    _UNIT_NANOS[_hd] = _nanos
    for _w in _rest:
        _UNIT_NANOS[_w] = _UNIT_NANOS[_w + "s"] = _nanos


def _to_i32(x: int) -> int:
    x &= 0xffffffff
    return x - (1 << 32) if x & 0x80000000 else x


def duration_seconds(s: str) -> int:
    """`Duration(s).toSeconds.toInt` (URAlgorithm.scala:543): whitespace dropped, the trailing letters name the unit, the
    length is parsed as a double (rounded to whole nanoseconds) or, beyond 2^53, as a long; seconds truncate toward zero and
    wrap to 32 bits like `.toInt`.  Anything else raises ValueError (Scala throws NumberFormatException)."""
    s1 = "".join(ch for ch in s if not ch.isspace())
    unit = re.search(r"[^\W\d_]*$", s1).group(0)
    if unit not in _UNIT_NANOS:
        raise ValueError(f"format error {s}")
    value = s1[:len(s1) - len(unit)]
    v = float(value)
    if abs(v) <= 2.0 ** 53:
        nanos = int(_UNIT_NANOS[unit] * v + 0.5)      # Duration.fromNanos(double): (nanos + 0.5).toLong
    else:
        nanos = int(value) * _UNIT_NANOS[unit]
    secs = abs(nanos) // 10 ** 9 * (1 if nanos >= 0 else -1)
    return _to_i32(secs)


def _parse_end_ms(offset_date: Optional[str], now_ms: int) -> int:
    """PopModel.scala:66-74: the ISO-8601 offsetDate, or now when there is none or it does not parse.  A date-time without
    a zone is read as UTC."""
    if offset_date is None:
        return now_ms
    try:
        d = datetime.fromisoformat(offset_date)
    except ValueError:
        return now_ms
    if d.tzinfo is None:
        d = d.replace(tzinfo=timezone.utc)
    return (d - datetime(1970, 1, 1, tzinfo=timezone.utc)) // timedelta(milliseconds=1)


@dataclass
class ResolvedRanking:
    name: str
    type: str          # popular | trending | hot
    eventNames: list
    start_ms: int
    end_ms: int


def model_event_names(ap: URAlgorithmParams) -> list:
    """URAlgorithm.scala:230-234"""
    if ap.indicators:
        return [i.name for i in ap.indicators]
    if not ap.eventNames:
        raise ValueError("No eventNames or indicators in engine.json and one of these is required")
    return list(ap.eventNames)


def resolve_rankings(ap: URAlgorithmParams, now_ms: Optional[int] = None) -> list[ResolvedRanking]:
    """The rank fields getRanksRDD computes (URAlgorithm.scala:250-256, 537-546): the default popRank / popular / 3650 days
    over the first model event when `rankings` is absent; the first ranking of each type (`groupBy(_.type).map(_._2.head)`,
    kept in order of first appearance); userDefined, random and unknown types dropped -- they reach the document as
    properties the caller passes, or not at all.  The interval is [end - duration, end), end = offsetDate or now."""
    if now_ms is None:
        now_ms = int(time.time() * 1000)
    params = ap.rankings if ap.rankings is not None else [
        RankingParams(BACKFILL_FIELD_NAME, BACKFILL_TYPE, model_event_names(ap)[:1], None, None, BACKFILL_DURATION)]
    first_of_type: dict = {}
    for p in params:
        first_of_type.setdefault(p.type, p)
    out = []
    for p in first_of_type.values():
        typ = p.type or BACKFILL_TYPE
        if typ not in RANK_FIELD_BY_TYPE:
            continue
        end = _parse_end_ms(p.offsetDate, now_ms)
        secs = duration_seconds(p.duration or BACKFILL_DURATION)
        events = list(p.eventNames) if p.eventNames is not None else model_event_names(ap)[:1]
        out.append(ResolvedRanking(p.name or RANK_FIELD_BY_TYPE[typ], typ, events, end - 1000 * secs, end))
    return out


def write_model(ctx: CcoContext, handle, names, row_ids, col_ids, ap: URAlgorithmParams, events, properties=None,
                now_ms: Optional[int] = None) -> bytes:
    """The documents calcAll hands to URModel.save (URAlgorithm.scala:351-367) as the Elasticsearch bulk body, for a kept
    result `handle` of the whole model.  events = [(event name, item id, time_ms)]: every event of the app, any user;
    properties = {item id: fragment} or (ids, fragments), the item's $set properties (and userDefined / random ranks) as JSON
    object members without braces.  recsModel "all" adds the rank fields and the properties (format_model_bulk);
    "collabFiltering" writes the correlators only (calcAll(calcPopular = false) saves an empty propertiesRDD), exactly
    format_es_bulk's bytes."""
    if ap.recsModel == "collabFiltering":
        return ctx.format_es_bulk(handle, names, row_ids, col_ids)
    if ap.recsModel != "all":
        raise ValueError(f"recsModel {ap.recsModel!r}: write_model builds the documents of calcAll (all, collabFiltering)")
    rankings = []
    for r in resolve_rankings(ap, now_ms):
        want = set(r.eventNames)
        sel = [(item, t) for (ev, item, t) in events if ev in want]
        rankings.append((r.name, r.type, [i for i, _ in sel], np.array([t for _, t in sel], dtype=np.int64), r.start_ms, r.end_ms))
    return ctx.format_model_bulk(handle, names, row_ids, col_ids, rankings, properties)
