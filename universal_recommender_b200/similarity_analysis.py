"""Python mirror of org.apache.mahout.math.cf.SimilarityAnalysis as the reference calls it
(/root/reference/src/main/scala/URAlgorithm.scala:323-329, 343-346), running on the B200 through the
C ABI of include/cco_b200.h.  Same names, argument meaning and error behaviour; the arithmetic is
the hand-written sm_100a path in csrc/ -- there is no CPU implementation in this package."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _native as N
from .indexed_dataset import IndexedDataset


@dataclass
class DownsamplableCrossOccurrenceDataset:
    """org.apache.mahout.math.cf.DownsamplableCrossOccurrenceDataset as constructed at
    URAlgorithm.scala:336-340 (defaults 500 / 50 / None)."""
    iD: IndexedDataset
    maxElementsPerRow: int = 500
    maxInterestingElements: int = 50
    minLLROpt: Optional[float] = None
    parOpts: object = None   # Spark partitioning hints: meaningless here, accepted and ignored


@dataclass
class TrainStats:
    n_users: int
    nnz_in_total: int
    nnz_downsampled: list
    products: list
    distinct_cells: list
    out_nnz: list
    llr_evaluated: list
    ms_h2d: float
    ms_prepare: float
    ms_cooccurrence: float
    ms_total: float
    ms_indicator: list
    n_kernel_launches: int
    ms_prep_stage: list = None


class CcoContext:
    """One GPU context (= cco_ctx_t).  One process per GPU; for world_size > 1 pass the 128-byte NCCL id
    from `CcoContext.nccl_unique_id()` of rank 0 (distribute it with any host transport)."""

    def __init__(self, device: int = 0, rank: int = 0, world_size: int = 1, nccl_unique_id: bytes | None = None,
                 devices: Sequence[int] | None = None, result_arena: np.ndarray | None = None):
        """devices=[...]: a GROUP context over several GPUs of this process (cco_create_group): train_csr then returns the
        merged model of all of them.  result_arena: a writable uint8 array (e.g. np.memmap of a /dev/shm file) the result
        arrays are placed in (cco_config_t.result_arena)."""
        L = N.lib()
        self._L = L
        self._uid = None
        self._arena = result_arena
        self.last_stats: TrainStats | None = None
        self._pinned_addr: dict = {}
        if devices is not None:
            h = C.c_void_p()
            arr = (C.c_int32 * len(devices))(*devices)
            N.check(L.cco_create_group(len(devices), arr, C.byref(h)))
            self._h = h
            self.rank, self.world_size, self.device, self.devices = 0, 1, devices[0], list(devices)
            return
        cfg = N.ConfigT(device, rank, world_size, 0, None, None, 0)
        if result_arena is not None:
            cfg.result_arena = result_arena.ctypes.data
            cfg.result_arena_bytes = result_arena.nbytes
        if world_size > 1:
            if nccl_unique_id is None or len(nccl_unique_id) != 128:
                raise N.CcoInvalidArgument(N.E_INVALID_ARG, "world_size > 1 needs the 128-byte nccl_unique_id")
            self._uid = (C.c_ubyte * 128).from_buffer_copy(nccl_unique_id)
            cfg.nccl_unique_id = C.cast(self._uid, C.POINTER(C.c_ubyte))
        h = C.c_void_p()
        N.check(L.cco_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.rank, self.world_size, self.device, self.devices = rank, world_size, device, [device]

    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = (C.c_ubyte * 128)()
        N.check(N.lib().cco_nccl_unique_id(buf))
        return bytes(buf)

    def close(self):
        if getattr(self, "_h", None):
            self._L.cco_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- pinned host buffers (what the JNI shim wraps as direct ByteBuffers) -------------------------
    def host_array(self, n: int, dtype) -> np.ndarray:
        dt = np.dtype(dtype)
        p = C.c_void_p()
        N.check(self._L.cco_host_alloc(self._h, max(n, 1) * dt.itemsize, C.byref(p)))
        buf = (C.c_byte * (max(n, 1) * dt.itemsize)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dt, count=n)
        self._pinned_addr[arr.ctypes.data if n else p.value] = p
        return arr

    def host_free(self, arr: np.ndarray):
        p = self._pinned_addr.pop(arr.ctypes.data, None)
        if p is not None:
            self._L.cco_host_free(self._h, p)

    # ---- the hot path ---------------------------------------------------------------------------------------
    def _csr_array(self, mats):
        n = len(mats)
        keep = []
        cm = (N.CsrT * n)()
        for i, (nr, nc, rp, ci) in enumerate(mats):
            rp = np.ascontiguousarray(rp, dtype=np.int64)
            ci = np.ascontiguousarray(ci, dtype=np.int32)
            keep.append((rp, ci))
            cm[i] = N.as_csr_t(nr, nc, rp, ci)
        return cm, keep

    @staticmethod
    def _params_array(params):
        return (N.ParamsT * len(params))(*[N.ParamsT(int(m), int(k), 0 if ml is None else 1, 0.0 if ml is None else float(ml))
                                           for (m, k, ml) in params])

    def _collect(self, res, n, copy_arrays=True, keep=False):
        """copy_arrays: numpy copies of the result arrays (default).  keep=True: zero-copy VIEWS of the library-owned pinned
        result buffers instead; the caller must call free_result(handle) when done (returns (views, handle))."""
        L = self._L
        try:
            out = []
            for i in range(n):
                rb, re_ = C.c_int64(), C.c_int64()
                N.check(L.cco_result_row_range(res, i, C.byref(rb), C.byref(re_)))
                nr, nc = C.c_int64(), C.c_int32()
                prp, pci, pll, pcn = C.POINTER(C.c_int64)(), C.POINTER(C.c_int32)(), C.POINTER(C.c_double)(), C.POINTER(C.c_int32)()
                N.check(L.cco_result_matrix(res, i, C.byref(nr), C.byref(nc), C.byref(prp), C.byref(pci), C.byref(pll), C.byref(pcn)))
                rp = np.ctypeslib.as_array(prp, shape=(nr.value + 1,))
                if not keep:
                    rp = rp.copy()
                nnz = int(rp[-1])
                if nnz and (copy_arrays or keep):
                    ci = np.ctypeslib.as_array(pci, shape=(nnz,))
                    ll = np.ctypeslib.as_array(pll, shape=(nnz,)) if pll else np.zeros(0, np.float64)
                    cn = np.ctypeslib.as_array(pcn, shape=(nnz,)) if pcn else np.zeros(0, np.int32)
                    if not keep:
                        ci, ll, cn = ci.copy(), ll.copy(), cn.copy()
                else:
                    ci, ll, cn = np.zeros(0, np.int32), np.zeros(0, np.float64), np.zeros(0, np.int32)
                out.append((rb.value, re_.value, nc.value, rp, ci, ll, cn))
            st = N.StatsT()
            N.check(L.cco_result_stats(res, C.byref(st)))
            self.last_stats = TrainStats(st.n_users, st.nnz_in_total, list(st.nnz_downsampled)[:n], list(st.products)[:n],
                                         list(st.distinct_cells)[:n], list(st.out_nnz)[:n], list(st.llr_evaluated)[:n], st.ms_h2d, st.ms_prepare,
                                         st.ms_cooccurrence, st.ms_total, list(st.ms_indicator)[:n], st.n_kernel_launches, list(st.ms_prep_stage))
            if keep:
                h, res = res, None
                return out, h
            return out
        finally:
            if res is not None:
                L.cco_result_free(res)

    def free_result(self, handle):
        self._L.cco_result_free(handle)

    # ---- next row (SURVEY.md 8f-3): PopModel rank histograms ---------------------------------------------------------------
    def pop_model(self, mode: str, items, times_ms, n_items: int, start_ms: int, end_ms: int):
        """PopModel.calcPopular / calcTrending / calcHot (PopModel.scala:113-182) -> {item index: score} for the items the
        reference's RDD would contain."""
        code = {"popular": 0, "trending": 1, "hot": 2}[mode]
        it = np.ascontiguousarray(items, dtype=np.int32)
        tm = np.ascontiguousarray(times_ms, dtype=np.int64)
        score = np.zeros(max(n_items, 1), dtype=np.float64)
        present = np.zeros(max(n_items, 1), dtype=np.uint8)
        N.check(self._L.cco_pop_model(self._h, code, len(it), it.ctypes.data_as(C.POINTER(C.c_int32)), tm.ctypes.data_as(C.POINTER(C.c_int64)),
                                      n_items, int(start_ms), int(end_ms), score.ctypes.data_as(C.POINTER(C.c_double)),
                                      present.ctypes.data_as(C.POINTER(C.c_ubyte))))
        return {int(j): float(score[j]) for j in np.nonzero(present[:n_items])[0]}

    # ---- next row (SURVEY.md 8f-2): the model as the Elasticsearch bulk body -------------------------------------------
    @staticmethod
    def _dictionary(ids):
        """list of id strings -> (DictionaryT, keep-alive): UTF-8 bytes + offsets"""
        enc = [x.encode("utf-8") for x in ids]
        off = np.zeros(len(enc) + 1, dtype=np.int64)
        np.cumsum([len(b) for b in enc], out=off[1:])
        blob = b"".join(enc)
        buf = C.create_string_buffer(blob, max(len(blob), 1))
        return N.DictionaryT(len(enc), off.ctypes.data_as(C.POINTER(C.c_int64)), C.cast(buf, C.c_char_p)), (off, buf)

    def format_es_bulk(self, handle, names, row_ids, col_ids) -> bytes:
        """cco_format_es_bulk on a kept result (train_csr(..., keep=True)): one Elasticsearch bulk index action per row,
        `{"index":{"_id":id}}\\n{"id":id,"<event>":[ordered correlator ids],...}\\n` -- what toStringMapRDD + URModel.save +
        saveToEs produce for the reference (package.scala:82-110, URModel.scala:47-102, EsClient.scala:300-313)."""
        n = len(names)
        keep = []
        rd, k = self._dictionary(row_ids)
        keep.append(k)
        cds = (N.DictionaryT * n)()
        for i, ids in enumerate(col_ids):
            cds[i], k = self._dictionary(ids)
            keep.append(k)
        nm = (C.c_char_p * n)(*[x.encode("utf-8") for x in names])
        out, ln = C.c_void_p(), C.c_int64()
        N.check(self._L.cco_format_es_bulk(self._h, handle, n, nm, C.byref(rd), cds, C.byref(out), C.byref(ln)))
        try:
            return C.string_at(out.value, ln.value)
        finally:
            self._L.cco_host_free(self._h, out)

    @staticmethod
    def _raw_dictionary(ids, keep: list):
        """a `str` list or an (offsets int64[], bytes uint8[]) pair of preparator.encode_ids -> DictionaryRawT"""
        if isinstance(ids, tuple) and len(ids) == 2 and isinstance(ids[0], np.ndarray):
            off, data = ids
        else:
            from .preparator import encode_ids
            off, data = encode_ids(list(ids))
        off = np.ascontiguousarray(off, dtype=np.int64)
        data = np.ascontiguousarray(data, dtype=np.uint8)
        keep.append((off, data))
        return N.DictionaryRawT(len(off) - 1, off.ctypes.data_as(C.POINTER(C.c_int64)), data.ctypes.data if len(data) else None)

    def format_model_bulk(self, handle, names, row_ids, col_ids, rankings=(), properties=None, flags: int = 0) -> bytes:
        """cco_format_model_bulk on a kept result: the documents URModel.save writes with recsModel "all"
        (URAlgorithm.scala:351-367, 537-560; URModel.scala:57-102) -- format_es_bulk's rows plus one rank field per ranking in
        which an id is present and its property fragment, and a document of its own for every other id with a rank or a
        property entry.  rankings = [(field name, "popular" | "trending" | "hot", item ids of the ranking's events,
        times_ms int64[], start_ms, end_ms)]; properties = {id: fragment} or (ids, fragments), a fragment being JSON object
        members without braces.  Ids are `str` lists or encode_ids pairs."""
        keep: list = []
        n = len(names)
        rd = self._raw_dictionary(row_ids, keep)
        cds = (N.DictionaryRawT * n)(*[self._raw_dictionary(ids, keep) for ids in col_ids])
        nm = (C.c_char_p * n)(*[x.encode("utf-8") for x in names])
        rk = (N.RankingT * max(len(rankings), 1))()
        for r, (name, mode, items, times, start_ms, end_ms) in enumerate(rankings):
            code = {"popular": 0, "trending": 1, "hot": 2}[mode] if isinstance(mode, str) else int(mode)
            d = self._raw_dictionary(items, keep)
            t = np.ascontiguousarray(times, dtype=np.int64)
            keep.append(t)
            if len(t) != d.n:
                raise N.CcoInvalidArgument(N.E_INVALID_ARG, f"ranking {name}: {d.n} item ids but {len(t)} times")
            nb = None if name is None else name.encode("utf-8")
            keep.append(nb)
            rk[r] = N.RankingT(nb, code, 0, int(start_ms), int(end_ms), d, t.ctypes.data_as(C.POINTER(C.c_int64)))
        pid = pjs = None
        if properties is not None:
            ids, frags = (list(properties.keys()), list(properties.values())) if isinstance(properties, dict) else properties
            pid, pjs = self._raw_dictionary(ids, keep), self._raw_dictionary(frags, keep)
        out, ln = C.c_void_p(), C.c_int64()
        N.check(self._L.cco_format_model_bulk(self._h, handle, n, nm, C.byref(rd), cds, len(rankings), rk,
                                              C.byref(pid) if pid is not None else None, C.byref(pjs) if pjs is not None else None,
                                              flags, C.byref(out), C.byref(ln)))
        try:
            return C.string_at(out.value, ln.value)
        finally:
            self._L.cco_host_free(self._h, out)

    def train_csr(self, mats: Sequence[tuple[int, int, np.ndarray, np.ndarray]], params: Sequence[tuple[int, int, Optional[float]]],
                  seed: int, flags: int = 0, copy_arrays: bool = True, keep: bool = False):
        """Raw entry (cco_train): mats = [(n_rows, n_cols, row_ptr int64, col_idx int32)], params = [(m, k, minLLR|None)].
        -> list of (row_begin, row_end, n_cols, row_ptr, col_idx, llr, count) numpy copies, one per matrix
        (keep=True: zero-copy views + a handle for free_result)."""
        cm, alive = self._csr_array(mats)
        res = C.c_void_p()
        N.check(self._L.cco_train(self._h, len(mats), cm, self._params_array(params), C.c_int32(_to_i32(seed)), flags,
                                  C.byref(res)))
        return self._collect(res, len(mats), copy_arrays, keep)

    # ---- split form: matrices resident in HBM across trains ---------------------------------------------
    def upload(self, mats, flags: int = 0):
        cm, keep = self._csr_array(mats)
        ds = C.c_void_p()
        N.check(self._L.cco_dataset_upload(self._h, len(mats), cm, flags, C.byref(ds)))
        return (ds, len(mats))

    def train_dataset(self, dataset, params, seed: int, flags: int = 0, copy_arrays: bool = True, keep: bool = False):
        """keep=True: as for train_csr, zero-copy views + a handle for free_result / format_es_bulk."""
        ds, n = dataset
        res = C.c_void_p()
        N.check(self._L.cco_train_dataset(self._h, ds, self._params_array(params), C.c_int32(_to_i32(seed)), flags, C.byref(res)))
        return self._collect(res, n, copy_arrays, keep)

    def ingest(self, events, n_users_raw: int, min_events_per_user: int = 0):
        """Preparator.prepare on the device (SURVEY.md 8f-1).  events = [(users int64[], items int32[], n_items_raw)], type 0
        = primary.  -> (dataset for train_dataset, user_map int32[n_users_raw], [item_map int32[n_items_raw]])."""
        n = len(events)
        keep, ev = [], (N.EventsT * n)()
        item_maps = [np.zeros(max(ni, 1), dtype=np.int32) for (_, _, ni) in events]
        for t, (u, i, ni) in enumerate(events):
            u = np.ascontiguousarray(u, dtype=np.int64)
            i = np.ascontiguousarray(i, dtype=np.int32)
            keep.append((u, i))
            ev[t] = N.EventsT(len(u), u.ctypes.data_as(C.POINTER(C.c_int64)), i.ctypes.data_as(C.POINTER(C.c_int32)), ni)
        user_map = np.zeros(max(n_users_raw, 1), dtype=np.int32)
        maps = (C.POINTER(C.c_int32) * n)(*[m.ctypes.data_as(C.POINTER(C.c_int32)) for m in item_maps])
        ds = C.c_void_p()
        N.check(self._L.cco_ingest(self._h, n, ev, n_users_raw, min_events_per_user, user_map.ctypes.data_as(C.POINTER(C.c_int32)),
                                   maps, C.byref(ds)))
        return (ds, n), user_map[:n_users_raw], [m[:ni] for m, (_, _, ni) in zip(item_maps, events)]

    def ingest_strings(self, types, min_events_per_user: int = 0, flags: int = 0):
        """Preparator.prepare on the device from raw id strings (cco_ingest_strings).  types = [(user_offsets int64[],
        user_bytes uint8[], item_offsets int64[], item_bytes uint8[])], type 0 = primary; the ids of event e are
        bytes[offsets[e]:offsets[e + 1]].  -> (dataset for train_dataset, user ids, [item ids of each type]), the ids as
        `str` (UTF-8; bytes that are not UTF-8 come back as surrogate escapes) in dictionary order."""
        n = len(types)
        keep, ev = [], (N.StringEventsT * n)()

        def column(off, data):
            off = np.ascontiguousarray(off, dtype=np.int64)
            data = np.ascontiguousarray(data, dtype=np.uint8)
            keep.append((off, data))
            return N.DictionaryRawT(len(off) - 1, off.ctypes.data_as(C.POINTER(C.c_int64)), data.ctypes.data if len(data) else None)

        for t, (uo, ub, io, ib) in enumerate(types):
            ev[t] = N.StringEventsT(column(uo, ub), column(io, ib))
        user, items = N.DictionaryRawT(), (N.DictionaryRawT * n)()
        ds = C.c_void_p()
        N.check(self._L.cco_ingest_strings(self._h, n, ev, int(min_events_per_user), flags, C.byref(user), items, C.byref(ds)))
        return (ds, n), self._take_ids(user), [self._take_ids(items[t]) for t in range(n)]

    def _take_ids(self, d) -> list[str]:
        """decode a dictionary the library returned in pinned memory, then hand the memory back"""
        try:
            off = np.ctypeslib.as_array(d.offsets, shape=(d.n + 1,)).tolist()
            blob = C.string_at(d.bytes, off[-1]) if off[-1] else b""
            return [blob[a:b].decode("utf-8", "surrogateescape") for a, b in zip(off, off[1:])]
        finally:
            self._L.cco_host_free(self._h, C.cast(d.offsets, C.c_void_p))
            self._L.cco_host_free(self._h, d.bytes)

    def synth_dataset(self, types, n_users_raw: int, user_cdf: np.ndarray, user_perm: np.ndarray, min_events_per_user: int = 0,
                      raw_item_space: bool = False):
        """Bench/test utility (cco_synth_ingest): the synthetic event streams of synth.py generated in HBM and ingested there.
        types = [(n_events, seed, item_cdf float64[], item_perm int32[])].  -> resident dataset for train_dataset."""
        n = len(types)
        keep, tt = [], (N.SynthTypeT * n)()
        for t, (ne, seed, icdf, iperm) in enumerate(types):
            icdf = np.ascontiguousarray(icdf, dtype=np.float64)
            iperm = np.ascontiguousarray(iperm, dtype=np.int32)
            keep.append((icdf, iperm))
            tt[t] = N.SynthTypeT(int(ne), int(seed), len(icdf), 0, icdf.ctypes.data_as(C.POINTER(C.c_double)),
                                 iperm.ctypes.data_as(C.POINTER(C.c_int32)))
        ucdf = np.ascontiguousarray(user_cdf, dtype=np.float64)
        uperm = np.ascontiguousarray(user_perm, dtype=np.int32)
        ds = C.c_void_p()
        N.check(self._L.cco_synth_ingest(self._h, n, tt, n_users_raw, ucdf.ctypes.data_as(C.POINTER(C.c_double)),
                                         uperm.ctypes.data_as(C.POINTER(C.c_int32)), min_events_per_user, 1 if raw_item_space else 0,
                                         C.byref(ds)))
        return (ds, n)

    def dataset_shape(self, dataset, i: int):
        nr, nc, nnz = C.c_int64(), C.c_int32(), C.c_int64()
        N.check(self._L.cco_dataset_shape(dataset[0], i, C.byref(nr), C.byref(nc), C.byref(nnz)))
        return nr.value, nc.value, nnz.value

    def dataset_to_host(self, dataset, i: int, pinned: bool = True):
        """(n_rows, n_cols, row_ptr, col_idx) of matrix i of a resident dataset in (pinned) host arrays."""
        nr, nc, nnz = self.dataset_shape(dataset, i)
        rp = self.host_array(nr + 1, np.int64) if pinned else np.zeros(nr + 1, np.int64)
        ci = self.host_array(nnz, np.int32) if pinned else np.zeros(max(nnz, 1), np.int32)[:nnz]
        N.check(self._L.cco_dataset_copy_to_host(dataset[0], i, rp.ctypes.data_as(C.POINTER(C.c_int64)),
                                                 ci.ctypes.data_as(C.POINTER(C.c_int32)) if nnz else None))
        return nr, nc, rp, ci

    def dataset_matrix(self, dataset, i: int):
        """(n_rows, n_cols, row_ptr, col_idx) of matrix i of a resident dataset, copied to the host (tests)."""
        ds, _ = dataset
        nr, nc, nnz = C.c_int64(), C.c_int32(), C.c_int64()
        N.check(self._L.cco_dataset_shape(ds, i, C.byref(nr), C.byref(nc), C.byref(nnz)))
        prp, pci = C.POINTER(C.c_int64)(), C.POINTER(C.c_int32)()
        N.check(self._L.cco_dataset_download(ds, i, C.byref(prp), C.byref(pci)))
        rp = np.ctypeslib.as_array(prp, shape=(nr.value + 1,)).copy()
        ci = np.ctypeslib.as_array(pci, shape=(nnz.value,)).copy() if nnz.value else np.zeros(0, np.int32)
        self._L.cco_free(prp)
        self._L.cco_free(pci)
        return nr.value, nc.value, rp, ci

    def free_dataset(self, dataset):
        self._L.cco_dataset_free(dataset[0])

    def timer_start(self):
        N.check(self._L.cco_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = C.c_float()
        N.check(self._L.cco_timer_stop(self._h, C.byref(ms)))
        return ms.value

    # ---- debug / parity entries ---------------------------------------------------------------------------
    def debug_llr(self, k11, k12, k21, k22, flags: int = 0) -> np.ndarray:
        a = [np.ascontiguousarray(x, dtype=np.int64) for x in (k11, k12, k21, k22)]
        out = np.zeros(len(a[0]), dtype=np.float64)
        p = C.POINTER(C.c_int64)
        N.check(self._L.cco_debug_llr(self._h, len(out), *[x.ctypes.data_as(p) for x in a], flags,
                                      out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def debug_downsample(self, n_rows, n_cols, row_ptr, col_idx, max_interactions: int, seed: int, flags: int = 0):
        rp = np.ascontiguousarray(row_ptr, dtype=np.int64)
        ci = np.ascontiguousarray(col_idx, dtype=np.int32)
        m = N.as_csr_t(n_rows, n_cols, rp, ci)
        orp, oci = C.POINTER(C.c_int64)(), C.POINTER(C.c_int32)()
        raw = np.zeros(max(n_cols, 1), np.int32)
        new = np.zeros(max(n_cols, 1), np.int32)
        N.check(self._L.cco_debug_downsample(self._h, C.byref(m), max_interactions, _to_i32(seed), flags, C.byref(orp),
                                             C.byref(oci), raw.ctypes.data_as(C.POINTER(C.c_int32)),
                                             new.ctypes.data_as(C.POINTER(C.c_int32))))
        r = np.ctypeslib.as_array(orp, shape=(n_rows + 1,)).copy()
        nnz = int(r[-1])
        c = np.ctypeslib.as_array(oci, shape=(nnz,)).copy() if nnz else np.zeros(0, np.int32)
        self._L.cco_free(orp)
        self._L.cco_free(oci)
        return r, c, raw[:n_cols], new[:n_cols]

    def debug_cooccurrence(self, a, b):
        """a, b = (n_rows, n_cols, row_ptr, col_idx) canonical binary matrices -> (row_ptr, col_idx, count) of A^T B."""
        keep = []
        cs = []
        for (nr, nc, rp, ci) in (a, b):
            rp = np.ascontiguousarray(rp, dtype=np.int64)
            ci = np.ascontiguousarray(ci, dtype=np.int32)
            keep.append((rp, ci))
            cs.append(N.as_csr_t(nr, nc, rp, ci))
        orp, oci, ocn = C.POINTER(C.c_int64)(), C.POINTER(C.c_int32)(), C.POINTER(C.c_int32)()
        N.check(self._L.cco_debug_cooccurrence(self._h, C.byref(cs[0]), C.byref(cs[1]), C.byref(orp), C.byref(oci), C.byref(ocn)))
        r = np.ctypeslib.as_array(orp, shape=(a[1] + 1,)).copy()
        nnz = int(r[-1])
        c = np.ctypeslib.as_array(oci, shape=(nnz,)).copy() if nnz else np.zeros(0, np.int32)
        n = np.ctypeslib.as_array(ocn, shape=(nnz,)).copy() if nnz else np.zeros(0, np.int32)
        for p in (orp, oci, ocn):
            self._L.cco_free(p)
        return r, c, n


def _to_i32(seed: int) -> int:
    """`.toInt` of a Long seed as in URAlgorithm.scala:325,345 (wraps)."""
    s = int(seed) & 0xffffffff
    return s - (1 << 32) if s & 0x80000000 else s


_default_ctx: CcoContext | None = None


def default_context() -> CcoContext:
    """Process-wide single-GPU context on device 0 (multi-GPU jobs build theirs with distributed.context_from_env)."""
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = CcoContext(device=0)
    return _default_ctx


class SimilarityAnalysis:
    """Drop-in for the two static calls of URAlgorithm.calcAll."""

    @staticmethod
    def crossOccurrenceDownsampled(datasets: Sequence[DownsamplableCrossOccurrenceDataset], randomSeed: int = 0xdeadbeef,
                                   ctx: CcoContext | None = None, flags: int = 0) -> list[IndexedDataset]:
        """URAlgorithm.scala:343-346.  datasets[0] is the primary (A).  Returns one IndexedDataset per input,
        rowIDs = A.columnIDs, columnIDs = B_i.columnIDs, values = LLR, rows sorted (llr desc, col asc)."""
        if len(datasets) == 0:
            raise N.CcoInvalidArgument(N.E_INVALID_ARG, "datasets is empty")
        ctx = ctx or default_context()
        a = datasets[0].iD
        mats = [(d.iD.n_rows, d.iD.n_cols, d.iD.row_ptr, d.iD.col_idx) for d in datasets]
        params = [(d.maxElementsPerRow, d.maxInterestingElements, d.minLLROpt) for d in datasets]
        res = ctx.train_csr(mats, params, randomSeed, flags)
        out = []
        for d, (rb, re_, nc, rp, ci, ll, cn) in zip(datasets, res):
            if ctx.world_size == 1:
                out.append(a.create(rp, ci, a.column_ids, d.iD.column_ids, ll, cn))
            else:   # this rank's row slice, padded to the full primary-item row space
                full = np.zeros(a.n_cols + 1, dtype=np.int64)
                full[rb + 1:re_ + 1] = rp[1:]
                full[re_ + 1:] = rp[-1]
                out.append(a.create(full, ci, a.column_ids, d.iD.column_ids, ll, cn))
        return out

    @staticmethod
    def cooccurrencesIDSs(indexedDatasets: Sequence[IndexedDataset], randomSeed: int = 0xdeadbeef,
                          maxInterestingItemsPerThing: int = 50, maxNumInteractions: int = 500,
                          ctx: CcoContext | None = None, flags: int = 0) -> list[IndexedDataset]:
        """URAlgorithm.scala:323-329: one global (k, m) for every matrix."""
        ds = [DownsamplableCrossOccurrenceDataset(i, maxNumInteractions, maxInterestingItemsPerThing, None)
              for i in indexedDatasets]
        return SimilarityAnalysis.crossOccurrenceDownsampled(ds, randomSeed, ctx, flags)
