#!/usr/bin/env python
"""bench.py -- CCO train events/sec to indicator model (BASELINE.json metric) on N B200s.

A "step" is one complete pass of the hot path (downsample -> A'^T A' / A'^T B'_i co-occurrence -> LLR -> top-k)
over the whole synthetic workload.  Default workload: BASELINE.json configs[2] ("C3": 1M users x 100K items,
50M events, 1 primary + 3 secondary event types, k=50), the configuration the 1/2/4/8-GPU metric is quoted on
and which fits one GPU.  `--workload C2` runs configs[1].

  value    : events/s with the input matrices already resident in HBM (cco_dataset_upload outside the timed
             region; results left packed in HBM), timed with CUDA events on the library's launch stream.
  e2e      : events/s through the public C-ABI call cco_train with HOST (pinned) buffers: H2D of every matrix,
             compute, D2H of every indicator inside the timed region.
  roofline : algorithmic bytes of the fused A'^T B' row kernel (SURVEY.md 8d formula) / its CUDA-event time.
  cpu_baseline : the oracle (CPU restatement of Mahout's algorithm, OpenMP) on a bounded sample, rank 0, N=1.

`--impl reference` times the reference's own CPU implementation of the path.  The reference's implementation is
Apache Mahout 0.13.0 on Spark (JVM), which is neither in /root/reference nor runnable in this image, so that arm
runs the oracle port on all host cores (kind "port").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import synth  # noqa: E402

METRIC = "CCO train events/sec to indicator model"
UNIT = "events/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("CCO_BENCH_WORKLOAD", "C3"))
    ap.add_argument("--cpu-sample", default="auto", help="oracle sample: 'full', 'none' or a user fraction like 0.1")
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the indicators of the last timed steps to DIR/<name>.npy (float64; see dump_outputs)")
    a = ap.parse_args()
    if a.dump_outputs is not None and a.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
    return a


# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.p = gpu_index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax = float(r[2])
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def algorithmic_bytes(st, i: int, n_items_a: int) -> float:
    """SURVEY.md 8(d): bytes_alg(A,B) = 4 nnz(A') + 8 (I_A+1) + 8 nnz(A') + 4 P + 4 nnz(C) + 4 I_A + 12 out_nnz."""
    nnz_a = st.nnz_downsampled[0]
    return (4.0 * nnz_a + 8.0 * (n_items_a + 1) + 8.0 * nnz_a + 4.0 * st.products[i] + 4.0 * st.distinct_cells[i]
            + 4.0 * n_items_a + 12.0 * st.out_nnz[i])


DUMP_BYTES = 56 << 20   # --dump-outputs stays under 64 MB: larger models are cut to a sample of their rows


def dump_outputs(out_dir: str, e2e, resident, top_k: int):
    """--dump-outputs: what the last timed steps returned, as float64 .npy files, so that two builds can be compared output
    for output.  e2e: the result of cco_train, [(row_begin, row_end, n_cols, row_ptr, col_idx, llr, count)] per indicator
    (the end-to-end leg asks for no counts); resident: the resident step's result, of which only row_ptr reaches the host.
      rows.npy                           primary-item rows written: every row, or a fixed seeded sample when the model is
                                         larger than DUMP_BYTES (the same rows for every indicator)
      indicator<i>_row_len.npy           kept cells per written row (cco_train)
      indicator<i>_col_idx.npy           their column ids, row after row, in result order (cco_train)
      indicator<i>_llr.npy               their LLR values (cco_train)
      indicator<i>_resident_row_len.npy  kept cells per written row (resident step)"""
    n_rows = len(e2e[0][3]) - 1
    per_row = 8 + len(e2e) * (8 + 8 + 16 * top_k)      # a row holds at most top_k cells
    n = min(n_rows, DUMP_BYTES // per_row)
    rows = np.arange(n_rows) if n == n_rows else np.sort(np.random.default_rng(0).choice(n_rows, n, replace=False))
    arrays = {"rows": rows}
    for i, (r, d) in enumerate(zip(e2e, resident)):
        rp = r[3]
        start, lens = rp[rows], rp[rows + 1] - rp[rows]
        take = np.repeat(start - np.cumsum(lens) + lens, lens) + np.arange(int(lens.sum()))
        arrays[f"indicator{i}_row_len"] = lens
        arrays[f"indicator{i}_col_idx"] = r[4][take]
        arrays[f"indicator{i}_llr"] = r[5][take]
        arrays[f"indicator{i}_resident_row_len"] = d[3][rows + 1] - d[3][rows]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def ncu_traffic(workload: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of the row-kernel launches of ONE indicator, from the committed
    `ncu --set full` capture (profiles/r02_k_rows_traffic.json) -- quoted only if that capture was taken on this very
    build of the kernels and on this workload, else None (never a stale figure)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_k_rows_traffic.json")))
        if d["workload"] == workload and d.get("build") == source_build_id():
            return d["dram_bytes_per_indicator"]
    except Exception:
        pass
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------------------
def _pin_openmp():
    """Thread placement of the CPU arm, set before libgomp is loaded: one thread per hardware thread, no migration.
    (torchrun exports OMP_NUM_THREADS=1 to its children; orc_train overrides the count itself.)"""
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "threads")
    os.environ.setdefault("OMP_DYNAMIC", "false")


def sample_workload(name: str, sample: str, ctx=None, pinned: bool = False):
    """the workload (sample == "full") or the same generator at a fraction of the users and events.  ctx: generate and
    ingest on the B200 (seconds); None: numpy on the host (minutes at the 50M-event shapes)."""
    if sample == "full":
        return synth.make(name, ctx=ctx, pinned=pinned), f"full {name} workload"
    f = float(sample)
    c = synth.CONFIGS[name]
    sw = synth.make(name, ctx=ctx, pinned=pinned, n_users=max(int(c["n_users"] * f), 1), n_events=max(int(c["n_events"] * f), c["n_types"]))
    return sw, (f"{name} generator at {f:g} of the users and events ({sw.n_users} users x {sw.n_items} items, "
                f"{sw.n_events} events, {sw.n_types} types), same item space/k/m")


def time_oracle(sw, seed: int, warmup: int, steps: int):
    """-> (median seconds per train, all step times, threads used).  Times orc_train only (no numpy copies)."""
    from oracle import oracle as orc
    orc.build()
    threads = host_threads()
    mats = [orc.Csr(*m) for m in sw.mats]
    prm = [orc.Params(*p) for p in sw.params]
    for _ in range(warmup):
        orc.time_train(mats, prm, seed, 0, threads)
    ts = [orc.time_train(mats, prm, seed, 0, threads)[0] for _ in range(max(steps, 1))]
    return float(np.median(ts)), ts, threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads_before = host_threads()
    _pin_openmp()
    sample = auto_sample(args.workload) if args.cpu_sample in ("auto", "none") else args.cpu_sample
    gen_ctx = None
    try:   # the input generator (not the thing measured) runs on the GPU when the box has one: seconds instead of minutes
        import universal_recommender_b200 as ur
        gen_ctx = ur.CcoContext(device=int(os.environ.get("LOCAL_RANK", "0")))
    except Exception:
        gen_ctx = None
    sw, desc = sample_workload(args.workload, sample, gen_ctx)
    if gen_ctx is not None:
        sw.mats = [(nr, nc, np.array(rp), np.array(ci)) for (nr, nc, rp, ci) in sw.mats]
        gen_ctx.close()
    dt, ts, threads = time_oracle(sw, args.seed, args.warmup, args.steps)
    v = sw.n_events / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "int32+f64", "data": "synthetic",
            "config": {"workload": workload_desc(args.workload), "sample": desc,
                       "timing": "median of the timed steps (orc_train only); min/max in step_ms_min_max",
                       "step_ms_min_max": [round(min(ts) * 1e3, 1), round(max(ts) * 1e3, 1)],
                       "omp": {k: os.environ.get(k) for k in ("OMP_PROC_BIND", "OMP_PLACES")}},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc,
                             "note": "CPU restatement of Mahout 0.13.0 SimilarityAnalysis (oracle/cco_oracle.c, OpenMP); the "
                                     "reference's own Mahout-on-Spark path needs a JVM and is not runnable in this image"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


try:   # taken at import time: an OpenMP runtime loaded later with OMP_PROC_BIND pins the main thread to ONE cpu
    _HOST_THREADS = max(len(os.sched_getaffinity(0)), 1)
except AttributeError:
    _HOST_THREADS = os.cpu_count() or 1


def host_threads() -> int:
    """All host threads this process may use -- NOT OMP_NUM_THREADS, which torchrun pins to 1 for its children."""
    return _HOST_THREADS


def auto_sample(workload: str) -> str:
    """The oracle finishes the whole C3 workload in a few seconds on the GPU box's host cores, so the CPU arm runs the
    FULL workload up to C3; the 10M-user shapes use a tenth of the users and events."""
    return "full" if synth.CONFIGS[workload]["n_events"] <= 50_000_000 else "0.1"


def workload_desc(name: str) -> str:
    c = synth.CONFIGS[name]
    return (f"{name}: synthetic Zipf (items s=1.0, users s=0.5), {c['n_users']} users x {c['n_items']} items, {c['n_events']} events, "
            f"1 primary + {c['n_types'] - 1} secondary event types, maxCorrelatorsPerItem=50, maxItemsPerUser=500")


# ---------------------------------------------------------------------------------------------------------
class ShmModel:
    """N > 1 end-to-end leg: the caller of the reference boundary is ONE process (URAlgorithm.train on the Spark driver,
    URAlgorithm.scala:292-307), so the model is only "back" when every rank's row slice sits in memory that process can
    read.  One /dev/shm segment holds a region per rank; the region (minus a 4 KB header) is that rank's RESULT ARENA
    (cco_config_t.result_arena): the library page-locks it and the device->host copies of the indicators land in it
    directly.  After the train a rank only publishes where its arrays are; rank 0 reads every slice in place."""

    HEAD = 4096

    def __init__(self, rank: int, world: int, n_types: int, n_items: int, top_k: int, tag: str):
        self.rank, self.world, self.n_types = rank, world, n_types
        per_ind = 8 * (n_items + 1) + 16 * n_items * top_k + 4096
        # a rank holds ~1/world of the rows (work-balanced): three times that share, at least 64 MB; a result that still
        # does not fit is allocated by the library outside the arena and publish() says so
        share = n_types * per_ind if world <= 2 else 3 * n_types * per_ind // world
        self.per_rank = (self.HEAD + max(share, 64 << 20) + (1 << 21) - 1) & ~((1 << 21) - 1)
        self.path = f"/dev/shm/cco_bench_model_{tag}"
        if rank == 0:
            with open(self.path, "wb") as f:
                f.truncate(self.per_rank * world)
        self.mm = None

    def open(self):
        self.mm = np.memmap(self.path, dtype=np.uint8, mode="r+")
        return self.mm[self.rank * self.per_rank + self.HEAD:(self.rank + 1) * self.per_rank]   # this rank's arena

    def publish(self, res):
        """res: views of this rank's result arrays (they live in the arena): record their offsets in the header"""
        base = self.rank * self.per_rank
        addr0 = self.mm.ctypes.data
        head = np.zeros(8 * self.n_types, dtype=np.int64)
        for i, (rb, re_, nc, rp, ci, ll, cn) in enumerate(res):
            nnz = int(rp[-1])
            offs = [a.ctypes.data - addr0 if a.size else 0 for a in (rp, ci, ll, cn)]
            assert all(o == 0 or base <= o < base + self.per_rank for o in offs), "result outside the arena"
            head[8 * i:8 * i + 8] = (rb, re_, nnz, offs[0], offs[1], offs[2], offs[3], nc)
        self.mm[base:base + head.nbytes] = head.view(np.uint8)

    def model(self):
        """rank 0: [(row_begin, row_end, row_ptr, col_idx, llr)] per indicator per rank, zero-copy views"""
        out = []
        for r in range(self.world):
            base = r * self.per_rank
            head = self.mm[base:base + 64 * self.n_types].view(np.int64)
            sl = []
            for i in range(self.n_types):
                rb, re_, nnz, o_rp, o_ci, o_ll, o_cn, nc = (int(x) for x in head[8 * i:8 * i + 8])
                rp = self.mm[o_rp:o_rp + 8 * (re_ - rb + 1)].view(np.int64)
                ci = self.mm[o_ci:o_ci + 4 * nnz].view(np.int32)
                ll = self.mm[o_ll:o_ll + 8 * nnz].view(np.float64) if o_ll else np.zeros(0, np.float64)
                cn = self.mm[o_cn:o_cn + 4 * nnz].view(np.int32) if o_cn else np.zeros(0, np.int32)
                sl.append((rb, re_, rp, ci, ll, cn, nc))
            out.append(sl)
        return out

    def close(self):
        self.mm = None
        if self.rank == 0:
            try:
                os.unlink(self.path)
            except OSError:
                pass


def source_build_id() -> str:
    """hash of the source file that holds k_rows (cco_kernels.cuh): the committed ncu DRAM-traffic figure of k_rows is
    only quoted for the row kernel it was measured on (the entry-parallel preparation kernels live in cco_sampler.cuh)"""
    import hashlib
    h = hashlib.sha1()
    for f in ("cco_kernels.cuh",):
        try:
            h.update(open(os.path.join(ROOT, "universal_recommender_b200", "csrc", f), "rb").read())
        except OSError:
            pass
    return h.hexdigest()[:12]


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist

    import universal_recommender_b200 as ur
    from universal_recommender_b200 import _native as N
    from universal_recommender_b200 import distributed as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this framework has no CPU fallback")
    if args.dump_outputs is not None and world > 1:
        raise SystemExit("bench.py: --dump-outputs writes one process's model: run it on one GPU")
    torch.cuda.set_device(local_rank)
    uid = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        box = [ur.CcoContext.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        uid = box[0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    shm, arena = None, None
    if world > 1:
        c = synth.CONFIGS[args.workload]
        shm = ShmModel(rank, world, c["n_types"], c["n_items"], 50, os.environ.get("MASTER_PORT", "0"))
        barrier()
        arena = shm.open()
    ctx = ur.CcoContext(device=local_rank, rank=rank, world_size=world, nccl_unique_id=uid, result_arena=arena)
    # synthetic events are generated and ingested on the device (cco_synth_ingest; every rank builds the same matrices on
    # its own GPU) and copied into pinned host memory: what the JNI shim's direct ByteBuffers would hold
    t_gen = time.perf_counter()
    w = synth.make(args.workload, ctx=ctx, pinned=True)
    t_gen = time.perf_counter() - t_gen
    n_items_a = w.mats[0][1]
    pinned = w.mats
    h2d_bytes = sum(m[2].nbytes + m[3].nbytes for m in pinned)
    flags = ur.FLAG_ASSUME_CANONICAL

    # ---- device-resident throughput ------------------------------------------------------------------------
    ds = ctx.upload(pinned, flags)
    for _ in range(args.warmup):
        ctx.train_dataset(ds, w.params, args.seed, flags | N.FLAG_RESULT_ON_DEVICE, copy_arrays=False)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:   # one NVML poller per job: eight of them contend for the driver lock and slow every rank's launches
        sampler.start()
    ctx.timer_start()
    rows_ms, launches = 0.0, 0
    alg_bytes = 0.0
    for _ in range(args.steps):
        resident_last = ctx.train_dataset(ds, w.params, args.seed, flags | N.FLAG_RESULT_ON_DEVICE, copy_arrays=False)
        st = ctx.last_stats
        rows_ms += sum(st.ms_indicator)
        launches += st.n_kernel_launches
        alg_bytes += sum(algorithmic_bytes(st, i, n_items_a) for i in range(w.n_types))
    ms_dev = ctx.timer_stop()
    barrier()
    clocks = sampler.stop()
    ms_dev = max_over_ranks(ms_dev)
    ms_per_step = ms_dev / args.steps
    value = w.n_events / (ms_per_step * 1e-3)
    st_last = ctx.last_stats
    ctx.free_dataset(ds)

    # ---- end to end through cco_train with host buffers ------------------------------------------------------
    # N > 1: the timed region ends when rank 0 can read the WHOLE model (every rank's row slice) from host memory
    # the indicator matrices of the reference boundary are (column id, LLR) per row (IndexedDataset values = LLR); the
    # co-occurrence count k11 is a by-product nothing downstream reads, so the end-to-end leg does not copy it back
    flags_e2e = flags | N.FLAG_RESULT_NO_COUNT

    def e2e_step(keep: bool = False):
        res, h = ctx.train_csr(pinned, w.params, args.seed, flags_e2e, keep=True)
        nbytes = sum(r[3].nbytes + r[4].nbytes + r[5].nbytes + r[6].nbytes for r in res)
        if shm is not None:
            shm.publish(res)
            dist.barrier()
            if rank == 0:
                model = shm.model()
                assert sum(sl[0][1] - sl[0][0] for sl in model) == n_items_a
                assert all(int(sl[i][2][-1]) == len(sl[i][3]) for sl in model for i in range(w.n_types))
            dist.barrier()          # the slices are read in place: nobody frees before rank 0 is done
        if keep:                    # --dump-outputs reads the last step's arrays after the timed region
            return nbytes, res, h
        ctx.free_result(h)
        return nbytes, None, None

    for _ in range(args.warmup):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    d2h_bytes, last_res, last_h = 0, None, None
    for s in range(args.steps):
        d2h_bytes, last_res, last_h = e2e_step(keep=args.dump_outputs is not None and s == args.steps - 1)
    torch.cuda.synchronize()
    wall_e2e = (time.perf_counter() - t0) * 1e3
    if last_h is not None:
        dump_outputs(args.dump_outputs, last_res, resident_last, max(p[1] for p in w.params))
        ctx.free_result(last_h)
    barrier()
    ms_e2e = max_over_ranks(wall_e2e) / args.steps
    e2e_value = w.n_events / (ms_e2e * 1e-3)
    d2h_total = int(sum_over_ranks(float(d2h_bytes)))

    # ---- parity gate of this run (SURVEY.md 8d): the CUDA path against the oracle on the same input --------------
    sample = auto_sample(args.workload) if args.cpu_sample in ("auto", "none") else args.cpu_sample
    if sample == "full":
        sw, sdesc, spinned = w, f"full {w.name} workload", pinned
    else:
        sw, sdesc = sample_workload(args.workload, sample, ctx, pinned=True)
        spinned = sw.mats
    parity = None
    if world == 1:
        merged = ctx.train_csr(spinned, sw.params, args.seed, flags)
        ph = None
    else:
        # every rank's slice sits in its result arena (= its region of the shared segment): rank 0 merges them in place
        local, ph = ctx.train_csr(spinned, sw.params, args.seed, flags, keep=True)
        shm.publish(local)
        dist.barrier()
        if rank == 0:
            model = shm.model()
            merged = []
            for i in range(sw.n_types):
                m = D.merge_row_slices([(sl[i][0], sl[i][1], sl[i][6], sl[i][2], sl[i][3], sl[i][4], sl[i][5]) for sl in model])
                merged.append((0, m[0], m[1], m[2], m[3], m[4], m[5]))
    if rank == 0:
        from oracle import oracle as orc
        from oracle import parity as par
        ref = orc.train([orc.Csr(*m) for m in sw.mats], [orc.Params(*p) for p in sw.params], args.seed, 0, host_threads())
        parity = par.compare(ref, merged, sw.n_users)
        parity["sample"] = sdesc
        parity["n_gpus"] = world
    if world > 1:
        dist.barrier()
        ctx.free_result(ph)

    # ---- roofline of the fused A'^T B' row kernel (all ranks' rows together) -----------------------------------
    peak, peak_src = measured_peaks()
    alg_total = sum_over_ranks(alg_bytes)
    rows_ms_max = max_over_ranks(rows_ms)
    achieved = alg_total / (rows_ms_max * 1e-3) / 1e9 / max(world, 1) if rows_ms_max > 0 else 0.0
    n_ind = w.n_types * args.steps
    roofline = {"bound": "hbm", "kernel": "k_rows (fused A'^T B' count + LLR + top-k; one set of work-binned launches per indicator, "
                                          "concurrent on separate streams)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                "traffic": ncu_traffic(args.workload),
                "algorithmic_bytes_per_indicator": alg_total / max(world, 1) / n_ind,
                "ms_per_indicator": rows_ms_max / n_ind,
                "note": "per GPU; one 'launch' = the bin launches of one indicator (they run concurrently, so only their common CUDA-event "
                        "bracket is a duration); achieved = SURVEY 8(d) algorithmic bytes of this rank's rows / that bracket",
                "secondary_ceilings": {"llr_cells_evaluated_per_step": int(sum_over_ranks(float(sum(st_last.llr_evaluated)))),
                                       "fp64_xlogx_per_s_measured": 3.48e11, "smem_atomic_products_per_s_measured": 1.03e12}}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int32+f64", "data": "synthetic",
            "config": {"workload": workload_desc(args.workload), "parallelism": f"item-row sharding x{world}",
                       "l2": "inputs (%.0f MB) larger than the 126 MB L2; no explicit flush" % (h2d_bytes / 1e6)
                       if h2d_bytes > 126e6 else "inputs fit L2 (%.0f MB); no explicit flush" % (h2d_bytes / 1e6),
                       "resident": "value: matrices resident in HBM, indicators left packed in HBM",
                       "e2e": "cco_train on pinned host CSR -> indicator arrays in host memory" +
                              (" readable by rank 0 (every rank's result arena is its region of one shared segment; the merge is "
                               "zero-copy and inside the timed region)" if world > 1 else ""),
                       "products_per_step": int(sum_over_ranks(float(sum(st_last.products)))),
                       "distinct_cells_per_step": int(sum_over_ranks(float(sum(st_last.distinct_cells)))),
                       "datagen_s": round(t_gen, 1), "build": source_build_id(),
                       "stage_ms_last_resident_step": {"prepare": round(st_last.ms_prepare, 3), "indicators_total": round(st_last.ms_cooccurrence, 3),
                                                       "row_kernels": [round(x, 3) for x in st_last.ms_indicator],
                                                       "prepare_stages": [round(x, 3) for x in (st_last.ms_prep_stage or [])[:7]]}},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": d2h_total,
                    "ms_per_step": ms_e2e},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "parity": parity}
    line["cpu_baseline"] = None
    if rank == 0 and world == 1 and args.cpu_sample != "none":
        # the CPU arm runs in its own process (thread pinning set before its OpenMP runtime loads, no GPU-arm threads
        # around): `bench.py --impl reference` on the same sample, 3 timed steps after 1 warm-up, median
        try:
            env = {k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS", "RANK", "WORLD_SIZE", "LOCAL_RANK")}
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload,
                                "--cpu-sample", sample, "--steps", "3", "--warmup", "1", "--seed", str(args.seed)],
                               capture_output=True, text=True, env=env, timeout=900)
            ref_line = json.loads([l for l in p.stdout.splitlines() if l.strip().startswith("{")][-1])
            cb = ref_line["cpu_baseline"]
            cb["seconds"] = round(ref_line["ms_per_step"] / 1e3, 3)
            cb["timing"] = "median of 3 timed steps after 1 warm-up, separate process"
            line["cpu_baseline"] = cb
        except Exception as e:   # the GPU numbers stand on their own; say why the CPU leg is missing
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": host_threads(), "kind": "port", "sample": sdesc,
                                    "error": repr(e)[:200]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if shm is not None:
        shm.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and parity is not None and not parity.get("ok"):
        raise SystemExit(f"bench.py: PARITY FAILURE against the oracle: {parity}")


if __name__ == "__main__":
    main()
