// cco_api.cu -- C ABI (include/cco_b200.h) and host orchestration of the sm_100a CCO model builder.
//
// Replaces Mahout's SimilarityAnalysis.cooccurrencesIDSs / crossOccurrenceDownsampled as called from
// /root/reference/src/main/scala/URAlgorithm.scala:323-329,343-346.  No CPU fallback: every compute
// entry fails with CCO_E_CUDA when no CUDA device is usable.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <cub/cub.cuh>
#include <nvtx3/nvToolsExt.h>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/cco_b200.h"
#include "cco_kernels.cuh"
#include "cco_sampler.cuh"
#include "cco_format.cuh"
#include "cco_strings.cuh"
#include "cco_model.cuh"

namespace cco {

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int set_error(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return code;
}
#define CK(expr)                                                                                      \
  do {                                                                                                \
    cudaError_t _e = (expr);                                                                          \
    if (_e != cudaSuccess)                                                                            \
      return set_error(_e == cudaErrorMemoryAllocation ? CCO_E_OOM : CCO_E_CUDA, "%s: %s (%s:%d)", #expr, \
                       cudaGetErrorString(_e), __FILE__, __LINE__);                                   \
  } while (0)
#define CKR(expr)            \
  do {                       \
    int _r = (expr);         \
    if (_r != CCO_OK) return _r; \
  } while (0)

// ------------------------------------------------------------------------------------------------
// NCCL, loaded lazily (only multi-GPU contexts need it)
// ------------------------------------------------------------------------------------------------
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
struct Nccl {
  void *h = nullptr;
  int (*GetUniqueId)(ncclUniqueId *) = nullptr;
  int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  int (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*Broadcast)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
};
static Nccl g_nccl;
static std::mutex g_nccl_mu;
static int load_nccl() {
  std::lock_guard<std::mutex> lk(g_nccl_mu);
  if (g_nccl.h) return CCO_OK;
  void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return set_error(CCO_E_NCCL, "cannot load libnccl.so.2: %s", dlerror());
#define SYM(field, name)                                                         \
  *(void **)(&g_nccl.field) = dlsym(h, name);                                    \
  if (!g_nccl.field) return set_error(CCO_E_NCCL, "libnccl: missing symbol %s", name);
  SYM(GetUniqueId, "ncclGetUniqueId")
  SYM(CommInitRank, "ncclCommInitRank")
  SYM(CommInitAll, "ncclCommInitAll")
  SYM(CommDestroy, "ncclCommDestroy")
  SYM(AllReduce, "ncclAllReduce")
  SYM(AllGather, "ncclAllGather")
  SYM(Broadcast, "ncclBroadcast")
  SYM(GroupStart, "ncclGroupStart")
  SYM(GroupEnd, "ncclGroupEnd")
  SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
  g_nccl.h = h;
  return CCO_OK;
}
constexpr int kNcclInt32 = 2, kNcclUint32 = 3, kNcclSum = 0, kNcclMax = 2;  // ncclInt32, ncclUint32, ncclSum, ncclMax (nccl.h enum values)

}  // namespace cco

using namespace cco;

// ------------------------------------------------------------------------------------------------
// context / result objects
// ------------------------------------------------------------------------------------------------
struct PinnedBuf {
  void *p;
  size_t cap;
  bool used;
};

// shared by the per-GPU member contexts of a group (single-process multi-GPU) context
struct GroupShared {
  int world = 0;
  std::mutex mu;
  std::condition_variable cv;
  int arrived = 0;
  unsigned long long generation = 0;
  std::vector<long long> totals;   // per rank: kept cells of the indicator being merged
  struct cco_result *merged = nullptr;
  int status = 0;                  // first failure of any member thread
  char err[512] = "";
  void barrier() {
    std::unique_lock<std::mutex> lk(mu);
    const unsigned long long g = generation;
    if (++arrived == world) {
      arrived = 0;
      ++generation;
      cv.notify_all();
    } else {
      cv.wait(lk, [&] { return generation != g; });
    }
  }
};

struct cco_ctx {
  int device = 0, rank = 0, world = 1;
  int sm_count = 0;
  size_t smem_optin = 0;
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  cudaEvent_t ev[8] = {};
  cudaEvent_t tev[2] = {};
  cudaEvent_t copy_ev[2] = {};
  cudaStream_t bin_stream[8] = {};
  cudaStream_t sched_stream = nullptr;   // row scheduling of indicator i+1 runs here, beside the row kernels of indicator i
  cudaEvent_t bin_ev[9] = {};
  std::vector<PinnedBuf> pinned;
  std::mutex mu;
  ncclComm_t comm = nullptr;
  int launches = 0;
  // mailbox for small device -> host results (mapped pinned memory written by k_mail_bytes).  Records are closed into
  // groups; a group is complete when its event has fired, so the host can wait for indicator i's numbers while the GPU
  // already runs indicator i + 1 (no stream-wide synchronisation).
  unsigned char *mail_h = nullptr, *mail_d = nullptr;
  size_t mail_used = 0;
  struct MailItem { void *dst; size_t off, n; int group; };
  std::vector<MailItem> mail_pending;
  std::vector<cudaEvent_t> mail_ev;
  int mail_group = 0;
  // optional caller-provided result arena (cco_config_t.result_arena): results are bump-allocated from it, e.g. a
  // shared-memory segment another process maps, so that no copy separates this rank's slice from the reader
  unsigned char *arena = nullptr;
  size_t arena_bytes = 0, arena_used = 0;
  int arena_live = 0;
  bool arena_registered = false;
  // small per-train device scratch comes from slabs the context keeps (bump allocation: no CUDA call per buffer), and the
  // per-train events come from a cached pool: a train of a small shape is bound by host API calls, not by its kernels
  struct Slab { unsigned char *p; size_t cap; };
  std::vector<Slab> slabs;
  size_t slab_idx = 0, slab_off = 0;
  bool slab_busy = false;
  std::vector<cudaEvent_t> ev_timing, ev_plain;
  size_t ev_timing_used = 0, ev_plain_used = 0;
  // group context: the leader owns one member context per GPU (members[0]->device = devices[0], ...)
  std::vector<cco_ctx *> members;
  GroupShared *gshared = nullptr;   // set on members

  void *pinned_get(size_t bytes, bool for_result = true) {
    std::lock_guard<std::mutex> lk(mu);
    if (bytes == 0) bytes = 16;
    if (arena && for_result) {
      const size_t off = (arena_used + 255) & ~(size_t)255;
      if (off + bytes <= arena_bytes) {
        arena_used = off + bytes;
        ++arena_live;
        return arena + off;
      }
    }
    int best = -1;
    for (size_t i = 0; i < pinned.size(); ++i)
      if (!pinned[i].used && pinned[i].cap >= bytes && (best < 0 || pinned[i].cap < pinned[best].cap)) best = (int)i;
    if (best >= 0) {
      pinned[best].used = true;
      return pinned[best].p;
    }
    void *p = nullptr;
    size_t cap = (bytes + (1u << 20) - 1) & ~((size_t)(1u << 20) - 1);
    if (cudaHostAlloc(&p, cap, cudaHostAllocPortable) != cudaSuccess) return nullptr;
    pinned.push_back({p, cap, true});
    return p;
  }
  void pinned_put(void *p) {
    std::lock_guard<std::mutex> lk(mu);
    if (arena && (unsigned char *)p >= arena && (unsigned char *)p < arena + arena_bytes) {
      if (--arena_live <= 0) { arena_live = 0; arena_used = 0; }   // every result freed: the arena starts over
      return;
    }
    for (auto &b : pinned)
      if (b.p == p) b.used = false;
  }
};

struct ResultMat {
  int64_t row_begin = 0, row_end = 0;
  int32_t n_cols = 0;
  int64_t *row_ptr = nullptr;
  int32_t *col = nullptr;
  double *llr = nullptr;
  int32_t *cnt = nullptr;
};
// A dataset holds, per event type, the block of user rows this context works on: the whole matrix on a single GPU,
// this rank's user block [row_base, row_base + n_local) in a multi-GPU job (each GPU uploads 1/N of the rows).
struct cco_dataset {
  cco_ctx *ctx = nullptr;
  int n_mats = 0;
  long long n_users = 0;           // U, global
  long long row_base = 0, n_local = 0;
  std::vector<long long> n_cols, nnz;   // nnz: stored entries of the WHOLE matrix as handed in
  std::vector<long long *> rp;   // device, indexable by local row 0 .. n_local (values index `col`)
  std::vector<int32_t *> col;    // device, indexable by the values of rp
  std::vector<void *> rp_alloc, col_alloc;   // what to free (rp/col may be offset views of these)
  std::vector<long long> block_cap;          // per matrix: largest raw entry count of any rank's user block
  std::vector<long long> q_lo, q_hi;         // per matrix: the offsets rp[0], rp[n_local] of the block (host-known)
  std::vector<cudaEvent_t> ready;  // per matrix: host->device copy finished (copy stream)
  bool h2d_pending = false;        // uploaded asynchronously: ms_h2d is read when the train joins
  bool validated = false;          // k_check_rows has run (and the rows are canonical)
  bool whole = false;              // rp_alloc / col_alloc hold the WHOLE matrices (device-built datasets, single-GPU uploads)
  float ms_h2d = 0;
};

struct cco_result {
  cco_ctx *ctx = nullptr;
  std::vector<ResultMat> mats;
  cco_stats_t stats;
};

namespace cco {

// per-call device arena on top of the stream-ordered allocator
struct Arena {
  cudaStream_t s;
  cco_ctx *c;   // non-null: buffers up to kSlabMax bytes are bump-allocated from the context's slabs
  std::vector<void *> ptrs;
  static constexpr size_t kSlabMax = 8u << 20, kSlabBytes = 64u << 20;
  explicit Arena(cudaStream_t st, cco_ctx *ctx = nullptr) : s(st), c(ctx && !ctx->slab_busy ? ctx : nullptr) {
    if (c) {
      c->slab_busy = true;
      c->slab_idx = 0;
      c->slab_off = 0;
    }
  }
  ~Arena() {
    for (void *p : ptrs) cudaFreeAsync(p, s);
    if (c) c->slab_busy = false;
  }
  void *bump(size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    while (true) {
      if (c->slab_idx < c->slabs.size()) {
        cco_ctx::Slab &sl = c->slabs[c->slab_idx];
        if (c->slab_off + bytes <= sl.cap) {
          void *p = sl.p + c->slab_off;
          c->slab_off += bytes;
          return p;
        }
        ++c->slab_idx;
        c->slab_off = 0;
        continue;
      }
      void *p = nullptr;
      if (cudaMalloc(&p, kSlabBytes) != cudaSuccess) return nullptr;   // warm-up trains only; kept until cco_destroy
      c->slabs.push_back({(unsigned char *)p, kSlabBytes});
    }
  }
  template <typename T>
  int alloc(T **out, size_t n) {
    void *p = nullptr;
    size_t bytes = std::max<size_t>(n * sizeof(T), 16);
    if (c && bytes <= kSlabMax) {
      p = bump(bytes);
      if (!p) return set_error(CCO_E_OOM, "cudaMalloc(scratch slab) failed");
      *out = (T *)p;
      return CCO_OK;
    }
    cudaError_t e = cudaMallocAsync(&p, bytes, s);
    if (e != cudaSuccess) return set_error(CCO_E_OOM, "cudaMallocAsync(%zu bytes): %s", bytes, cudaGetErrorString(e));
    ptrs.push_back(p);
    *out = (T *)p;
    return CCO_OK;
  }
  void release(void *p) {   // slab memory is simply not reused within a train
    for (size_t i = 0; i < ptrs.size(); ++i)
      if (ptrs[i] == p) {
        cudaFreeAsync(p, s);
        ptrs.erase(ptrs.begin() + i);
        return;
      }
  }
};
// cached events of a train (reset at its start)
static int pooled_event(cco_ctx *c, bool timing, cudaEvent_t *out) {
  std::vector<cudaEvent_t> &pool = timing ? c->ev_timing : c->ev_plain;
  size_t &used = timing ? c->ev_timing_used : c->ev_plain_used;
  if (used == pool.size()) {
    cudaEvent_t e;
    CK(timing ? cudaEventCreate(&e) : cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    pool.push_back(e);
  }
  *out = pool[used++];
  return CCO_OK;
}

// NVTX ranges per stage (SURVEY.md section 5: tracing); header-only NVTX3, a no-op unless a profiler is attached
static inline void nvtx_push(const char *name) { nvtxRangePushA(name); }
static inline void nvtx_pop() { nvtxRangePop(); }

static inline int grid_for(long long work_items, int block, int sm_count, int waves = 8) {
  long long g = (work_items + block - 1) / block;
  long long cap = (long long)sm_count * waves;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

constexpr size_t kMailBytes = 1 << 16;
// enqueue "copy n bytes from device to *dst_host"; the value is there after the group it belongs to has been waited for
static int mail_fetch(cco_ctx *c, void *dst_host, const void *src_dev, size_t n) {
  size_t off = (c->mail_used + 7) & ~(size_t)7;
  if (off + n > kMailBytes) return set_error(CCO_E_CUDA, "internal: mailbox overflow");
  k_mail_bytes<<<1, 128, 0, c->stream>>>(c->mail_d + off, (const unsigned char *)src_dev, (int)n);
  c->mail_pending.push_back({dst_host, off, n, c->mail_group});
  c->mail_used = off + n;
  return CCO_OK;
}
// close the current group: everything fetched so far is complete once the returned group's event has fired
static int mail_close(cco_ctx *c, int *group) {
  const int g = c->mail_group;
  while ((int)c->mail_ev.size() <= g) {
    cudaEvent_t e;
    CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    c->mail_ev.push_back(e);
  }
  CK(cudaEventRecord(c->mail_ev[g], c->stream));
  c->mail_group = g + 1;
  if (group) *group = g;
  return CCO_OK;
}
static int mail_wait_group(cco_ctx *c, int g) {
  CK(cudaEventSynchronize(c->mail_ev[g]));
  CK(cudaGetLastError());
  for (auto &m : c->mail_pending)
    if (m.group == g) memcpy(m.dst, c->mail_h + m.off, m.n);
  return CCO_OK;
}
static void mail_reset(cco_ctx *c) {
  c->mail_pending.clear();
  c->mail_used = 0;
  c->mail_group = 0;
}
// close + wait: the host needs the values now
static int mail_wait(cco_ctx *c) {
  int g = 0;
  CKR(mail_close(c, &g));
  return mail_wait_group(c, g);
}

struct DevRaw {  // a block of user rows of a matrix as uploaded (int64 row_ptr like the host)
  long long n_rows = 0;     // rows of the block (n_local)
  long long row_base = 0;   // global index of its first row
  int32_t n_cols = 0;
  long long nnz = 0;        // entries of the block
  long long nnz_cap = 0;    // entries of the whole matrix (upper bound for the sampled matrix)
  long long q_base = 0;     // value of rp[0] (host-known): a rank's block keeps the caller's absolute offsets
  long long *rp = nullptr;  // indexable by local row
  int32_t *col = nullptr;   // indexable by rp values
};
struct DevMat {  // after canonicalise + downsample
  long long n_rows = 0;
  int32_t n_cols = 0;
  uint32_t *rp = nullptr;  // [n_rows+1]
  int32_t *col = nullptr;
  int32_t *marg = nullptr;  // post-sample column counts
};

static int exclusive_sum_u32(cco_ctx *c, Arena &ar, const uint32_t *in, uint32_t *out, long long n) {
  size_t tb = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, n, c->stream));
  void *tmp;
  CKR(ar.alloc((char **)&tmp, tb));
  CK(cub::DeviceScan::ExclusiveSum(tmp, tb, in, out, n, c->stream));
  ar.release(tmp);
  return CCO_OK;
}
static int exclusive_sum_i64(cco_ctx *c, Arena &ar, const long long *in, long long *out, long long n, cudaStream_t on = nullptr) {
  if (!on) on = c->stream;
  size_t tb = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, n, on));
  void *tmp;
  CKR(ar.alloc((char **)&tmp, tb));   // a few KB: always slab memory when the arena has slabs
  CK(cub::DeviceScan::ExclusiveSum(tmp, tb, in, out, n, on));
  ar.release(tmp);
  return CCO_OK;
}

// canonicalisation slow path: sort (row,col) keys, drop duplicates, rebuild row_ptr
static int canonicalize_device(cco_ctx *c, Arena &ar, DevRaw &m) {
  if (m.nnz == 0) return CCO_OK;
  unsigned long long *k0, *k1;
  CKR(ar.alloc(&k0, m.nnz));
  CKR(ar.alloc(&k1, m.nnz));
  k_expand_keys<<<grid_for(m.n_rows * kSG, 256, c->sm_count), 256, 0, c->stream>>>(m.n_rows, m.rp, m.col, k0);
  c->launches++;
  int row_bits = 1;
  while ((1LL << row_bits) < m.n_rows) ++row_bits;
  cub::DoubleBuffer<unsigned long long> db(k0, k1);
  size_t tb = 0;
  CK(cub::DeviceRadixSort::SortKeys(nullptr, tb, db, m.nnz, 0, 32 + row_bits, c->stream));
  void *tmp;
  CKR(ar.alloc((char **)&tmp, tb));
  CK(cub::DeviceRadixSort::SortKeys(tmp, tb, db, m.nnz, 0, 32 + row_bits, c->stream));
  ar.release(tmp);
  unsigned long long *sorted = db.Current(), *other = db.Alternate();
  uint32_t *flag, *pos;
  CKR(ar.alloc(&flag, m.nnz + 1));
  CKR(ar.alloc(&pos, m.nnz + 1));
  CK(cudaMemsetAsync(flag + m.nnz, 0, 4, c->stream));
  k_unique_flags<<<grid_for(m.nnz, 256, c->sm_count), 256, 0, c->stream>>>(m.nnz, sorted, flag);
  c->launches++;
  CKR(exclusive_sum_u32(c, ar, flag, pos, m.nnz + 1));
  uint32_t n_unique = 0;
  CK(cudaMemcpyAsync(&n_unique, pos + m.nnz, 4, cudaMemcpyDeviceToHost, c->stream));
  // the canonical block is rewritten 0-based at the start of its own column storage
  k_unique_scatter<<<grid_for(m.nnz, 256, c->sm_count), 256, 0, c->stream>>>(m.nnz, sorted, flag, pos, other, m.col + m.q_base);
  CK(cudaStreamSynchronize(c->stream));
  k_rowptr_from_keys<<<grid_for(m.n_rows + 1, 256, c->sm_count), 256, 0, c->stream>>>(m.n_rows, n_unique, other, m.rp);
  c->launches += 2;
  m.col += m.q_base;
  m.q_base = 0;
  m.nnz = n_unique;
  CK(cudaGetLastError());
  ar.release(flag);
  ar.release(pos);
  ar.release(k0);
  ar.release(k1);
  return CCO_OK;
}

// rows with more than kHeavyRow entries of a block, listed once per train and matrix (k_list_heavy_rows)
struct HeavyRows {
  int32_t *list = nullptr;
  int *n = nullptr;
};
static int list_heavy_rows(cco_ctx *c, Arena &ar, const DevRaw &raw, HeavyRows *h) {
  CKR(ar.alloc(&h->list, std::max<long long>(raw.n_rows, 1)));
  CKR(ar.alloc(&h->n, 1));
  CK(cudaMemsetAsync(h->n, 0, 4, c->stream));
  if (raw.n_rows > 0) {
    k_list_heavy_rows<<<grid_for(raw.n_rows, 256, c->sm_count), 256, 0, c->stream>>>(raw.n_rows, raw.rp, h->list, h->n);
    c->launches++;
  }
  return CCO_OK;
}
// a row-parallel pass = one launch over the light rows (kSG lanes per row) + one over the listed heavy rows (a warp per
// row; a fixed few waves of CTAs loop over the list, whose length they read on the device)
static void launch_check(cco_ctx *c, const DevRaw &raw, const HeavyRows &h, int *flags) {
  if (raw.n_rows <= 0) return;
  const long long q_lo = raw.q_base, q_hi = raw.q_base + raw.nnz;
  k_check_rows<kSG><<<grid_for(raw.n_rows * kSG, 256, c->sm_count), 256, 0, c->stream>>>(raw.n_rows, raw.n_cols, raw.rp, raw.col, q_lo, q_hi,
                                                                                       nullptr, nullptr, flags);
  k_check_rows<32><<<c->sm_count * 4, 256, 0, c->stream>>>(raw.n_rows, raw.n_cols, raw.rp, raw.col, q_lo, q_hi, h.list, h.n, flags);
  c->launches += 2;
}
// per-matrix scratch of the two sampling passes: integer keep thresholds per column, one keep byte per stored entry
struct SampleScratch {
  unsigned long long *col_thr = nullptr;
  uint8_t *keep = nullptr;
};
static int sample_scratch(cco_ctx *c, Arena &ar, const DevRaw &raw, const int32_t *raw_counts, int32_t m, SampleScratch *sc) {
  CKR(ar.alloc(&sc->col_thr, std::max<int32_t>(raw.n_cols, 1)));
  CKR(ar.alloc(&sc->keep, std::max<long long>(raw.nnz, 1)));
  if (raw.n_cols > 0) {
    k_col_thresholds<<<grid_for(raw.n_cols, 256, c->sm_count, 4), 256, 0, c->stream>>>(raw.n_cols, raw_counts, m, sc->col_thr);
    c->launches++;
  }
  return CCO_OK;
}
// pass 1 (k_sample_count, cco_sampler.cuh): entry-parallel; `kept` must be zero for the block's rows; `bad` (nullable) is the
// device verdict of k_check_row_ptr / k_col_histogram_flat -- a malformed matrix keeps nothing, so pass 2 can never write more than row_ptr promises
static void launch_count(cco_ctx *c, const DevRaw &raw, const SampleScratch &sc, int32_t m, int32_t seed, uint32_t flags, const int *bad,
                         uint32_t *kept, int32_t *new_counts) {
  if (raw.n_rows <= 0 || raw.nnz <= 0) return;
  const long long q_lo = raw.q_base, q_hi = raw.q_base + raw.nnz;
  const long long n_chunks = (raw.nnz + kSampleChunk - 1) / kSampleChunk;
  k_sample_count<<<grid_for(n_chunks * 32, 256, c->sm_count), 256, 0, c->stream>>>(raw.n_rows, raw.row_base, raw.rp, raw.col, raw.n_cols, q_lo, q_hi,
                                                                                  sc.col_thr, m, seed, flags, bad, kept, new_counts, sc.keep);
  c->launches++;
}
// pass 2: order-preserving compaction of the block's column indices by the keep bytes.  Kept entries keep their global
// order, so entry ranks inside the block are offsets from the block's first kept entry: `dst` is where that one goes.
static int launch_write(cco_ctx *c, Arena &ar, const DevRaw &raw, const SampleScratch &sc, int32_t *dst) {
  if (raw.n_rows <= 0 || raw.nnz <= 0) return CCO_OK;
  long long *n_sel;
  CKR(ar.alloc(&n_sel, 1));
  size_t tb = 0;
  CK(cub::DeviceSelect::Flagged(nullptr, tb, raw.col + raw.q_base, sc.keep, dst, n_sel, (long long)raw.nnz, c->stream));
  void *tmp;
  CKR(ar.alloc((char **)&tmp, tb));
  CK(cub::DeviceSelect::Flagged(tmp, tb, raw.col + raw.q_base, sc.keep, dst, n_sel, (long long)raw.nnz, c->stream));
  ar.release(tmp);
  c->launches += 2;   // init + select kernel
  return CCO_OK;
}

// sampleDownAndBinarize of one whole matrix on this GPU (raw column counts already final in raw_counts)
static int downsample_device(cco_ctx *c, Arena &ar, const DevRaw &raw, const int *bad, const int32_t *raw_counts, int32_t m,
                             int32_t seed, uint32_t flags, DevMat *out) {
  out->n_rows = raw.n_rows;
  out->n_cols = raw.n_cols;
  uint32_t *kept;
  CKR(ar.alloc(&kept, raw.n_rows + 1));
  CKR(ar.alloc(&out->rp, raw.n_rows + 1));
  if (!out->marg) CKR(ar.alloc(&out->marg, std::max<int32_t>(raw.n_cols, 1)));
  CKR(ar.alloc(&out->col, std::max<long long>(raw.nnz, 1)));
  CK(cudaMemsetAsync(out->marg, 0, sizeof(int32_t) * std::max<int32_t>(raw.n_cols, 1), c->stream));
  CK(cudaMemsetAsync(kept, 0, sizeof(uint32_t) * ((size_t)raw.n_rows + 1), c->stream));
  SampleScratch sc;
  CKR(sample_scratch(c, ar, raw, raw_counts, m, &sc));
  launch_count(c, raw, sc, m, seed, flags, bad, kept, out->marg);
  CKR(exclusive_sum_u32(c, ar, kept, out->rp, raw.n_rows + 1));
  CKR(launch_write(c, ar, raw, sc, out->col));
  CK(cudaGetLastError());
  ar.release(kept);
  ar.release(sc.col_thr);
  ar.release(sc.keep);
  return CCO_OK;
}

static int nccl_check(int rc, const char *what) {
  if (rc != 0) return set_error(CCO_E_NCCL, "%s: %s", what, g_nccl.GetErrorString(rc));
  return CCO_OK;
}

// Multi-GPU form of sampleDownAndBinarize.  Rank r holds (and samples) only its block of users.  Four collectives over
// NVLink per train:
//   (1) [caller] all-reduce of the raw column counts            -> the sampling rates
//   (2) all-gather of the per-user kept counts (all matrices)   -> every rank scans the identical row_ptr
//   (3) all-reduce of the post-sample column counts             -> marginals (nothing is re-counted on the gathered matrix)
//   (4) all-gather of the sampled column blocks, each padded to the largest sampled block (the block sizes come from the
//       scanned row_ptr through one mailbox record: an event wait, not a stream sync), then a pack kernel.
static int downsample_sharded_all(cco_ctx *c, Arena &ar, const std::vector<DevRaw> &raw, const int *d_check /* [2 * n_mats] */,
                                  const std::vector<long long> &block_cap,
                                  long long U, const int32_t *raw_counts, int32_t *marg_all, const std::vector<long long> &col_off,
                                  const cco_indicator_params_t *params, int32_t seed, uint32_t flags, std::vector<DevMat> &dm,
                                  cudaEvent_t *stage_ev /* [4]: after pass 1, after collectives + scans, after pass 2, after gather + pack */) {
  cudaStream_t s = c->stream;
  const int W = c->world, r = c->rank, n_mats = (int)raw.size();
  const long long S = (U + W - 1) / W;
  const long long row_base = raw[0].row_base;
  std::vector<uint32_t *> kept(n_mats, nullptr);
  std::vector<SampleScratch> sc(n_mats);
  for (int i = 0; i < n_mats; ++i) {
    DevMat *out = &dm[i];
    out->n_rows = U;
    out->n_cols = raw[i].n_cols;
    out->marg = marg_all + col_off[i];
    CKR(ar.alloc(&kept[i], (size_t)(W * S + 1)));
    CKR(ar.alloc(&out->rp, U + 1));
    CK(cudaMemsetAsync(kept[i], 0, sizeof(uint32_t) * (size_t)(W * S + 1), s));
    CKR(sample_scratch(c, ar, raw[i], raw_counts + col_off[i], params[i].max_interactions, &sc[i]));
    launch_count(c, raw[i], sc[i], params[i].max_interactions, seed, flags, d_check + 2 * i, kept[i], out->marg);
  }
  CK(cudaEventRecord(stage_ev[0], s));
  if (S > 0) {
    g_nccl.GroupStart();
    for (int i = 0; i < n_mats; ++i) {
      int rc = g_nccl.AllGather(kept[i] + (size_t)r * S, kept[i], (size_t)S, kNcclUint32, c->comm, s);
      if (rc != 0) { g_nccl.GroupEnd(); return nccl_check(rc, "ncclAllGather(kept counts)"); }
    }
    CKR(nccl_check(g_nccl.GroupEnd(), "ncclGroupEnd(kept counts)"));
  }
  if (col_off[n_mats] > 0)
    CKR(nccl_check(g_nccl.AllReduce(marg_all, marg_all, (size_t)col_off[n_mats], kNcclInt32, kNcclSum, c->comm, s), "ncclAllReduce(marginals)"));
  std::vector<int32_t *> gathered(n_mats, nullptr);
  // NCCL's all-gather moves equal counts per rank.  The raw block size (host-known) would do as the padding, but after
  // downsampling a block is 2-3x smaller than its raw size at the 10M-user shapes (C4: 1.8 GB received per GPU, 4.7 ms).
  // The sampled block sizes sit in row_ptr on the device: one mailbox record per train brings them to the host (one event
  // wait, no stream-wide sync) and the gather is padded to the largest SAMPLED block only.
  std::vector<uint32_t> edge((size_t)n_mats * (W + 1), 0);
  for (int i = 0; i < n_mats; ++i) {
    CKR(exclusive_sum_u32(c, ar, kept[i], dm[i].rp, U + 1));
    ar.release(kept[i]);
    for (int q = 0; q <= W; ++q) CKR(mail_fetch(c, &edge[(size_t)i * (W + 1) + q], dm[i].rp + std::min<long long>((long long)q * S, U), 4));
  }
  CK(cudaEventRecord(stage_ev[1], s));
  CKR(mail_wait(c));
  std::vector<long long> cap(n_mats, 0);
  for (int i = 0; i < n_mats; ++i) {
    for (int q = 0; q < W; ++q) cap[i] = std::max<long long>(cap[i], (long long)edge[(size_t)i * (W + 1) + q + 1] - edge[(size_t)i * (W + 1) + q]);
    CKR(ar.alloc(&dm[i].col, std::max<long long>(edge[(size_t)i * (W + 1) + W], 1)));
    if (cap[i] == 0) continue;
    CKR(ar.alloc(&gathered[i], (size_t)(cap[i] * W)));
    // this rank's block goes straight into its slot of the gather buffer, relative to the block's first entry
    CKR(launch_write(c, ar, raw[i], sc[i], gathered[i] + (size_t)r * cap[i]));
    ar.release(sc[i].col_thr);
    ar.release(sc[i].keep);
  }
  CK(cudaEventRecord(stage_ev[2], s));
  g_nccl.GroupStart();
  for (int i = 0; i < n_mats; ++i) {
    if (!gathered[i]) continue;
    int rc = g_nccl.AllGather(gathered[i] + (size_t)r * cap[i], gathered[i], (size_t)cap[i], kNcclInt32, c->comm, s);
    if (rc != 0) { g_nccl.GroupEnd(); return nccl_check(rc, "ncclAllGather(column blocks)"); }
  }
  CKR(nccl_check(g_nccl.GroupEnd(), "ncclGroupEnd(column blocks)"));
  for (int i = 0; i < n_mats; ++i) {
    if (!gathered[i]) continue;
    dim3 grid((unsigned)std::max(1, std::min(c->sm_count * 8 / W, 1024)), (unsigned)W);
    k_pack_blocks<<<grid, 256, 0, s>>>(W, S, U, cap[i], dm[i].rp, gathered[i], dm[i].col);
    c->launches++;
    ar.release(gathered[i]);
  }
  CK(cudaEventRecord(stage_ev[3], s));
  CK(cudaGetLastError());
  return CCO_OK;
}

// ---- row-kernel configurations -----------------------------------------------------------------

struct BinCfg {
  int group;    // threads that own one row: 32 (warp), 256 or 1024 (whole CTA)
  int slots;    // table words per group
  int cap;      // distinct keys a hashed table may hold per pass
  int cbuf;     // candidate buffer entries per group
  int caux, keep_max, final_max;
  bool dense;
  size_t region;  // shared-memory bytes per group
  size_t smem;    // per CTA
  int ctas_per_sm;
};

static int next_pow2(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

template <int GROUP>
static int launch_rows_t(cco_ctx *c, const RowArgs &a, BinCfg &cfg, cudaStream_t st) {
  constexpr int CTA = GROUP == 32 ? 64 : GROUP;   // warp-owned rows: two independent warps per CTA (fine-grained smem packing)
  int occ = 1;
  void (*kern)(const RowArgs) = cfg.dense ? k_rows<GROUP, true> : k_rows<GROUP, false>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg.smem));
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, CTA, cfg.smem));
  // 4 waves of CTAs over the work-sorted row list: a CTA that draws cheap rows retires early and the hardware
  // scheduler backfills, which balances the tail better than one persistent wave (round-1 launch sweep: -6 % at C3)
  kern<<<c->sm_count * std::max(occ, 1) * 4, CTA, cfg.smem, st>>>(a);
  cfg.ctas_per_sm = occ;
  c->launches++;
  CK(cudaGetLastError());
  return CCO_OK;
}
static int launch_rows(cco_ctx *c, const RowArgs &a, BinCfg &cfg, cudaStream_t st) {
  switch (cfg.group) {
    case 1024: return launch_rows_t<1024>(c, a, cfg, st);
    case 512: return launch_rows_t<512>(c, a, cfg, st);
    case 256: return launch_rows_t<256>(c, a, cfg, st);
    case 128: return launch_rows_t<128>(c, a, cfg, st);
    case 32: return launch_rows_t<32>(c, a, cfg, st);
  }
  return set_error(CCO_E_INVALID_ARG, "internal: bad bin config");
}

// Candidate-buffer invariant of k_rows (checked by cfg_ok before any launch):
//   top_k <= keep_max <= cbuf - group   and   final_max <= cbuf,   caux >= max(keep_max, final_max) for CTA groups.
// A round appends at most `group` candidates to a buffer that holds at most prune_limit = cbuf - group of them (no
// prune) or keep_max (after a prune), so it never writes past cbuf; the CTA-path select compacts up to keep_max (or
// final_max) survivors into aux.  keep_max is capped at cbuf - group: without the cap, final_max = next_pow2(top_k)
// exceeds the prune limit in some CTA configurations (group 128: top_k 257-384, 513-896, 1025-1920; group 256: 513-768,
// 1025-1792; group 512: 1025-1536; e.g. top_k 300, group 128: cbuf 512, limit 384, keep_max 512), a prune may stop
// with nearly every candidate kept, and the next round overflows tk into aux.  The cap changes keep_max in those
// configurations only; caux (max(keep_max, final_max)), hence the shared-memory layout, is the same as before everywhere.
static BinCfg make_cfg(cco_ctx *c, int group, int want_slots, int top_k, int n_cols_b) {
  BinCfg f;
  const int groups = group == 32 ? 2 : 1;
  f.group = group;
  f.final_max = next_pow2(top_k);
  f.cbuf = next_pow2(top_k + std::max(group, 128) + (group == 32 ? 64 : 0));
  if (group == 32 && top_k + 32 <= 96) f.cbuf = 128;  // small top_k: a 128-entry buffer doubles the warps per SM (-4 % at C3)
  f.keep_max = std::min(std::max(f.final_max, (f.cbuf - group) / 2), f.cbuf - group);
  f.caux = group == 32 ? 0 : std::max(f.keep_max, f.final_max);
  // candidates, x12/x11 tables, ctrl, radix-select histogram (aliased by the level-1 cut bins), queues
  size_t fixed = (size_t)(f.cbuf + f.caux) * 16 + 2 * 256 + 512 + 1024 + (size_t)(group / 32) * 256;
  size_t avail = (c->smem_optin - 1024) / groups;  // slack for static shared memory
  int max_slots = (int)((avail - fixed) / 4) & ~1023;
  f.slots = std::min(want_slots, max_slots);
  f.cap = f.slots / 2;  // load factor <= 1/2: 2/3 and 3/4 are 8 % and 17 % slower (probe chains), round-1 launch sweep
  f.dense = n_cols_b <= f.slots;
  f.region = (fixed + (size_t)f.slots * 4 + 15) & ~(size_t)15;
  f.smem = f.region * groups;
  f.ctas_per_sm = 1;
  return f;
}

static bool cfg_ok(const BinCfg &f, int top_k, size_t smem_optin) {
  return top_k <= f.keep_max && f.keep_max <= f.cbuf - f.group && f.final_max <= f.cbuf &&
         (f.group == 32 || f.caux >= std::max(f.keep_max, f.final_max)) && f.slots > 0 && f.smem <= smem_optin;
}

// ---- one indicator = rows [lo, hi) of A'^T B' on this rank ---------------------------------------------------------------
// enqueue_indicator puts everything of one indicator on the stream without a single host round trip (the rank partition,
// the bin bounds and the packed sizes stay on the device); finish_indicator waits for that indicator's mailbox record
// only -- while the GPU already runs the next indicator -- and starts the device->host copy of its packed arrays.
struct IndicatorState {
  int mail_group = -1;
  long long rec[7] = {0, 0, 0, 0, 0, 0, 0};   // k_indicator_record
  cudaEvent_t packed = nullptr;                // compaction done (the copy stream waits for it)
  long long *out_ptr = nullptr;                // [n_items_a + 1], 0 outside the rank's rows
  int32_t *p_col = nullptr, *p_cnt = nullptr;
  double *p_llr = nullptr;
  int32_t n_items_a = 0, n_cols_b = 0;
  bool emit_all = false;
};

static int enqueue_indicator(cco_ctx *c, Arena &ar, const uint32_t *at_ptr, const int32_t *at_users, int32_t n_items_a,
                             const int32_t *marg_a, int32_t max_marg_a, int32_t max_marg_b, const DevMat &B, long long n_users,
                             bool self, const cco_indicator_params_t &prm, uint32_t flags, bool emit_all, cudaEvent_t inputs_ready,
                             cudaEvent_t ev_begin, cudaEvent_t ev_end, IndicatorState *st) {
  cudaStream_t s = c->stream;
  const int32_t n_cols_b = B.n_cols;
  const int rank = c->rank, world = c->world;
  st->n_items_a = n_items_a;
  st->n_cols_b = n_cols_b;
  st->emit_all = emit_all;
  // 1. work per output row, rank partition, schedule --------------------------------------------------
  // The schedule reads only the prepared matrices, so it does not have to queue behind the previous indicator's row
  // kernels: with `inputs_ready` (recorded on s once the preparation is complete) it runs on the scheduling stream and s
  // joins it before the bins launch.  Everything it touches must then be slab memory (no stream-ordered allocation on s).
  uint32_t *row_work, *masked, *sorted_work;
  unsigned long long *work64;
  long long *work_prefix;
  int32_t *ids, *rows_sorted, *d_pb = nullptr;
  size_t sort_tb = 0;
  if (n_items_a > 0)
    CK(cub::DeviceRadixSort::SortPairsDescending(nullptr, sort_tb, (const uint32_t *)nullptr, (uint32_t *)nullptr, (const int32_t *)nullptr,
                                                 (int32_t *)nullptr, n_items_a, 0, 32, s));
  const bool beside = inputs_ready && ar.c && ((size_t)n_items_a + 1) * 8 <= Arena::kSlabMax && sort_tb <= Arena::kSlabMax;
  cudaStream_t ss = beside ? c->sched_stream : s;
  if (beside) CK(cudaStreamWaitEvent(ss, inputs_ready, 0));
  CKR(ar.alloc(&row_work, n_items_a + 1));
  CKR(ar.alloc(&masked, n_items_a + 1));
  CKR(ar.alloc(&work64, n_items_a + 1));
  CKR(ar.alloc(&work_prefix, n_items_a + 1));
  CKR(ar.alloc(&ids, n_items_a + 1));
  CKR(ar.alloc(&sorted_work, n_items_a + 1));
  CKR(ar.alloc(&rows_sorted, n_items_a + 1));
  CK(cudaMemsetAsync(work64 + n_items_a, 0, 8, ss));
  k_row_work<<<grid_for((long long)n_items_a * kSG, 256, c->sm_count), 256, 0, ss>>>(n_items_a, at_ptr, at_users, B.rp,
                                                                                  row_work, work64, ids, nullptr);
  c->launches++;
  CKR(exclusive_sum_i64(c, ar, (const long long *)work64, work_prefix, (long long)n_items_a + 1, ss));
  if (world > 1) {
    // contiguous item ranges balanced by work prefix, identical on every rank; they never leave the device
    CKR(ar.alloc(&d_pb, world + 1));
    k_partition_rows<<<1, ((world + 1 + 31) / 32) * 32, 0, ss>>>(work_prefix, n_items_a, world, d_pb);
    c->launches++;
  }
  k_mask_work<<<grid_for(n_items_a, 256, c->sm_count), 256, 0, ss>>>(n_items_a, row_work, d_pb, rank, masked);
  c->launches++;
  if (n_items_a > 0) {
    void *tmp;
    CKR(ar.alloc((char **)&tmp, sort_tb));
    CK(cub::DeviceRadixSort::SortPairsDescending(tmp, sort_tb, masked, sorted_work, ids, rows_sorted, n_items_a, 0, 32, ss));
    ar.release(tmp);
  }
  // 2. bins -----------------------------------------------------------------------------------------
  const int k_eff = emit_all ? 1 : prm.top_k;
  const bool warp_ok = k_eff + 32 <= 256;  // warp-owned rows keep a 256-entry candidate buffer
  // Work bins, largest rows first.  {threads that own a row, table words, largest row work w the bin takes}.
  // Bin 0 is the multi-pass bin (same config as bin 1).  Rows up to 1024 products are WARP-owned: no CTA barrier
  // anywhere in their count / compact / score / select pipeline; larger rows need the table and the parallelism of a CTA.
  struct BinSpec { int group, slots; uint32_t max_w; };
  std::vector<BinSpec> spec = {{1024, 1 << 20, 0xffffffffu}, {1024, 1 << 20, 0xffffffffu}, {512, 16384, 8192u}, {256, 8192, 4096u}};
  if (warp_ok) {
    // rows of 1025..2048 products: a 128-thread CTA shares one 4096-word table -- a warp-owned 4096-word table leaves
    // too few warps per SM (round-1 launch sweep: -4 % at C3); up to 1024 products rows are warp-owned
    spec.push_back({128, 4096, 2048u});
    spec.push_back({32, 2048, 1024u});
    spec.push_back({32, 1024, 512u});
    spec.push_back({32, 512, 256u});
  } else {
    spec.push_back({128, 4096, 2048u});
  }
  const int kBins = (int)spec.size();
  std::vector<BinCfg> cfgs(kBins);
  for (int b = 0; b < kBins; ++b) {
    cfgs[b] = make_cfg(c, spec[b].group, spec[b].slots, k_eff, n_cols_b);
    if (!cfg_ok(cfgs[b], k_eff, c->smem_optin))
      return set_error(CCO_E_INVALID_ARG, "internal: row-kernel bin %d (group %d, top_k %d) violates the candidate-buffer "
                       "invariant: cbuf %d, keep_max %d, final_max %d, caux %d", b, spec[b].group, k_eff, cfgs[b].cbuf,
                       cfgs[b].keep_max, cfgs[b].final_max, cfgs[b].caux);
  }
  BinCfg &cfgL = cfgs[1];
  // packed word: key bits must leave room for the largest possible count
  int key_bits = 1;
  while (((1LL << key_bits) - 1) <= (long long)n_cols_b) ++key_bits;  // keys <= 2^kb - 2
  int count_bits = 32 - key_bits;
  // a co-occurrence count is bounded by both marginals: k11 <= min(rowA, colB) <= min(max rowA, max colB).  With the
  // reference's default downsampling (m = 500) that is ~560, i.e. 10 count bits next to 22 key bits (4M columns).
  const long long k11_max = std::min<long long>(max_marg_a, max_marg_b);
  if (count_bits < 1 || k11_max >= (1LL << count_bits))
    return set_error(CCO_E_UNSUPPORTED,
                     "co-occurrence counts up to %lld over %d columns do not fit the packed 32-bit accumulator word "
                     "(key %d bits + count %d bits): lower maxItemsPerUser/maxEventsPerEventType for this event type "
                     "(\"Limits\" in include/cco_b200.h)", k11_max, n_cols_b, key_bits, count_bits);
  // thresholds on w, descending: bin b takes rows with h_thr[b-1] >= w > h_thr[b]; a hashed table also needs w <= cap
  std::vector<uint32_t> h_thr(kBins);
  for (int b = 0; b < kBins; ++b) {
    const BinCfg &f = cfgs[std::min(b + 1, kBins - 1)];   // h_thr[b] = upper limit of bin b+1
    uint32_t lim = b + 1 < kBins ? spec[b + 1].max_w : 0u;
    if (b + 1 < kBins && !f.dense) lim = std::min<uint32_t>(lim, (uint32_t)f.cap);
    h_thr[b] = lim;
    if (b > 0) h_thr[b] = std::min(h_thr[b], h_thr[b - 1]);
  }
  int32_t *d_bounds;
  CKR(ar.alloc(&d_bounds, kBins + 3));
  BinThresholds bt;
  memset(&bt, 0, sizeof bt);
  for (int b = 0; b < kBins; ++b) bt.t[b] = h_thr[b];
  k_bin_bounds<<<1, 32, 0, ss>>>(n_items_a, sorted_work, kBins, bt, d_bounds);
  c->launches++;
  if (beside) {
    cudaEvent_t scheduled;
    CKR(pooled_event(c, false, &scheduled));
    CK(cudaEventRecord(scheduled, ss));
    CK(cudaStreamWaitEvent(s, scheduled, 0));
  }
  // per-column constants of B' for the fused LLR
  ColTerm *col_terms;
  CKR(ar.alloc(&col_terms, std::max<int32_t>(n_cols_b, 1)));
  if (n_cols_b > 0) {
    k_col_terms<<<grid_for(n_cols_b, 256, c->sm_count, 4), 256, 0, s>>>(n_cols_b, B.marg, n_users, flags, col_terms);
    c->launches++;
  }
  // 3. outputs ----------------------------------------------------------------------------------------
  int32_t stride = emit_all ? n_cols_b : std::min<int32_t>(prm.top_k, n_cols_b);
  if (stride < 1) stride = 1;
  int32_t *o_col, *o_cnt, *o_len;
  double *o_llr = nullptr;
  unsigned long long *d_distinct;
  int *d_err;
  size_t cells = (size_t)std::max(n_items_a, 1) * stride;
  CKR(ar.alloc(&o_col, cells));
  CKR(ar.alloc(&o_cnt, cells));
  if (!emit_all) CKR(ar.alloc(&o_llr, cells));
  CKR(ar.alloc(&o_len, n_items_a + 1));
  CKR(ar.alloc(&d_distinct, 2));
  CKR(ar.alloc(&d_err, 1));
  CK(cudaMemsetAsync(o_len, 0, sizeof(int32_t) * ((size_t)n_items_a + 1), s));
  CK(cudaMemsetAsync(d_distinct, 0, 16, s));
  CK(cudaMemsetAsync(d_err, 0, 4, s));
  RowArgs a;
  memset(&a, 0, sizeof a);
  a.at_ptr = at_ptr;
  a.at_users = at_users;
  a.b_ptr = B.rp;
  a.b_col = B.col;
  a.marg_a = marg_a;
  a.marg_b = B.marg;
  a.max_marg_b = max_marg_b;
  a.col_terms = col_terms;
  a.rows_sorted = rows_sorted;
  a.row_work = row_work;
  a.bin_bounds = d_bounds;
  a.n_cols_b = n_cols_b;
  a.n_users = n_users;
  a.self = self ? 1 : 0;
  a.top_k = k_eff;
  a.has_min_llr = prm.has_min_llr;
  a.min_llr = prm.min_llr;
  a.flags = flags;
  a.count_bits = count_bits;
  a.out_stride = stride;
  a.out_col = o_col;
  a.out_llr = o_llr;
  a.out_cnt = o_cnt;
  a.out_len = o_len;
  a.stat_distinct = d_distinct;
  a.stat_evaluated = d_distinct + 1;
  a.err_flag = d_err;
  a.emit_all = emit_all ? 1 : 0;
  if (ev_begin) CK(cudaEventRecord(ev_begin, s));
  if (n_items_a > 0) {
    // the bins touch disjoint rows: run them concurrently (tails of one bin overlap the bulk of another)
    CK(cudaEventRecord(c->bin_ev[8], s));
    for (int b = 0; b < kBins; ++b) {
      if (b == 0 && cfgL.dense) continue;                 // dense L takes every large row in bin 1
      RowArgs ab = a;
      ab.bin = b;
      ab.slots = cfgs[b].slots;
      ab.cap = cfgs[b].cap;
      ab.tsize_x16 = 32;
      ab.cbuf = cfgs[b].cbuf;
      ab.caux = cfgs[b].caux;
      ab.keep_max = cfgs[b].keep_max;
      ab.final_max = cfgs[b].final_max;
      ab.group_smem_bytes = (int32_t)cfgs[b].region;
      CK(cudaStreamWaitEvent(c->bin_stream[b], c->bin_ev[8], 0));
      CKR(launch_rows(c, ab, cfgs[b], c->bin_stream[b]));
      CK(cudaEventRecord(c->bin_ev[b], c->bin_stream[b]));
      CK(cudaStreamWaitEvent(s, c->bin_ev[b], 0));
    }
  }
  if (ev_end) CK(cudaEventRecord(ev_end, s));
  // 4. pack ---------------------------------------------------------------------------------------------
  long long *len64, *rec_d;
  CKR(ar.alloc(&len64, n_items_a + 1));
  CKR(ar.alloc(&st->out_ptr, n_items_a + 1));
  CKR(ar.alloc(&rec_d, 8));
  k_len_to_i64<<<grid_for((long long)n_items_a + 1, 256, c->sm_count), 256, 0, s>>>(n_items_a, o_len, d_pb, rank, len64);
  c->launches++;
  CKR(exclusive_sum_i64(c, ar, len64, st->out_ptr, (long long)n_items_a + 1));
  // the packed size is only known on the device: the buffers take the worst case (every row of the item space full)
  CKR(ar.alloc(&st->p_col, cells));
  if (!(flags & CCO_FLAG_RESULT_NO_COUNT) || emit_all) CKR(ar.alloc(&st->p_cnt, cells));
  if (!emit_all && !(flags & CCO_FLAG_RESULT_NO_LLR)) CKR(ar.alloc(&st->p_llr, cells));
  if (n_items_a > 0) {
    k_compact_rows<<<grid_for((long long)n_items_a * 32, 256, c->sm_count), 256, 0, s>>>(n_items_a, stride, st->out_ptr, o_col, o_llr,
                                                                                      o_cnt, st->p_col, st->p_llr, st->p_cnt);
    c->launches++;
  }
  k_indicator_record<<<1, 32, 0, s>>>(n_items_a, d_pb, rank, st->out_ptr, work_prefix, d_distinct, d_err, rec_d);
  c->launches++;
  CKR(mail_fetch(c, st->rec, rec_d, sizeof(long long) * 7));
  CKR(mail_close(c, &st->mail_group));
  if (!st->packed) CK(cudaEventCreateWithFlags(&st->packed, cudaEventDisableTiming));
  CK(cudaEventRecord(st->packed, s));
  CK(cudaGetLastError());
  // the strided buffers are dead once k_compact_rows has been enqueued (stream order)
  for (void *p : {(void *)o_col, (void *)o_cnt, (void *)o_llr, (void *)len64})
    if (p) ar.release(p);
  return CCO_OK;
}

struct IndicatorOut {
  int64_t row_begin = 0, row_end = 0;
  int64_t nnz = 0;
  int64_t products = 0, distinct = 0, evaluated = 0;
};

// wait for the indicator's record, allocate its host arrays, start the device->host copies on the copy stream
static int finish_indicator(cco_ctx *c, IndicatorState *st, uint32_t flags, int index, ResultMat *rm, IndicatorOut *io) {
  CKR(mail_wait_group(c, st->mail_group));
  const int32_t lo = (int32_t)st->rec[0], hi = (int32_t)st->rec[1];
  const long long total = st->rec[2];
  io->row_begin = lo;
  io->row_end = hi;
  io->nnz = total;
  io->products = st->rec[3];
  io->distinct = st->rec[4];
  io->evaluated = st->rec[5];
  if (st->rec[6]) return set_error(CCO_E_CUDA, "internal: shared-memory hash table overflow");
  const int32_t n_my = hi - lo;
  cudaStream_t cs = c->copy_stream;
  CK(cudaStreamWaitEvent(cs, st->packed, 0));
  GroupShared *gs = c->gshared;
  int64_t *h_rp;
  int32_t *h_col, *h_cnt = nullptr;
  double *h_llr = nullptr;
  long long base = 0;
  if (gs) {
    // group mode: every rank's slice lands in ONE set of host arrays (rank 0 of the group allocates them once all
    // ranks know their sizes); row pointers are rebased on the device by the cells of the ranks before this one
    {
      std::lock_guard<std::mutex> lk(gs->mu);
      gs->totals[c->rank] = total;
    }
    gs->barrier();
    long long grand = 0;
    for (int q = 0; q < gs->world; ++q) {
      if (q < c->rank) base += gs->totals[q];
      grand += gs->totals[q];
    }
    ResultMat &mm = gs->merged->mats[index];
    if (c->rank == 0) {
      cco_ctx *owner = gs->merged->ctx;
      mm.row_begin = 0;
      mm.row_end = st->n_items_a;
      mm.n_cols = st->n_cols_b;
      mm.row_ptr = (int64_t *)owner->pinned_get(sizeof(int64_t) * ((size_t)st->n_items_a + 1));
      mm.col = (int32_t *)owner->pinned_get(sizeof(int32_t) * (size_t)std::max<long long>(grand, 1));
      if (st->p_cnt) mm.cnt = (int32_t *)owner->pinned_get(sizeof(int32_t) * (size_t)std::max<long long>(grand, 1));
      if (st->p_llr) mm.llr = (double *)owner->pinned_get(sizeof(double) * (size_t)std::max<long long>(grand, 1));
    }
    gs->barrier();
    if (!mm.row_ptr || !mm.col || (st->p_cnt && !mm.cnt) || (st->p_llr && !mm.llr)) return set_error(CCO_E_OOM, "pinned host allocation failed");
    h_rp = mm.row_ptr + lo;
    h_col = mm.col + base;
    h_cnt = mm.cnt ? mm.cnt + base : nullptr;
    h_llr = mm.llr ? mm.llr + base : nullptr;
    if (base != 0 && n_my >= 0) {
      k_add_i64<<<grid_for((long long)n_my + 1, 256, c->sm_count, 2), 256, 0, cs>>>((long long)n_my + 1, base, st->out_ptr + lo);
      c->launches++;
    }
    rm->row_begin = lo;   // the member's own record (stats only; the arrays belong to the merged result)
    rm->row_end = hi;
    rm->n_cols = st->n_cols_b;
  } else {
    rm->row_begin = lo;
    rm->row_end = hi;
    rm->n_cols = st->n_cols_b;
    rm->row_ptr = (int64_t *)c->pinned_get(sizeof(int64_t) * ((size_t)n_my + 1));
    rm->col = (int32_t *)c->pinned_get(sizeof(int32_t) * (size_t)std::max<long long>(total, 1));
    if (st->p_cnt) rm->cnt = (int32_t *)c->pinned_get(sizeof(int32_t) * (size_t)std::max<long long>(total, 1));
    if (st->p_llr) rm->llr = (double *)c->pinned_get(sizeof(double) * (size_t)std::max<long long>(total, 1));
    if (!rm->row_ptr || !rm->col || (st->p_cnt && !rm->cnt) || (st->p_llr && !rm->llr))
      return set_error(CCO_E_OOM, "pinned host allocation failed");
    h_rp = rm->row_ptr;
    h_col = rm->col;
    h_cnt = rm->cnt;
    h_llr = rm->llr;
  }
  // out_ptr is 0 up to row lo, so out_ptr[lo .. hi] are the row pointers of this rank's slice relative to its first row
  CK(cudaMemcpyAsync(h_rp, st->out_ptr + lo, sizeof(int64_t) * ((size_t)n_my + 1), cudaMemcpyDeviceToHost, cs));
  if (total > 0 && !(flags & CCO_FLAG_RESULT_ON_DEVICE)) {
    CK(cudaMemcpyAsync(h_col, st->p_col, sizeof(int32_t) * (size_t)total, cudaMemcpyDeviceToHost, cs));
    if (h_cnt) CK(cudaMemcpyAsync(h_cnt, st->p_cnt, sizeof(int32_t) * (size_t)total, cudaMemcpyDeviceToHost, cs));
    if (h_llr) CK(cudaMemcpyAsync(h_llr, st->p_llr, sizeof(double) * (size_t)total, cudaMemcpyDeviceToHost, cs));
  }
  return CCO_OK;
}

static int validate_host(int32_t n_mats, const cco_csr_t *mats, const cco_indicator_params_t *params) {
  if (n_mats < 1 || !mats || !params) return set_error(CCO_E_INVALID_ARG, "need at least the primary matrix and its params");
  for (int i = 0; i < n_mats; ++i) {
    const cco_csr_t &m = mats[i];
    if (!m.row_ptr) return set_error(CCO_E_INVALID_ARG, "matrix %d: null row_ptr", i);
    if (m.n_rows < 0 || m.n_rows >= 0x7fffffffLL) return set_error(CCO_E_INVALID_ARG, "matrix %d: n_rows out of range", i);
    if (m.n_cols < 0 || m.n_cols >= 0x7ffffffe) return set_error(CCO_E_INVALID_ARG, "matrix %d: n_cols out of range", i);
    if (m.n_rows != mats[0].n_rows)
      return set_error(CCO_E_SHAPE_MISMATCH, "matrix %d has %lld rows, the primary has %lld: all event types share the user dictionary",
                       i, (long long)m.n_rows, (long long)mats[0].n_rows);
    if (m.row_ptr[0] != 0) return set_error(CCO_E_INVALID_ARG, "matrix %d: row_ptr[0] != 0", i);
    long long nnz = m.row_ptr[m.n_rows];
    if (nnz < 0 || nnz >= 0xffffffffLL) return set_error(CCO_E_UNSUPPORTED, "matrix %d: nnz %lld outside [0, 2^32)", i, nnz);
    if (nnz > 0 && !m.col_idx) return set_error(CCO_E_INVALID_ARG, "matrix %d: null col_idx", i);
    if (params[i].max_interactions < 1) return set_error(CCO_E_INVALID_ARG, "matrix %d: max_interactions must be >= 1", i);
    if (params[i].top_k < 1) return set_error(CCO_E_INVALID_ARG, "matrix %d: top_k must be >= 1", i);
    if (params[i].top_k > CCO_MAX_TOP_K)
      return set_error(CCO_E_UNSUPPORTED, "matrix %d: top_k %d > CCO_MAX_TOP_K (%d)", i, params[i].top_k, CCO_MAX_TOP_K);
    if (params[i].has_min_llr && params[i].min_llr != params[i].min_llr)
      return set_error(CCO_E_INVALID_ARG, "matrix %d: min_llr is NaN", i);
  }
  return CCO_OK;
}

// the block of user rows rank r of a W-rank job works on
static inline void user_block(long long U, int W, int r, long long *lo, long long *hi) {
  const long long S = (U + W - 1) / W;
  *lo = std::min<long long>((long long)r * S, U);
  *hi = std::min<long long>(*lo + S, U);
}

static void dataset_release(cco_dataset *d) {
  if (!d) return;
  cudaSetDevice(d->ctx->device);
  for (auto p : d->rp_alloc)
    if (p) cudaFreeAsync(p, d->ctx->stream);
  for (auto p : d->col_alloc)
    if (p) cudaFreeAsync(p, d->ctx->stream);
  for (auto e : d->ready)
    if (e) cudaEventDestroy(e);
  delete d;
}

// device check of the uploaded block(s) + canonicalisation of unsorted / duplicated rows (synchronous).  In a multi-GPU
// job the "malformed" verdict is all-reduced so that every rank fails (or proceeds) together.
static int dataset_validate(cco_ctx *c, cco_dataset *d, bool canonicalise) {
  cudaStream_t s = c->stream;
  const int n_mats = d->n_mats;
  Arena ar(s);
  int *d_flags;
  CKR(ar.alloc(&d_flags, 2 * n_mats));
  CK(cudaMemsetAsync(d_flags, 0, sizeof(int) * 2 * n_mats, s));
  for (int i = 0; i < n_mats; ++i) {
    CK(cudaStreamWaitEvent(s, d->ready[i], 0));
    if (d->n_local == 0) continue;
    DevRaw r;
    r.n_rows = d->n_local;
    r.n_cols = (int32_t)d->n_cols[i];
    r.q_base = d->q_lo[i];
    r.nnz = d->q_hi[i] - d->q_lo[i];
    r.rp = d->rp[i];
    r.col = d->col[i];
    HeavyRows hv;
    CKR(list_heavy_rows(c, ar, r, &hv));
    launch_check(c, r, hv, d_flags + 2 * i);
  }
  if (c->world > 1)
    CKR(nccl_check(g_nccl.AllReduce(d_flags, d_flags, (size_t)(2 * n_mats), kNcclInt32, kNcclMax, c->comm, s), "ncclAllReduce(check flags)"));
  std::vector<int> h(2 * n_mats);
  CK(cudaMemcpyAsync(h.data(), d_flags, sizeof(int) * 2 * n_mats, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  for (int i = 0; i < n_mats; ++i)
    if (h[2 * i]) return set_error(CCO_E_INVALID_ARG, "matrix %d: row_ptr not monotone or column index out of [0, n_cols)", i);
  if (canonicalise)
    for (int i = 0; i < n_mats; ++i)
      if (h[2 * i + 1] && d->n_local > 0) {
        // (the flag is all-reduced: every rank canonicalises its own block, the blocks are independent)
        DevRaw r;
        r.n_rows = d->n_local;
        r.row_base = d->row_base;
        r.n_cols = (int32_t)d->n_cols[i];
        r.q_base = d->q_lo[i];
        r.nnz = d->q_hi[i] - d->q_lo[i];
        r.rp = d->rp[i];
        r.col = d->col[i];
        CKR(canonicalize_device(c, ar, r));
        d->col[i] = r.col;
        d->q_lo[i] = 0;
        d->q_hi[i] = r.nnz;
        if (c->world == 1) d->nnz[i] = r.nnz;
      }
  CK(cudaStreamSynchronize(s));
  d->validated = canonicalise;
  return CCO_OK;
}

// host CSR -> device: this rank's block of user rows only (the dataset owns its buffers until cco_dataset_free)
static int dataset_upload(cco_ctx *c, int32_t n_mats, const cco_csr_t *mats, uint32_t flags, cco_dataset **out, bool async = false) {
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  cco_dataset *d = new cco_dataset();
  d->ctx = c;
  d->n_mats = n_mats;
  d->n_users = mats[0].n_rows;
  long long u_lo, u_hi;
  user_block(d->n_users, c->world, c->rank, &u_lo, &u_hi);
  d->row_base = u_lo;
  d->n_local = u_hi - u_lo;
  d->whole = c->world == 1;
  d->rp.assign(n_mats, nullptr);
  d->col.assign(n_mats, nullptr);
  d->rp_alloc.assign(n_mats, nullptr);
  d->col_alloc.assign(n_mats, nullptr);
  d->n_cols.assign(n_mats, 0);
  d->nnz.assign(n_mats, 0);
  d->block_cap.assign(n_mats, 0);
  d->q_lo.assign(n_mats, 0);
  d->q_hi.assign(n_mats, 0);
  d->ready.assign(n_mats, nullptr);
  struct G {
    cco_dataset *d;
    bool ok = false;
    ~G() {
      if (!ok) dataset_release(d);
    }
  } g{d};
  // allocations are ordered on the main stream; the copies run on the copy stream (H2D engine) so that the caller
  // of the async form can start preparing matrix i while matrix i+1 is still in flight
  cudaStream_t cs = c->copy_stream;
  for (int i = 0; i < n_mats; ++i) {
    const cco_csr_t &m = mats[i];
    d->n_cols[i] = m.n_cols;
    d->nnz[i] = m.row_ptr[m.n_rows];
    for (int q = 0; q < c->world; ++q) {
      long long a0, a1;
      user_block(d->n_users, c->world, q, &a0, &a1);
      d->block_cap[i] = std::max<long long>(d->block_cap[i], m.row_ptr[a1] - m.row_ptr[a0]);
    }
    const long long q0 = m.row_ptr[u_lo], q1 = m.row_ptr[u_hi];
    d->q_lo[i] = q0;
    d->q_hi[i] = q1;
    void *p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, sizeof(int64_t) * ((size_t)d->n_local + 1), s);
    if (e != cudaSuccess) return set_error(CCO_E_OOM, "cudaMallocAsync row_ptr: %s", cudaGetErrorString(e));
    d->rp_alloc[i] = p;
    d->rp[i] = (long long *)p;
    e = cudaMallocAsync(&p, sizeof(int32_t) * (size_t)std::max<long long>(q1 - q0, 4), s);
    if (e != cudaSuccess) return set_error(CCO_E_OOM, "cudaMallocAsync col_idx: %s", cudaGetErrorString(e));
    d->col_alloc[i] = p;
    d->col[i] = (int32_t *)p - q0;   // the block keeps the caller's absolute offsets: col[rp[r]] addresses its own storage
    CK(cudaEventCreateWithFlags(&d->ready[i], cudaEventDisableTiming));
  }
  CK(cudaEventRecord(c->copy_ev[0], s));
  CK(cudaStreamWaitEvent(cs, c->copy_ev[0], 0));
  CK(cudaEventRecord(c->ev[6], cs));
  for (int i = 0; i < n_mats; ++i) {
    const cco_csr_t &m = mats[i];
    const long long q0 = m.row_ptr[u_lo], q1 = m.row_ptr[u_hi];
    CK(cudaMemcpyAsync(d->rp_alloc[i], m.row_ptr + u_lo, sizeof(int64_t) * ((size_t)d->n_local + 1), cudaMemcpyHostToDevice, cs));
    if (q1 > q0)
      CK(cudaMemcpyAsync(d->col_alloc[i], m.col_idx + q0, sizeof(int32_t) * (size_t)(q1 - q0), cudaMemcpyHostToDevice, cs));
    CK(cudaEventRecord(d->ready[i], cs));
  }
  CK(cudaEventRecord(c->ev[7], cs));
  if (async && (flags & CCO_FLAG_ASSUME_CANONICAL)) {
    d->h2d_pending = true;   // the malformed-input check runs inside the train, next to the first pass over the data
    g.ok = true;
    *out = d;
    return CCO_OK;
  }
  CKR(dataset_validate(c, d, !(flags & CCO_FLAG_ASSUME_CANONICAL)));
  CK(cudaEventElapsedTime(&d->ms_h2d, c->ev[6], c->ev[7]));
  g.ok = true;
  *out = d;
  return CCO_OK;
}

// The whole hot path on this rank, for the block of users the dataset holds.
static int train_dataset(cco_ctx *c, const cco_dataset *ds, const cco_indicator_params_t *params, int32_t seed, uint32_t flags,
                         cco_result **out) {
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const int n_mats = ds->n_mats;
  mail_reset(c);
  c->ev_timing_used = c->ev_plain_used = 0;
  Arena ar(s, c);
  struct CopyJoin {  // destroyed before `ar`: no packed buffer is freed while the copy stream still reads it
    cco_ctx *c;
    ~CopyJoin() {
      cudaStreamSynchronize(c->copy_stream);
      cudaStreamSynchronize(c->sched_stream);   // error paths: no schedule kernel outlives the train's slab memory
    }
  } copy_join{c};
  cco_result *res = new cco_result();
  res->ctx = c;
  res->mats.resize(n_mats);
  memset(&res->stats, 0, sizeof res->stats);
  struct Guard {
    cco_result *r;
    bool ok = false;
    ~Guard() {
      if (!ok) cco_result_free(r);
    }
  } guard{res};
  std::vector<IndicatorState> ist(n_mats);
  for (auto &x : ist) CKR(pooled_event(c, false, &x.packed));
  cco_stats_t &st = res->stats;
  st.n_mats = n_mats;
  st.n_users = ds->n_users;
  st.ms_h2d = ds->ms_h2d;
  const bool h2d_pending = ds->h2d_pending;
  const long long n_users = ds->n_users;
  std::vector<DevRaw> raw(n_mats);
  for (int i = 0; i < n_mats; ++i) {
    raw[i].n_rows = ds->n_local;
    raw[i].row_base = ds->row_base;
    raw[i].n_cols = (int32_t)ds->n_cols[i];
    raw[i].q_base = ds->q_lo[i];
    raw[i].nnz = ds->q_hi[i] - ds->q_lo[i];   // entries of the block
    raw[i].nnz_cap = ds->nnz[i];
    raw[i].rp = ds->rp[i];
    raw[i].col = ds->col[i];
    st.nnz_in_total += ds->nnz[i];
  }
  CK(cudaEventRecord(c->ev[1], s));
  nvtx_push("cco:prepare");
  std::vector<cudaEvent_t> sev(8, nullptr);   // stage boundaries of the preparation (cco_stats_t.ms_prep_stage)
  for (auto &e : sev) CKR(pooled_event(c, true, &e));
  auto mark = [&](int k) { return cudaEventRecord(sev[k], s); };
  // raw column counts: this rank histograms its user block; ONE allreduce sums all matrices' counts
  long long total_cols = 0;
  std::vector<long long> col_off(n_mats + 1, 0);
  for (int i = 0; i < n_mats; ++i) {
    col_off[i] = total_cols;
    total_cols += raw[i].n_cols;
  }
  col_off[n_mats] = total_cols;
  constexpr int kHistCopies = 16;
  const long long copy_stride = std::max<long long>(total_cols, 1);
  int32_t *raw_counts, *marg_all;
  int *d_check;
  CKR(ar.alloc(&raw_counts, (size_t)copy_stride * kHistCopies));
  CKR(ar.alloc(&marg_all, (size_t)copy_stride));
  CKR(ar.alloc(&d_check, 2 * n_mats));
  CK(cudaMemsetAsync(raw_counts, 0, sizeof(int32_t) * (size_t)copy_stride * kHistCopies, s));
  CK(cudaMemsetAsync(marg_all, 0, sizeof(int32_t) * (size_t)copy_stride, s));
  CK(cudaMemsetAsync(d_check, 0, sizeof(int) * 2 * n_mats, s));
  for (int i = 0; i < n_mats; ++i) {
    CK(cudaStreamWaitEvent(s, ds->ready[i], 0));  // matrix i has landed (async upload: later ones may still be in flight)
    if (ds->n_local == 0) continue;
    // CCO_FLAG_ASSUME_CANONICAL skips the canonicalisation, not the safety net: a malformed matrix still fails the call
    // (until the verdict is read, the histogram skips ids outside the column space and the sampler keeps nothing)
    int *verdict = ds->validated ? nullptr : d_check + 2 * i;
    if (verdict) {
      k_check_row_ptr<<<grid_for(raw[i].n_rows, 256, c->sm_count), 256, 0, s>>>(raw[i].n_rows, raw[i].rp, raw[i].q_base, raw[i].q_base + raw[i].nnz,
                                                                              verdict);
      c->launches++;
    }
    if (raw[i].nnz > 0) {
      // warp-aggregated (__match_any_sync) before the atomics: 0.50 ms for the four C3 matrices against 0.53 ms without
      k_col_histogram_flat<true><<<grid_for(raw[i].nnz, 256, c->sm_count), 256, 0, s>>>(raw[i].nnz, raw[i].col + raw[i].q_base, raw[i].n_cols,
                                                                                       raw_counts + col_off[i], kHistCopies, copy_stride, verdict);
      c->launches++;
    }
  }
  if (total_cols > 0) {
    k_sum_copies<<<grid_for(total_cols, 256, c->sm_count), 256, 0, s>>>(total_cols, kHistCopies, copy_stride, raw_counts);
    c->launches++;
  }
  CK(mark(0));
  if (c->world > 1) {
    if (total_cols > 0)
      CKR(nccl_check(g_nccl.AllReduce(raw_counts, raw_counts, (size_t)total_cols, kNcclInt32, kNcclSum, c->comm, s), "ncclAllReduce(raw counts)"));
    CKR(nccl_check(g_nccl.AllReduce(d_check, d_check, (size_t)(2 * n_mats), kNcclInt32, kNcclMax, c->comm, s), "ncclAllReduce(check flags)"));
  }
  CK(mark(1));
  // sampleDownAndBinarize every matrix
  std::vector<DevMat> dm(n_mats);
  if (c->world > 1) {
    CKR(downsample_sharded_all(c, ar, raw, d_check, ds->block_cap, n_users, raw_counts, marg_all, col_off, params, seed, flags, dm, &sev[2]));
  } else {
    for (int i = 0; i < n_mats; ++i) {
      dm[i].marg = marg_all + col_off[i];
      CKR(downsample_device(c, ar, raw[i], d_check + 2 * i, raw_counts + col_off[i], params[i].max_interactions, seed, flags, &dm[i]));
    }
    CK(mark(2));   // single GPU: both passes are booked on stage 2 ... 4 as one block
    CK(mark(3));
    CK(mark(4));
    CK(mark(5));
  }
  // `drmA.t`
  const int32_t n_items_a = dm[0].n_cols;
  uint32_t *at_ptr, *cursor;
  int32_t *at_users, *d_max;
  CKR(ar.alloc(&at_ptr, n_items_a + 1));
  CKR(ar.alloc(&cursor, n_items_a + 1));
  CKR(ar.alloc(&d_max, n_mats));
  CKR(ar.alloc(&at_users, std::max<long long>(ds->nnz[0], 1)));
  CK(cudaMemsetAsync(d_max, 0, 4 * (size_t)n_mats, s));
  {
    uint32_t *marg_pad;
    CKR(ar.alloc(&marg_pad, n_items_a + 1));
    CK(cudaMemcpyAsync(marg_pad, dm[0].marg, sizeof(int32_t) * (size_t)n_items_a, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemsetAsync(marg_pad + n_items_a, 0, 4, s));
    CKR(exclusive_sum_u32(c, ar, marg_pad, at_ptr, (long long)n_items_a + 1));
    ar.release(marg_pad);
  }
  CK(cudaMemcpyAsync(cursor, at_ptr, sizeof(uint32_t) * ((size_t)n_items_a + 1), cudaMemcpyDeviceToDevice, s));
  k_transpose_scatter<<<grid_for(n_users * kSG, 256, c->sm_count), 256, 0, s>>>(n_users, dm[0].rp, dm[0].col, cursor, at_users);
  c->launches++;
  for (int i = 0; i < n_mats; ++i)
    if (dm[i].n_cols > 0) {
      k_max_i32<<<grid_for(dm[i].n_cols, 256, c->sm_count, 2), 256, 0, s>>>(dm[i].n_cols, dm[i].marg, d_max + i);
      c->launches++;
    }
  std::vector<int32_t> max_marg(n_mats, 0);
  std::vector<uint32_t> h_nnz(n_mats);
  std::vector<int> h_check(2 * n_mats, 0);
  CKR(mail_fetch(c, max_marg.data(), d_max, 4 * (size_t)n_mats));
  CKR(mail_fetch(c, h_check.data(), d_check, sizeof(int) * 2 * (size_t)n_mats));
  for (int i = 0; i < n_mats; ++i) CKR(mail_fetch(c, &h_nnz[i], dm[i].rp + n_users, 4));
  CK(mark(6));
  CK(cudaEventRecord(c->ev[2], s));
  nvtx_pop();
  CKR(mail_wait(c));   // the one host round trip of the preparation: the packed-word check needs the largest marginals
  for (int i = 0; i < n_mats; ++i)
    if (h_check[2 * i]) return set_error(CCO_E_INVALID_ARG, "matrix %d: row_ptr not monotone or column index out of [0, n_cols)", i);
  for (int i = 0; i < n_mats && i < 16; ++i) st.nnz_downsampled[i] = h_nnz[i];

  // indicators, software-pipelined: indicator i+1 is on the stream before the host waits for indicator i's record
  std::vector<IndicatorOut> io(n_mats);
  std::vector<cudaEvent_t> ev_rows(2 * n_mats, nullptr);
  for (auto &e : ev_rows) CKR(pooled_event(c, true, &e));
  for (int i = 0; i < n_mats; ++i) {
    nvtx_push("cco:indicator");
    CKR(enqueue_indicator(c, ar, at_ptr, at_users, n_items_a, dm[0].marg, max_marg[0], max_marg[i], dm[i], n_users, i == 0, params[i],
                          flags, false, c->ev[2], ev_rows[2 * i], ev_rows[2 * i + 1], &ist[i]));
    nvtx_pop();
    if (i > 0) CKR(finish_indicator(c, &ist[i - 1], flags, i - 1, &res->mats[i - 1], &io[i - 1]));
  }
  CKR(finish_indicator(c, &ist[n_mats - 1], flags, n_mats - 1, &res->mats[n_mats - 1], &io[n_mats - 1]));
  CK(cudaEventRecord(c->copy_ev[1], c->copy_stream));
  CK(cudaStreamWaitEvent(s, c->copy_ev[1], 0));
  CK(cudaEventRecord(c->ev[3], s));
  CK(cudaStreamSynchronize(s));
  CK(cudaStreamSynchronize(c->copy_stream));
  for (int i = 0; i < n_mats && i < 16; ++i) {
    st.products[i] = io[i].products;
    st.distinct_cells[i] = io[i].distinct;
    st.llr_evaluated[i] = io[i].evaluated;
    st.out_nnz[i] = io[i].nnz;
    CK(cudaEventElapsedTime(&st.ms_indicator[i], ev_rows[2 * i], ev_rows[2 * i + 1]));
  }
  if (h2d_pending) CK(cudaEventElapsedTime(&st.ms_h2d, c->ev[6], c->ev[7]));
  CK(cudaEventElapsedTime(&st.ms_prep_stage[0], c->ev[1], sev[0]));
  for (int k = 1; k <= 6; ++k) CK(cudaEventElapsedTime(&st.ms_prep_stage[k], sev[k - 1], sev[k]));
  CK(cudaEventElapsedTime(&st.ms_prepare, c->ev[1], c->ev[2]));
  CK(cudaEventElapsedTime(&st.ms_cooccurrence, c->ev[2], c->ev[3]));
  CK(cudaEventElapsedTime(&st.ms_total, c->ev[1], c->ev[3]));
  if (!h2d_pending) st.ms_total += st.ms_h2d;  // async upload overlaps the prepare stage: already inside the bracket
  st.n_kernel_launches = c->launches;
  guard.ok = true;
  *out = res;
  return CCO_OK;
}

static int train_impl(cco_ctx *c, int32_t n_mats, const cco_csr_t *mats, const cco_indicator_params_t *params, int32_t seed,
                      uint32_t flags, cco_result **out) {
  c->launches = 0;
  cco_dataset *ds = nullptr;
  CKR(dataset_upload(c, n_mats, mats, flags, &ds, /*async=*/true));
  int rc = train_dataset(c, ds, params, seed, flags, out);
  cudaStreamSynchronize(c->copy_stream);  // the caller's host buffers are free again when cco_train returns
  dataset_release(ds);
  return rc;
}

// cco_train on a group context: one host thread per GPU runs the per-rank train on its member context (same host
// matrices, each thread uploads its block of users); the slices meet in one merged result owned by the leader.
static int train_group(cco_ctx *leader, int32_t n_mats, const cco_csr_t *mats, const cco_indicator_params_t *params, int32_t seed,
                       uint32_t flags, cco_result **out) {
  const int W = (int)leader->members.size();
  GroupShared *gs = leader->members[0]->gshared;
  cco_result *merged = new cco_result();
  merged->ctx = leader;
  merged->mats.resize(n_mats);
  memset(&merged->stats, 0, sizeof merged->stats);
  gs->merged = merged;
  gs->totals.assign(W, 0);
  gs->status = CCO_OK;
  gs->err[0] = 0;
  std::vector<cco_result *> part(W, nullptr);
  std::vector<std::thread> th;
  for (int r = 0; r < W; ++r)
    th.emplace_back([&, r]() {
      int rc = train_impl(leader->members[r], n_mats, mats, params, seed, flags, &part[r]);
      if (rc != CCO_OK) {
        std::lock_guard<std::mutex> lk(gs->mu);
        if (gs->status == CCO_OK) {
          gs->status = rc;
          snprintf(gs->err, sizeof gs->err, "GPU %d: %s", leader->members[r]->device, cco_last_error());
        }
      }
    });
  for (auto &t : th) t.join();
  gs->merged = nullptr;
  if (gs->status != CCO_OK) {
    for (auto p : part)
      if (p) cco_result_free(p);
    cco_result_free(merged);
    return set_error(gs->status, "%s", gs->err);
  }
  cco_stats_t &st = merged->stats;
  st = part[0]->stats;
  for (int r = 1; r < W; ++r) {
    const cco_stats_t &p = part[r]->stats;
    for (int i = 0; i < 16; ++i) {
      st.products[i] += p.products[i];
      st.distinct_cells[i] += p.distinct_cells[i];
      st.out_nnz[i] += p.out_nnz[i];
      st.llr_evaluated[i] += p.llr_evaluated[i];
      st.ms_indicator[i] = std::max(st.ms_indicator[i], p.ms_indicator[i]);
    }
    st.ms_h2d = std::max(st.ms_h2d, p.ms_h2d);
    st.ms_prepare = std::max(st.ms_prepare, p.ms_prepare);
    st.ms_cooccurrence = std::max(st.ms_cooccurrence, p.ms_cooccurrence);
    st.ms_total = std::max(st.ms_total, p.ms_total);
    st.n_kernel_launches += p.n_kernel_launches;
  }
  for (auto p : part) cco_result_free(p);
  *out = merged;
  return CCO_OK;
}

}  // namespace cco

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int cco_abi_version(void) { return CCO_ABI_VERSION; }
const char *cco_last_error(void) { return g_err; }
const char *cco_status_string(int s) {
  switch (s) {
    case CCO_OK: return "ok";
    case CCO_E_INVALID_ARG: return "invalid argument";
    case CCO_E_CUDA: return "CUDA error";
    case CCO_E_NCCL: return "NCCL error";
    case CCO_E_OOM: return "out of memory";
    case CCO_E_SHAPE_MISMATCH: return "shape mismatch";
    case CCO_E_UNSUPPORTED: return "unsupported";
  }
  return "unknown";
}

int cco_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) return set_error(CCO_E_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ++ok;
  }
  return ok;
}

int cco_nccl_unique_id(unsigned char out[128]) {
  if (!out) return set_error(CCO_E_INVALID_ARG, "null output");
  CKR(load_nccl());
  ncclUniqueId id;
  int r = g_nccl.GetUniqueId(&id);
  if (r != 0) return set_error(CCO_E_NCCL, "ncclGetUniqueId: %s", g_nccl.GetErrorString(r));
  memcpy(out, id.internal, 128);
  return CCO_OK;
}

// streams, events, mailbox, memory pool of one per-GPU context (the NCCL communicator is attached by the caller)
static int ctx_init_device(cco_ctx *c) {
  CK(cudaSetDevice(c->device));
  CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  for (auto &ev : c->ev) CK(cudaEventCreate(&ev));
  for (auto &ev : c->tev) CK(cudaEventCreate(&ev));
  for (auto &ev : c->copy_ev) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  for (auto &st : c->bin_stream) CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&c->sched_stream, cudaStreamNonBlocking));
  for (auto &ev : c->bin_ev) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  CK(cudaHostAlloc((void **)&c->mail_h, kMailBytes, cudaHostAllocMapped | cudaHostAllocPortable));
  CK(cudaHostGetDevicePointer((void **)&c->mail_d, c->mail_h, 0));
  cudaMemPool_t pool;
  CK(cudaDeviceGetDefaultMemPool(&pool, c->device));
  uint64_t thr = UINT64_MAX;  // keep freed blocks: steady-state trains allocate nothing
  CK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
  return CCO_OK;
}

static int check_device(int device, cudaDeviceProp *p) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return set_error(CCO_E_CUDA, "no CUDA device (%s): this library has no CPU fallback",
                     e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  if (device < 0 || device >= n) return set_error(CCO_E_INVALID_ARG, "device %d not in [0,%d)", device, n);
  CK(cudaGetDeviceProperties(p, device));
  if (p->major != 10)
    return set_error(CCO_E_CUDA, "device %d is sm_%d%d; this build contains sm_100a code only", device, p->major, p->minor);
  return CCO_OK;
}

static int create_failed(cco_ctx *c, int st) {
  char keep[sizeof g_err];
  memcpy(keep, g_err, sizeof keep);   // cco_destroy must not clobber the message
  cco_destroy(c);
  memcpy(g_err, keep, sizeof keep);
  return st;
}

int cco_create(const cco_config_t *cfg, cco_ctx_t **out) {
  if (!cfg || !out) return set_error(CCO_E_INVALID_ARG, "null argument");
  if (cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size)
    return set_error(CCO_E_INVALID_ARG, "bad rank/world_size %d/%d", cfg->rank, cfg->world_size);
  if (cfg->world_size > 1023) return set_error(CCO_E_UNSUPPORTED, "world_size %d > 1023", cfg->world_size);
  cudaDeviceProp p;
  CKR(check_device(cfg->device, &p));
  if (cfg->world_size > 1 && !cfg->nccl_unique_id) return set_error(CCO_E_INVALID_ARG, "world_size > 1 needs nccl_unique_id");
  cco_ctx *c = new cco_ctx();
  c->device = cfg->device;
  c->rank = cfg->rank;
  c->world = cfg->world_size;
  c->sm_count = p.multiProcessorCount;
  c->smem_optin = p.sharedMemPerBlockOptin;
  // every failure below releases what was created so far (cco_destroy tolerates a half-built context)
  auto init = [&]() -> int {
    CKR(ctx_init_device(c));
    if (cfg->result_arena && cfg->result_arena_bytes > 0) {
      // caller-provided result memory (e.g. a shared-memory segment the reading process maps): page-lock it so the
      // device->host copies of the indicators land there directly
      CK(cudaHostRegister(cfg->result_arena, cfg->result_arena_bytes, cudaHostRegisterPortable));
      c->arena = (unsigned char *)cfg->result_arena;
      c->arena_bytes = cfg->result_arena_bytes;
      c->arena_registered = true;
    }
    if (c->world > 1) {
      CKR(load_nccl());
      ncclUniqueId id;
      memcpy(id.internal, cfg->nccl_unique_id, 128);
      int rc = g_nccl.CommInitRank(&c->comm, c->world, id, c->rank);
      if (rc != 0) return set_error(CCO_E_NCCL, "ncclCommInitRank: %s", g_nccl.GetErrorString(rc));
    }
    return CCO_OK;
  };
  const int st = init();
  if (st != CCO_OK) return create_failed(c, st);
  *out = c;
  return CCO_OK;
}

// One context over several GPUs of this process (what a single JVM thread can drive): member r runs on devices[r] with
// its own streams; the communicator comes from ncclCommInitAll; cco_train runs one host thread per member.
int cco_create_group(int32_t n_devices, const int32_t *devices, cco_ctx_t **out) {
  if (!devices || !out || n_devices < 1) return set_error(CCO_E_INVALID_ARG, "bad argument");
  if (n_devices > 1023) return set_error(CCO_E_UNSUPPORTED, "more than 1023 devices");
  std::vector<cudaDeviceProp> props(n_devices);
  for (int r = 0; r < n_devices; ++r) {
    CKR(check_device(devices[r], &props[r]));
    for (int q = 0; q < r; ++q)
      if (devices[q] == devices[r]) return set_error(CCO_E_INVALID_ARG, "device %d listed twice", devices[r]);
  }
  cco_ctx *leader = new cco_ctx();
  leader->device = devices[0];
  leader->world = 1;
  GroupShared *gs = new GroupShared();
  gs->world = n_devices;
  auto init = [&]() -> int {
    std::vector<ncclComm_t> comms(n_devices, nullptr);
    if (n_devices > 1) {
      CKR(load_nccl());
      std::vector<int> devs(devices, devices + n_devices);
      int rc = g_nccl.CommInitAll(comms.data(), n_devices, devs.data());
      if (rc != 0) return set_error(CCO_E_NCCL, "ncclCommInitAll: %s", g_nccl.GetErrorString(rc));
    }
    for (int r = 0; r < n_devices; ++r) {
      cco_ctx *m = new cco_ctx();
      m->device = devices[r];
      m->rank = r;
      m->world = n_devices;
      m->sm_count = props[r].multiProcessorCount;
      m->smem_optin = props[r].sharedMemPerBlockOptin;
      m->comm = comms[r];
      m->gshared = gs;
      leader->members.push_back(m);
      CKR(ctx_init_device(m));
    }
    CK(cudaSetDevice(devices[0]));
    return CCO_OK;
  };
  const int st = init();
  if (st != CCO_OK) {
    if (leader->members.empty()) delete gs;
    return create_failed(leader, st);
  }
  *out = leader;
  return CCO_OK;
}

int cco_destroy(cco_ctx_t *c) {
  if (!c) return CCO_OK;
  if (!c->members.empty()) {
    GroupShared *gs = c->members[0]->gshared;
    for (cco_ctx *m : c->members) {
      m->gshared = nullptr;
      cco_destroy(m);
    }
    c->members.clear();
    delete gs;
  }
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
  if (c->comm) g_nccl.CommDestroy(c->comm);
  for (auto &b : c->pinned) cudaFreeHost(b.p);
  if (c->arena_registered) cudaHostUnregister(c->arena);
  if (c->mail_h) cudaFreeHost(c->mail_h);
  for (auto &ev : c->mail_ev) cudaEventDestroy(ev);
  for (auto &ev : c->ev_timing) cudaEventDestroy(ev);
  for (auto &ev : c->ev_plain) cudaEventDestroy(ev);
  for (auto &sl : c->slabs) cudaFree(sl.p);
  for (auto &ev : c->ev)
    if (ev) cudaEventDestroy(ev);
  for (auto &ev : c->tev)
    if (ev) cudaEventDestroy(ev);
  for (auto &ev : c->copy_ev)
    if (ev) cudaEventDestroy(ev);
  for (auto &st : c->bin_stream)
    if (st) cudaStreamDestroy(st);
  if (c->sched_stream) cudaStreamDestroy(c->sched_stream);
  for (auto &ev : c->bin_ev)
    if (ev) cudaEventDestroy(ev);
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  delete c;
  return CCO_OK;
}

int cco_host_alloc(cco_ctx_t *c, size_t bytes, void **out) {
  if (!c || !out) return set_error(CCO_E_INVALID_ARG, "null argument");
  CK(cudaSetDevice(c->device));
  void *p = c->pinned_get(bytes, /*for_result=*/false);
  if (!p) return set_error(CCO_E_OOM, "cudaHostAlloc(%zu) failed", bytes);
  *out = p;
  return CCO_OK;
}
int cco_host_free(cco_ctx_t *c, void *p) {
  if (!c) return set_error(CCO_E_INVALID_ARG, "null context");
  if (p) c->pinned_put(p);
  return CCO_OK;
}

int cco_train(cco_ctx_t *ctx, int32_t n_mats, const cco_csr_t *mats, const cco_indicator_params_t *params, int32_t seed,
              uint32_t flags, cco_result_t **out) {
  if (!ctx || !out) return set_error(CCO_E_INVALID_ARG, "null argument");
  *out = nullptr;
  CKR(validate_host(n_mats, mats, params));   // everything the host can check, before any GPU (or thread) starts
  if (!ctx->members.empty()) return train_group(ctx, n_mats, mats, params, seed, flags, out);
  return train_impl(ctx, n_mats, mats, params, seed, flags, out);
}

int cco_cooccurrences_idss(cco_ctx_t *ctx, int32_t n_mats, const cco_csr_t *mats, int32_t seed,
                           int32_t max_interesting_items_per_thing, int32_t max_num_interactions, uint32_t flags,
                           cco_result_t **out) {
  if (n_mats < 1) return set_error(CCO_E_INVALID_ARG, "need at least the primary matrix");
  std::vector<cco_indicator_params_t> p(n_mats);
  for (auto &q : p) {
    q.max_interactions = max_num_interactions;
    q.top_k = max_interesting_items_per_thing;
    q.has_min_llr = 0;
    q.min_llr = 0.0;
  }
  return cco_train(ctx, n_mats, mats, p.data(), seed, flags, out);
}

int cco_dataset_shape(const cco_dataset_t *ds, int32_t i, int64_t *n_rows, int32_t *n_cols, int64_t *nnz) {
  if (!ds || i < 0 || i >= ds->n_mats) return set_error(CCO_E_INVALID_ARG, "bad dataset/index");
  if (n_rows) *n_rows = ds->n_users;
  if (n_cols) *n_cols = (int32_t)ds->n_cols[i];
  if (nnz) *nnz = ds->nnz[i];
  return CCO_OK;
}

int cco_dataset_download(const cco_dataset_t *ds, int32_t i, int64_t **row_ptr, int32_t **col_idx) {
  if (!ds || !row_ptr || !col_idx || i < 0 || i >= ds->n_mats) return set_error(CCO_E_INVALID_ARG, "bad argument");
  if (!ds->whole) return set_error(CCO_E_UNSUPPORTED, "this dataset holds one rank's block of users only");
  cco_ctx *c = ds->ctx;
  CK(cudaSetDevice(c->device));
  int64_t *rp = (int64_t *)malloc(sizeof(int64_t) * ((size_t)ds->n_users + 1));
  int32_t *ci = (int32_t *)malloc(sizeof(int32_t) * (size_t)std::max<long long>(ds->nnz[i], 1));
  if (!rp || !ci) return set_error(CCO_E_OOM, "malloc failed");
  CK(cudaStreamSynchronize(c->copy_stream));
  CK(cudaMemcpyAsync(rp, ds->rp_alloc[i], sizeof(int64_t) * ((size_t)ds->n_users + 1), cudaMemcpyDeviceToHost, c->stream));
  if (ds->nnz[i] > 0)
    CK(cudaMemcpyAsync(ci, ds->col_alloc[i], sizeof(int32_t) * (size_t)ds->nnz[i], cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  *row_ptr = rp;
  *col_idx = ci;
  return CCO_OK;
}

// Preparator.prepare on the device (SURVEY.md 8f-1): histogram + scans for the dictionaries, one radix sort + unique
// per event type for the binary CSR.  The events of a type reach the device through `fill` (a host->device copy for
// cco_ingest, the generator kernel for cco_synth_ingest) right before the type is processed.
struct IngestSource {
  int n_types = 0;
  long long n_users_raw = 0;
  std::vector<long long> n_events;
  std::vector<int32_t> n_items_raw;
  bool keep_item_space = false;   // synthetic workloads: the item dictionary is the raw id space (identity map)
  // fill(t, d_user, d_item): enqueue on the context's stream whatever puts type t's raw events into the two arrays
  std::function<int(int, long long *, int32_t *)> fill;
};

static int ingest_core(cco_ctx *c, const IngestSource &src, int32_t min_events_per_user, int32_t *user_map,
                       int32_t *const *item_maps, cco_dataset **out) {
  const int n_types = src.n_types;
  const long long n_users_raw = src.n_users_raw;
  *out = nullptr;
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  mail_reset(c);
  Arena ar(s);
  cco_dataset *d = new cco_dataset();
  d->ctx = c;
  d->n_mats = n_types;
  d->rp.assign(n_types, nullptr);
  d->col.assign(n_types, nullptr);
  d->rp_alloc.assign(n_types, nullptr);
  d->col_alloc.assign(n_types, nullptr);
  d->block_cap.assign(n_types, 0);
  d->q_lo.assign(n_types, 0);
  d->q_hi.assign(n_types, 0);
  d->n_cols.assign(n_types, 0);
  d->nnz.assign(n_types, 0);
  d->ready.assign(n_types, nullptr);
  d->validated = true;   // built here: canonical by construction
  d->whole = true;
  struct G {
    cco_dataset *d;
    bool ok = false;
    ~G() {
      if (!ok) dataset_release(d);
    }
  } g{d};
  const long long nu = std::max<long long>(n_users_raw, 1);
  int32_t *cnt, *d_user_map;
  uint32_t *uflag, *upos;
  CKR(ar.alloc(&cnt, nu));
  CKR(ar.alloc(&uflag, nu + 1));
  CKR(ar.alloc(&upos, nu + 1));
  CKR(ar.alloc(&d_user_map, nu));
  uint32_t n_users = 0;
  for (int t = 0; t < n_types; ++t) {
    const long long ne = src.n_events[t], ni = std::max<int32_t>(src.n_items_raw[t], 1);
    long long *d_user;
    int32_t *d_item;
    CKR(ar.alloc(&d_user, std::max<long long>(ne, 1)));
    CKR(ar.alloc(&d_item, std::max<long long>(ne, 1)));
    if (ne > 0) CKR(src.fill(t, d_user, d_item));
    if (t == 0) {
      // user dictionary from the primary events (duplicates count: Preparator.scala:129-132)
      CK(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (size_t)nu, s));
      CK(cudaMemsetAsync(uflag, 0, sizeof(uint32_t) * ((size_t)nu + 1), s));
      if (ne > 0) k_ingest_count_users<<<grid_for(ne, 256, c->sm_count), 256, 0, s>>>(ne, d_user, cnt);
      const int32_t need = min_events_per_user > 1 ? min_events_per_user : 1;
      if (n_users_raw > 0)
        k_ingest_user_flags<<<grid_for(n_users_raw, 256, c->sm_count), 256, 0, s>>>(n_users_raw, cnt, need, uflag);
      CKR(exclusive_sum_u32(c, ar, uflag, upos, nu + 1));
      if (n_users_raw > 0)
        k_ingest_make_map<<<grid_for(n_users_raw, 256, c->sm_count), 256, 0, s>>>(n_users_raw, uflag, upos, d_user_map);
      c->launches += 3;
      CKR(mail_fetch(c, &n_users, upos + n_users_raw, 4));
      if (n_users_raw > 0 && user_map)
        CK(cudaMemcpyAsync(user_map, d_user_map, sizeof(int32_t) * (size_t)n_users_raw, cudaMemcpyDeviceToHost, s));
      CKR(mail_wait(c));
      d->n_users = n_users;
    }
    uint32_t *iflag, *ipos;
    int32_t *d_item_map;
    CKR(ar.alloc(&iflag, ni + 1));
    CKR(ar.alloc(&ipos, ni + 1));
    CKR(ar.alloc(&d_item_map, ni));
    if (src.keep_item_space) {
      CK(cudaMemsetAsync(iflag + ni, 0, 4, s));
      k_fill_u32<<<grid_for(ni, 256, c->sm_count), 256, 0, s>>>(ni, 1u, iflag);
    } else {
      CK(cudaMemsetAsync(iflag, 0, sizeof(uint32_t) * ((size_t)ni + 1), s));
      if (ne > 0) k_ingest_item_flags<<<grid_for(ne, 256, c->sm_count), 256, 0, s>>>(ne, d_user, d_item, d_user_map, iflag);
    }
    CKR(exclusive_sum_u32(c, ar, iflag, ipos, ni + 1));
    k_ingest_make_map<<<grid_for(ni, 256, c->sm_count), 256, 0, s>>>(src.n_items_raw[t], iflag, ipos, d_item_map);
    uint32_t n_items = 0;
    CKR(mail_fetch(c, &n_items, ipos + src.n_items_raw[t], 4));
    if (src.n_items_raw[t] > 0 && item_maps && item_maps[t])
      CK(cudaMemcpyAsync(item_maps[t], d_item_map, sizeof(int32_t) * (size_t)src.n_items_raw[t], cudaMemcpyDeviceToHost, s));
    // sort surviving (user, item) keys, drop duplicates, rebuild row_ptr
    unsigned long long *k0, *k1, *d_kept;
    CKR(ar.alloc(&k0, std::max<long long>(ne, 1)));
    CKR(ar.alloc(&k1, std::max<long long>(ne, 1)));
    CKR(ar.alloc(&d_kept, 1));
    CK(cudaMemsetAsync(d_kept, 0, 8, s));
    if (ne > 0) k_ingest_keys<<<grid_for(ne, 256, c->sm_count), 256, 0, s>>>(ne, d_user, d_item, d_user_map, d_item_map, k0, d_kept);
    c->launches += 3;
    unsigned long long kept = 0;
    CKR(mail_fetch(c, &kept, d_kept, 8));
    CKR(mail_wait(c));
    ar.release(d_user);   // the raw events are dead once the keys exist
    ar.release(d_item);
    d->n_cols[t] = n_items;
    void *p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, sizeof(int64_t) * ((size_t)n_users + 1), s);
    if (e != cudaSuccess) return set_error(CCO_E_OOM, "cudaMallocAsync row_ptr: %s", cudaGetErrorString(e));
    d->rp[t] = (long long *)p;
    d->rp_alloc[t] = p;
    e = cudaMallocAsync(&p, sizeof(int32_t) * (size_t)std::max<unsigned long long>(kept, 4), s);
    if (e != cudaSuccess) return set_error(CCO_E_OOM, "cudaMallocAsync col_idx: %s", cudaGetErrorString(e));
    d->col[t] = (int32_t *)p;
    d->col_alloc[t] = p;
    CK(cudaEventCreateWithFlags(&d->ready[t], cudaEventDisableTiming));
    long long n_unique = 0;
    if (kept > 0) {
      int row_bits = 1;
      while ((1LL << row_bits) < (long long)n_users) ++row_bits;
      cub::DoubleBuffer<unsigned long long> db(k0, k1);
      size_t tb = 0;
      // dropped events carry the key ~0 and sort to the end: all 64 bits take part
      CK(cub::DeviceRadixSort::SortKeys(nullptr, tb, db, (long long)ne, 0, 64, s));
      void *tmp;
      CKR(ar.alloc((char **)&tmp, tb));
      CK(cub::DeviceRadixSort::SortKeys(tmp, tb, db, (long long)ne, 0, 64, s));
      ar.release(tmp);
      unsigned long long *sorted = db.Current(), *other = db.Alternate();
      uint32_t *flag, *pos;
      CKR(ar.alloc(&flag, kept + 1));
      CKR(ar.alloc(&pos, kept + 1));
      CK(cudaMemsetAsync(flag + kept, 0, 4, s));
      k_unique_flags<<<grid_for((long long)kept, 256, c->sm_count), 256, 0, s>>>((long long)kept, sorted, flag);
      CKR(exclusive_sum_u32(c, ar, flag, pos, (long long)kept + 1));
      uint32_t nuq = 0;
      CKR(mail_fetch(c, &nuq, pos + kept, 4));
      k_unique_scatter<<<grid_for((long long)kept, 256, c->sm_count), 256, 0, s>>>((long long)kept, sorted, flag, pos, other, d->col[t]);
      CKR(mail_wait(c));
      n_unique = nuq;
      k_rowptr_from_keys<<<grid_for((long long)n_users + 1, 256, c->sm_count), 256, 0, s>>>((long long)n_users, n_unique, other, d->rp[t]);
      c->launches += 3;
      ar.release(flag);
      ar.release(pos);
    } else {
      CK(cudaMemsetAsync(d->rp[t], 0, sizeof(int64_t) * ((size_t)n_users + 1), s));
    }
    d->nnz[t] = n_unique;
    CK(cudaEventRecord(d->ready[t], s));
    ar.release(k0);
    ar.release(k1);
    ar.release(iflag);
    ar.release(ipos);
    ar.release(d_item_map);
  }
  // every rank of a multi-GPU job builds the whole matrices (the events are all here) and then works on its block of
  // users like an uploaded dataset does; the block sizes (padding of the column-block all-gather) come from row_ptr
  long long u_lo, u_hi;
  user_block(n_users, c->world, c->rank, &u_lo, &u_hi);
  d->row_base = u_lo;
  d->n_local = u_hi - u_lo;
  std::vector<std::vector<long long>> edge(n_types, std::vector<long long>((size_t)c->world + 1, 0));
  for (int t = 0; t < n_types; ++t)
    for (int q = 0; q <= c->world; ++q) {
      long long a0, a1;
      user_block(n_users, c->world, std::min(q, c->world - 1), &a0, &a1);
      CKR(mail_fetch(c, &edge[t][q], d->rp[t] + (q < c->world ? a0 : a1), 8));
    }
  CKR(mail_wait(c));
  for (int t = 0; t < n_types; ++t) {
    for (int q = 0; q < c->world; ++q) d->block_cap[t] = std::max(d->block_cap[t], edge[t][q + 1] - edge[t][q]);
    d->q_lo[t] = edge[t][c->rank];
    d->q_hi[t] = edge[t][c->rank + 1];
    d->rp[t] += u_lo;   // views of the block; rp_alloc / col_alloc keep the whole matrices
  }
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  g.ok = true;
  *out = d;
  return CCO_OK;
}

int cco_ingest(cco_ctx_t *c, int32_t n_types, const cco_events_t *ev, int64_t n_users_raw, int32_t min_events_per_user,
               int32_t *user_map, int32_t *const *item_maps, cco_dataset_t **out) {
  if (!c || !ev || !user_map || !item_maps || !out || n_types < 1) return set_error(CCO_E_INVALID_ARG, "bad argument");
  if (n_users_raw < 0 || n_users_raw >= 0x7fffffffLL) return set_error(CCO_E_INVALID_ARG, "n_users_raw out of range");
  IngestSource src;
  src.n_types = n_types;
  src.n_users_raw = n_users_raw;
  for (int t = 0; t < n_types; ++t) {
    if (ev[t].n_events < 0 || ev[t].n_events >= 0xffffffffLL || ev[t].n_items_raw < 0)
      return set_error(CCO_E_INVALID_ARG, "type %d: bad event count / item space", t);
    if (ev[t].n_events > 0 && (!ev[t].user || !ev[t].item)) return set_error(CCO_E_INVALID_ARG, "type %d: null event arrays", t);
    if (!item_maps[t] && ev[t].n_items_raw > 0) return set_error(CCO_E_INVALID_ARG, "type %d: null item_map", t);
    // ids are range-checked on the host: they index device arrays
    for (int64_t i = 0; i < ev[t].n_events; ++i)
      if (ev[t].user[i] < 0 || ev[t].user[i] >= n_users_raw || ev[t].item[i] < 0 || ev[t].item[i] >= ev[t].n_items_raw)
        return set_error(CCO_E_INVALID_ARG, "type %d: user or item id out of range at event %lld", t, (long long)i);
    src.n_events.push_back(ev[t].n_events);
    src.n_items_raw.push_back(ev[t].n_items_raw);
  }
  cudaStream_t s = c->stream;
  src.fill = [&](int t, long long *d_user, int32_t *d_item) -> int {
    CK(cudaMemcpyAsync(d_user, ev[t].user, sizeof(int64_t) * (size_t)ev[t].n_events, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_item, ev[t].item, sizeof(int32_t) * (size_t)ev[t].n_events, cudaMemcpyHostToDevice, s));
    return CCO_OK;
  };
  return ingest_core(c, src, min_events_per_user, user_map, item_maps, out);
}

// The synthetic workload of bench.py / the tests (SURVEY.md 8d spec; synth.py holds the numpy twin of the stream):
// event e of a type draws  h1 = mix64(mix64(seed) + (e + 1) * golden), h2 = mix64(h1 ^ 0x6a09e667f3bcc909);
// user = user_perm[upper_bound(user_cdf, u01(h1))], item = item_perm[upper_bound(item_cdf, u01(h2))]; the events are
// generated straight into HBM and go through the same ingest as cco_ingest.
int cco_synth_ingest(cco_ctx_t *c, int32_t n_types, const cco_synth_type_t *types, int64_t n_users_raw, const double *user_cdf,
                     const int32_t *user_perm, int32_t min_events_per_user, int32_t keep_item_space, cco_dataset_t **out) {
  if (!c || !types || !out || n_types < 1 || !user_cdf || !user_perm) return set_error(CCO_E_INVALID_ARG, "bad argument");
  if (n_users_raw < 1 || n_users_raw >= 0x7fffffffLL) return set_error(CCO_E_INVALID_ARG, "n_users_raw out of range");
  IngestSource src;
  src.n_types = n_types;
  src.n_users_raw = n_users_raw;
  src.keep_item_space = keep_item_space != 0;
  for (int t = 0; t < n_types; ++t) {
    if (types[t].n_events < 0 || types[t].n_events >= 0xffffffffLL || types[t].n_items < 1 || !types[t].item_cdf || !types[t].item_perm)
      return set_error(CCO_E_INVALID_ARG, "type %d: bad generator spec", t);
    src.n_events.push_back(types[t].n_events);
    src.n_items_raw.push_back(types[t].n_items);
  }
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  double *d_ucdf = nullptr, *d_icdf = nullptr;
  int32_t *d_uperm = nullptr, *d_iperm = nullptr;
  int32_t max_items = 1;
  for (int t = 0; t < n_types; ++t) max_items = std::max(max_items, types[t].n_items);
  auto drop = [&]() {
    for (void *p : {(void *)d_ucdf, (void *)d_icdf, (void *)d_uperm, (void *)d_iperm})
      if (p) cudaFreeAsync(p, s);
  };
  auto up = [&]() -> int {
    CK(cudaMallocAsync((void **)&d_ucdf, sizeof(double) * (size_t)n_users_raw, s));
    CK(cudaMallocAsync((void **)&d_uperm, sizeof(int32_t) * (size_t)n_users_raw, s));
    CK(cudaMallocAsync((void **)&d_icdf, sizeof(double) * (size_t)max_items, s));
    CK(cudaMallocAsync((void **)&d_iperm, sizeof(int32_t) * (size_t)max_items, s));
    CK(cudaMemcpyAsync(d_ucdf, user_cdf, sizeof(double) * (size_t)n_users_raw, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_uperm, user_perm, sizeof(int32_t) * (size_t)n_users_raw, cudaMemcpyHostToDevice, s));
    return CCO_OK;
  };
  int rc = up();
  if (rc != CCO_OK) { drop(); return rc; }
  src.fill = [&](int t, long long *d_user, int32_t *d_item) -> int {
    CK(cudaMemcpyAsync(d_icdf, types[t].item_cdf, sizeof(double) * (size_t)types[t].n_items, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_iperm, types[t].item_perm, sizeof(int32_t) * (size_t)types[t].n_items, cudaMemcpyHostToDevice, s));
    k_synth_events<<<grid_for(types[t].n_events, 256, c->sm_count), 256, 0, s>>>(types[t].n_events, types[t].seed, d_ucdf, d_uperm,
                                                                                (int32_t)n_users_raw, d_icdf, d_iperm, types[t].n_items,
                                                                                d_user, d_item);
    c->launches++;
    CK(cudaGetLastError());
    return CCO_OK;
  };
  rc = ingest_core(c, src, min_events_per_user, nullptr, nullptr, out);
  drop();
  return rc;
}

// ---- SURVEY.md 8f-1 from raw id strings (kernels in cco_strings.cuh) ---------------------------------------------------
// The strings are turned into raw integer ids whose ascending order is the dictionary order (primary users by first
// appearance, items by first appearance among surviving events); ingest_core then builds the matrices exactly as for
// cco_ingest.
namespace cco {
struct MaxU32 {
  __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};
static int inclusive_max_u32(cco_ctx *c, Arena &ar, const uint32_t *in, uint32_t *out, unsigned long long n) {
  size_t tb = 0;
  CK(cub::DeviceScan::InclusiveScan(nullptr, tb, in, out, MaxU32(), (long long)n, c->stream));
  void *tmp;
  CKR(ar.alloc((char **)&tmp, tb));
  CK(cub::DeviceScan::InclusiveScan(tmp, tb, in, out, MaxU32(), (long long)n, c->stream));
  ar.release(tmp);
  return CCO_OK;
}

// rep[i] = the smallest j < n with bytes(j) == bytes(i), n < 2^32.  Sorting by a 48-bit hash brings equal ids together;
// each id is compared with the first id of its equal-hash run, and the few that differ from it (hash collisions) are
// grouped by an exact sort on (hash, bytes, index).  A collision costs time, never a merge of two different ids.
static int group_ids(cco_ctx *c, Arena &ar, unsigned long long n, const StrCols &cols, bool short_hash, uint32_t *rep) {
  if (n == 0) return CCO_OK;
  cudaStream_t s = c->stream;
  const int bits = short_hash ? 2 : 48;
  const int G = grid_for((long long)n, 256, c->sm_count);
  unsigned long long *h, *hs, *n_un;
  uint32_t *idx, *is, *head, *run, *un;
  CKR(ar.alloc(&h, n));
  CKR(ar.alloc(&hs, n));
  CKR(ar.alloc(&idx, n));
  CKR(ar.alloc(&is, n));
  CKR(ar.alloc(&head, n));
  CKR(ar.alloc(&run, n));
  CKR(ar.alloc(&un, n));
  CKR(ar.alloc(&n_un, 1));
  k_ingest_str_hash<<<G, 256, 0, s>>>(n, cols, (1ULL << bits) - 1, h, idx);
  size_t tb = 0;
  CK(cub::DeviceRadixSort::SortPairs(nullptr, tb, h, hs, idx, is, (long long)n, 0, bits, s));
  void *tmp;
  CKR(ar.alloc((char **)&tmp, tb));
  CK(cub::DeviceRadixSort::SortPairs(tmp, tb, h, hs, idx, is, (long long)n, 0, bits, s));
  ar.release(tmp);
  k_ingest_str_run_heads<<<G, 256, 0, s>>>(n, hs, head);
  CKR(inclusive_max_u32(c, ar, head, run, n));
  CK(cudaMemsetAsync(n_un, 0, 8, s));
  k_ingest_str_resolve<<<G, 256, 0, s>>>(n, cols, is, run, rep, un, n_un);
  c->launches += 3;
  unsigned long long nu = 0;
  CKR(mail_fetch(c, &nu, n_un, 8));
  CKR(mail_wait(c));
  if (nu > 0) {
    const StrLess less{cols, h};
    tb = 0;
    CK(cub::DeviceMergeSort::SortKeys(nullptr, tb, un, (long long)nu, less, s));
    CKR(ar.alloc((char **)&tmp, tb));
    CK(cub::DeviceMergeSort::SortKeys(tmp, tb, un, (long long)nu, less, s));
    ar.release(tmp);
    const int g = grid_for((long long)nu, 256, c->sm_count);
    k_ingest_str_class_heads<<<g, 256, 0, s>>>(nu, cols, un, h, head);
    CKR(inclusive_max_u32(c, ar, head, run, nu));
    k_ingest_str_class_rep<<<g, 256, 0, s>>>(nu, un, run, rep);
    c->launches += 2;
  }
  for (void *p : {(void *)h, (void *)hs, (void *)idx, (void *)is, (void *)head, (void *)run, (void *)un, (void *)n_un}) ar.release(p);
  return CCO_OK;
}

struct DevCol {
  long long n = 0;
  long long *off = nullptr;
  unsigned char *bytes = nullptr;
};
static StrCols one_column(const DevCol &d) {
  StrCols s;
  s.n_a = d.n;
  s.off_a = d.off;
  s.bytes_a = d.bytes;
  return s;
}

// the ids src[0 .. n) of `cols`, in that order, as a compact device dictionary and, unless host is null, as a copy in pinned
// host memory (offsets and bytes, appended to `held`; the copy is complete at the next synchronisation of the stream)
static int gather_dict(cco_ctx *c, Arena &ar, const StrCols &cols, const uint32_t *src, long long n, DevCol *dev, cco_dictionary_t *host,
                       std::vector<void *> &held) {
  cudaStream_t s = c->stream;
  long long *len, *off;
  CKR(ar.alloc(&len, n + 1));
  CKR(ar.alloc(&off, n + 1));
  CK(cudaMemsetAsync(len + n, 0, 8, s));
  if (n > 0) {
    k_ingest_str_lengths<<<grid_for(n, 256, c->sm_count), 256, 0, s>>>(n, cols, src, len);
    c->launches++;
  }
  CKR(exclusive_sum_i64(c, ar, len, off, n + 1));
  long long total = 0;
  CKR(mail_fetch(c, &total, off + n, 8));
  CKR(mail_wait(c));
  unsigned char *bytes;
  CKR(ar.alloc(&bytes, std::max<long long>(total, 1)));
  if (total > 0) {
    k_ingest_str_gather<<<grid_for(n, 256, c->sm_count), 256, 0, s>>>(n, cols, src, off, bytes);
    c->launches++;
  }
  ar.release(len);
  dev->n = n;
  dev->off = off;
  dev->bytes = bytes;
  if (!host) return CCO_OK;
  int64_t *ho = (int64_t *)c->pinned_get(sizeof(int64_t) * ((size_t)n + 1), /*for_result=*/false);
  if (!ho) return set_error(CCO_E_OOM, "pinned host allocation failed");
  held.push_back(ho);
  char *hb = (char *)c->pinned_get((size_t)std::max<long long>(total, 1), /*for_result=*/false);
  if (!hb) return set_error(CCO_E_OOM, "pinned host allocation failed");
  held.push_back(hb);
  CK(cudaMemcpyAsync(ho, off, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyDeviceToHost, s));
  if (total > 0) CK(cudaMemcpyAsync(hb, bytes, (size_t)total, cudaMemcpyDeviceToHost, s));
  host->n = n;
  host->offsets = ho;
  host->bytes = hb;
  return CCO_OK;
}
}  // namespace cco

int cco_ingest_strings(cco_ctx_t *c, int32_t n_types, const cco_string_events_t *ev, int32_t min_events_per_user, uint32_t flags,
                       cco_dictionary_t *user_dict, cco_dictionary_t *item_dicts, cco_dataset_t **out) {
  if (!c || !ev || !user_dict || !item_dicts || !out || n_types < 1) return set_error(CCO_E_INVALID_ARG, "null argument or n_types < 1");
  *out = nullptr;
  if (!c->members.empty()) return set_error(CCO_E_UNSUPPORTED, "cco_ingest_strings needs a single-GPU context, not a group context");
  const char *const which[2] = {"user", "item"};
  for (int t = 0; t < n_types; ++t) {
    if (ev[t].user.n != ev[t].item.n)
      return set_error(CCO_E_INVALID_ARG, "type %d: %lld user ids but %lld item ids", t, (long long)ev[t].user.n, (long long)ev[t].item.n);
    const long long n = ev[t].user.n;
    if (n < 0 || n >= (1LL << 32)) return set_error(CCO_E_INVALID_ARG, "type %d: %lld events (at most 2^32 - 1 per type)", t, n);
    for (int w = 0; w < 2; ++w) {
      const cco_dictionary_t &d = w ? ev[t].item : ev[t].user;
      if (!d.offsets) return set_error(CCO_E_INVALID_ARG, "type %d: null %s offsets", t, which[w]);
      if (d.offsets[0] != 0) return set_error(CCO_E_INVALID_ARG, "type %d: %s offsets[0] != 0", t, which[w]);
      if (d.offsets[n] < 0) return set_error(CCO_E_INVALID_ARG, "type %d: %s offsets decrease", t, which[w]);
      if (d.offsets[n] > 0 && !d.bytes) return set_error(CCO_E_INVALID_ARG, "type %d: null %s bytes", t, which[w]);
    }
  }
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  nvtx_push("cco:ingest_strings");
  struct Pop { ~Pop() { nvtx_pop(); } } pop;
  mail_reset(c);
  Arena ar(s);
  const bool sh = (flags & CCO_FLAG_INGEST_SHORT_HASH) != 0;
  // pinned dictionary copies: handed to the caller on success, returned to the pool otherwise
  struct Held {
    cco_ctx *c;
    std::vector<void *> p;
    bool ok = false;
    ~Held() {
      if (!ok)
        for (void *q : p) c->pinned_put(q);
    }
  } held{c};
  // offsets first: no byte is read before every column's offsets are known not to decrease
  std::vector<DevCol> col(2 * (size_t)n_types);
  int *bad;
  CKR(ar.alloc(&bad, 1));
  CK(cudaMemsetAsync(bad, 0x7f, sizeof(int), s));
  for (int t = 0; t < n_types; ++t)
    for (int w = 0; w < 2; ++w) {
      const cco_dictionary_t &d = w ? ev[t].item : ev[t].user;
      DevCol &dc = col[2 * t + w];
      dc.n = d.n;
      CKR(ar.alloc(&dc.off, d.n + 1));
      CK(cudaMemcpyAsync(dc.off, d.offsets, sizeof(int64_t) * ((size_t)d.n + 1), cudaMemcpyHostToDevice, s));
      if (d.n > 0) {
        k_ingest_str_check_offsets<<<grid_for(d.n, 256, c->sm_count), 256, 0, s>>>(d.n, dc.off, 2 * t + w, bad);
        c->launches++;
      }
    }
  int first_bad = 0;
  CKR(mail_fetch(c, &first_bad, bad, sizeof(int)));
  CKR(mail_wait(c));
  if (first_bad != 0x7f7f7f7f) return set_error(CCO_E_INVALID_ARG, "type %d: %s offsets decrease", first_bad / 2, which[first_bad & 1]);
  for (int t = 0; t < n_types; ++t)
    for (int w = 0; w < 2; ++w) {
      const cco_dictionary_t &d = w ? ev[t].item : ev[t].user;
      DevCol &dc = col[2 * t + w];
      const long long nb = d.offsets[d.n];
      CKR(ar.alloc(&dc.bytes, std::max<long long>(nb, 1)));
      if (nb > 0) CK(cudaMemcpyAsync(dc.bytes, d.bytes, (size_t)nb, cudaMemcpyHostToDevice, s));
    }

  // users of the primary type: group, count, rank by first appearance
  std::vector<cco_dictionary_t> host(1 + (size_t)n_types);
  std::vector<long long *> uraw(n_types, nullptr);
  std::vector<uint32_t *> surv(n_types, nullptr);
  std::vector<int32_t *> iraw(n_types, nullptr);
  std::vector<int32_t> n_items(n_types, 0);
  const long long n0 = col[0].n;
  const StrCols u0 = one_column(col[0]);
  uint32_t *rep0, *cnt, *first, *kept, *fpos, *kpos;
  CKR(ar.alloc(&rep0, n0));
  CKR(ar.alloc(&cnt, n0));
  CKR(ar.alloc(&first, n0 + 1));
  CKR(ar.alloc(&kept, n0 + 1));
  CKR(ar.alloc(&fpos, n0 + 1));
  CKR(ar.alloc(&kpos, n0 + 1));
  CKR(group_ids(c, ar, n0, u0, sh, rep0));
  CK(cudaMemsetAsync(cnt, 0, sizeof(uint32_t) * (size_t)std::max<long long>(n0, 1), s));
  CK(cudaMemsetAsync(first + n0, 0, sizeof(uint32_t), s));
  CK(cudaMemsetAsync(kept + n0, 0, sizeof(uint32_t), s));
  const uint32_t need = min_events_per_user > 1 ? (uint32_t)min_events_per_user : 1u;
  if (n0 > 0) {
    const int G = grid_for(n0, 256, c->sm_count);
    k_ingest_str_user_count<<<G, 256, 0, s>>>(n0, rep0, cnt);
    k_ingest_str_user_flags<<<G, 256, 0, s>>>(n0, rep0, cnt, need, first, kept);
    c->launches += 2;
  }
  CKR(exclusive_sum_u32(c, ar, first, fpos, n0 + 1));
  CKR(exclusive_sum_u32(c, ar, kept, kpos, n0 + 1));
  uint32_t n_primary = 0, n_users = 0;
  CKR(mail_fetch(c, &n_primary, fpos + n0, 4));
  CKR(mail_fetch(c, &n_users, kpos + n0, 4));
  CKR(mail_wait(c));
  if (n_primary > 0x7ffffffeu) return set_error(CCO_E_UNSUPPORTED, "%u distinct primary users (at most 2^31 - 2)", n_primary);
  uint32_t *dict_ev, *dict_raw;
  CKR(ar.alloc(&dict_ev, n_users));
  CKR(ar.alloc(&dict_raw, n_users));
  CKR(ar.alloc(&uraw[0], n0));
  CKR(ar.alloc(&surv[0], n0));
  if (n0 > 0) {
    k_ingest_str_user_tokens<<<grid_for(n0, 256, c->sm_count), 256, 0, s>>>(n0, rep0, fpos, kept, kpos, uraw[0], surv[0], dict_ev, dict_raw);
    c->launches++;
  }
  DevCol udict;
  CKR(gather_dict(c, ar, u0, dict_ev, n_users, &udict, &host[0], held.p));
  for (void *p : {(void *)rep0, (void *)cnt, (void *)first, (void *)kept, (void *)fpos, (void *)kpos, (void *)dict_ev}) ar.release(p);

  // users of the other types: grouped together with the user dictionary (elements [0, n_users)), in chunks that keep
  // the element count below 2^32
  for (int t = 1; t < n_types; ++t) {
    const long long n = col[2 * t].n;
    CKR(ar.alloc(&uraw[t], n));
    CKR(ar.alloc(&surv[t], n));
    const long long kChunk = 1LL << 31;
    for (long long c0 = 0; c0 < n; c0 += kChunk) {
      const long long m = std::min(kChunk, n - c0);
      StrCols sc = one_column(udict);
      sc.off_b = col[2 * t].off + c0;
      sc.bytes_b = col[2 * t].bytes;
      uint32_t *rep;
      CKR(ar.alloc(&rep, n_users + m));
      CKR(group_ids(c, ar, n_users + m, sc, sh, rep));
      k_ingest_str_match_users<<<grid_for(m, 256, c->sm_count), 256, 0, s>>>(m, n_users, rep, dict_raw, n_primary, uraw[t] + c0,
                                                                            surv[t] + c0);
      c->launches++;
      ar.release(rep);
    }
  }

  // items of every type: group, rank by first surviving appearance
  for (int t = 0; t < n_types; ++t) {
    const DevCol &ic = col[2 * t + 1];
    const long long n = ic.n;
    const StrCols cols = one_column(ic);
    uint32_t *rep, *fs, *flag, *ipos;
    CKR(ar.alloc(&iraw[t], n));
    CKR(ar.alloc(&rep, n));
    CKR(ar.alloc(&fs, n));
    CKR(ar.alloc(&flag, n + 1));
    CKR(ar.alloc(&ipos, n + 1));
    CKR(group_ids(c, ar, n, cols, sh, rep));
    CK(cudaMemsetAsync(fs, 0xff, sizeof(uint32_t) * (size_t)std::max<long long>(n, 1), s));
    CK(cudaMemsetAsync(flag + n, 0, sizeof(uint32_t), s));
    if (n > 0) {
      const int G = grid_for(n, 256, c->sm_count);
      k_ingest_str_first_surv<<<G, 256, 0, s>>>(n, rep, surv[t], fs);
      k_ingest_str_item_flags<<<G, 256, 0, s>>>(n, rep, fs, flag);
      c->launches += 2;
    }
    CKR(exclusive_sum_u32(c, ar, flag, ipos, n + 1));
    uint32_t q = 0;
    CKR(mail_fetch(c, &q, ipos + n, 4));
    CKR(mail_wait(c));
    if (q > 0x7ffffffeu) return set_error(CCO_E_UNSUPPORTED, "type %d: %u distinct items (at most 2^31 - 2)", t, q);
    n_items[t] = (int32_t)q;
    uint32_t *idict;
    CKR(ar.alloc(&idict, q));
    if (n > 0) {
      k_ingest_str_item_tokens<<<grid_for(n, 256, c->sm_count), 256, 0, s>>>(n, rep, surv[t], fs, flag, ipos, iraw[t], idict);
      c->launches++;
    }
    DevCol idev;
    CKR(gather_dict(c, ar, cols, idict, q, &idev, &host[1 + t], held.p));
    for (void *p : {(void *)rep, (void *)fs, (void *)flag, (void *)ipos, (void *)idict, (void *)ic.off, (void *)ic.bytes}) ar.release(p);
  }

  // the matrices: raw user id n_primary has no primary event, so the users unknown to the dictionary drop out there
  IngestSource src;
  src.n_types = n_types;
  src.n_users_raw = (long long)n_primary + 1;
  for (int t = 0; t < n_types; ++t) {
    src.n_events.push_back(col[2 * t].n);
    src.n_items_raw.push_back(n_items[t]);
  }
  src.fill = [&](int t, long long *d_user, int32_t *d_item) -> int {
    const size_t n = (size_t)col[2 * t].n;
    CK(cudaMemcpyAsync(d_user, uraw[t], sizeof(int64_t) * n, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemcpyAsync(d_item, iraw[t], sizeof(int32_t) * n, cudaMemcpyDeviceToDevice, s));
    return CCO_OK;
  };
  cco_dataset *d = nullptr;
  CKR(ingest_core(c, src, min_events_per_user, nullptr, nullptr, &d));   // ends in a stream synchronise: the dictionaries are home
  held.ok = true;
  *user_dict = host[0];
  for (int t = 0; t < n_types; ++t) item_dicts[t] = host[1 + t];
  *out = d;
  return CCO_OK;
}

// copy matrix i of a resident dataset into caller-provided host arrays (pinned ones from cco_host_alloc copy at PCIe speed)
int cco_dataset_copy_to_host(const cco_dataset_t *ds, int32_t i, int64_t *row_ptr, int32_t *col_idx) {
  if (!ds || !row_ptr || i < 0 || i >= ds->n_mats) return set_error(CCO_E_INVALID_ARG, "bad argument");
  if (ds->nnz[i] > 0 && !col_idx) return set_error(CCO_E_INVALID_ARG, "null col_idx");
  if (!ds->whole) return set_error(CCO_E_UNSUPPORTED, "this dataset holds one rank's block of users only");
  cco_ctx *c = ds->ctx;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->copy_stream));
  CK(cudaMemcpyAsync(row_ptr, ds->rp_alloc[i], sizeof(int64_t) * ((size_t)ds->n_users + 1), cudaMemcpyDeviceToHost, c->stream));
  if (ds->nnz[i] > 0)
    CK(cudaMemcpyAsync(col_idx, ds->col_alloc[i], sizeof(int32_t) * (size_t)ds->nnz[i], cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return CCO_OK;
}

int cco_partition_rows(const int64_t *work_prefix, int32_t n_items, int32_t world_size, int32_t *bounds) {
  if (!work_prefix || !bounds || n_items < 0 || world_size < 1) return set_error(CCO_E_INVALID_ARG, "bad argument");
  // weight of row i = its products + 1 (so rows without work are spread too); contiguous ranges of equal weight
  const long long total = (long long)work_prefix[n_items] + n_items;
  for (int r = 0; r <= world_size; ++r) {
    if (r == 0) { bounds[r] = 0; continue; }
    if (r == world_size) { bounds[r] = n_items; continue; }
    const long long target = (long long)((__int128)total * r / world_size);
    int lo = 0, hi = n_items;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if ((long long)work_prefix[mid] + mid < target) lo = mid + 1; else hi = mid;
    }
    bounds[r] = lo;
  }
  return CCO_OK;
}

int cco_dataset_upload(cco_ctx_t *ctx, int32_t n_mats, const cco_csr_t *mats, uint32_t flags, cco_dataset_t **out) {
  if (!ctx || !out) return set_error(CCO_E_INVALID_ARG, "null argument");
  if (!ctx->members.empty()) return set_error(CCO_E_UNSUPPORTED, "resident datasets are per GPU: use cco_train on a group context");
  *out = nullptr;
  std::vector<cco_indicator_params_t> p(std::max(n_mats, 1), cco_indicator_params_t{1, 1, 0, 0.0});
  CKR(validate_host(n_mats, mats, p.data()));
  return dataset_upload(ctx, n_mats, mats, flags, out);
}
int cco_dataset_free(cco_dataset_t *ds) {
  dataset_release(ds);
  return CCO_OK;
}
int cco_train_dataset(cco_ctx_t *ctx, const cco_dataset_t *ds, const cco_indicator_params_t *params, int32_t seed,
                      uint32_t flags, cco_result_t **out) {
  if (!ctx || !ds || !params || !out) return set_error(CCO_E_INVALID_ARG, "null argument");
  if (ds->ctx != ctx) return set_error(CCO_E_INVALID_ARG, "dataset belongs to another context");
  *out = nullptr;
  for (int i = 0; i < ds->n_mats; ++i) {
    if (params[i].max_interactions < 1) return set_error(CCO_E_INVALID_ARG, "matrix %d: max_interactions must be >= 1", i);
    if (params[i].top_k < 1) return set_error(CCO_E_INVALID_ARG, "matrix %d: top_k must be >= 1", i);
    if (params[i].top_k > CCO_MAX_TOP_K)
      return set_error(CCO_E_UNSUPPORTED, "matrix %d: top_k %d > CCO_MAX_TOP_K (%d)", i, params[i].top_k, CCO_MAX_TOP_K);
  }
  ctx->launches = 0;
  return train_dataset(ctx, ds, params, seed, flags, out);
}
int cco_timer_start(cco_ctx_t *ctx) {
  if (!ctx) return set_error(CCO_E_INVALID_ARG, "null context");
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventRecord(ctx->tev[0], ctx->stream));
  return CCO_OK;
}
int cco_timer_stop(cco_ctx_t *ctx, float *ms) {
  if (!ctx || !ms) return set_error(CCO_E_INVALID_ARG, "null argument");
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventRecord(ctx->tev[1], ctx->stream));
  CK(cudaEventSynchronize(ctx->tev[1]));
  CK(cudaEventElapsedTime(ms, ctx->tev[0], ctx->tev[1]));
  return CCO_OK;
}

int cco_result_num_matrices(const cco_result_t *r) { return r ? (int)r->mats.size() : set_error(CCO_E_INVALID_ARG, "null result"); }

int cco_result_row_range(const cco_result_t *r, int32_t i, int64_t *row_begin, int64_t *row_end) {
  if (!r || i < 0 || i >= (int)r->mats.size()) return set_error(CCO_E_INVALID_ARG, "bad result/index");
  if (row_begin) *row_begin = r->mats[i].row_begin;
  if (row_end) *row_end = r->mats[i].row_end;
  return CCO_OK;
}

int cco_result_matrix(const cco_result_t *r, int32_t i, int64_t *n_rows, int32_t *n_cols, const int64_t **row_ptr,
                      const int32_t **col_idx, const double **llr, const int32_t **count) {
  if (!r || i < 0 || i >= (int)r->mats.size()) return set_error(CCO_E_INVALID_ARG, "bad result/index");
  const ResultMat &m = r->mats[i];
  if (n_rows) *n_rows = m.row_end - m.row_begin;
  if (n_cols) *n_cols = m.n_cols;
  if (row_ptr) *row_ptr = m.row_ptr;
  if (col_idx) *col_idx = m.col;
  if (llr) *llr = m.llr;
  if (count) *count = m.cnt;
  return CCO_OK;
}

int cco_result_stats(const cco_result_t *r, cco_stats_t *out) {
  if (!r || !out) return set_error(CCO_E_INVALID_ARG, "null argument");
  *out = r->stats;
  return CCO_OK;
}

int cco_result_free(cco_result_t *r) {
  if (!r) return CCO_OK;
  for (auto &m : r->mats) {
    for (void *p : {(void *)m.row_ptr, (void *)m.col, (void *)m.llr, (void *)m.cnt})
      if (p) r->ctx->pinned_put(p);
  }
  delete r;
  return CCO_OK;
}

// ---- SURVEY.md 8f-2: indicator model -> Elasticsearch bulk body (cco_format.cuh) --------------------------------------
namespace cco {
static int upload_dict(cco_ctx *c, Arena &ar, const cco_dictionary_t &d, DevDict *raw) {
  if (d.n < 0 || (d.n > 0 && (!d.offsets || (d.offsets[d.n] > 0 && !d.bytes)))) return set_error(CCO_E_INVALID_ARG, "bad dictionary");
  long long *off;
  unsigned char *bytes;
  const long long nb = d.n > 0 ? d.offsets[d.n] : 0;
  CKR(ar.alloc(&off, d.n + 1));
  CKR(ar.alloc(&bytes, std::max<long long>(nb, 1)));
  if (d.n > 0) {
    CK(cudaMemcpyAsync(off, d.offsets, sizeof(int64_t) * ((size_t)d.n + 1), cudaMemcpyHostToDevice, c->stream));
    if (nb > 0) CK(cudaMemcpyAsync(bytes, d.bytes, (size_t)nb, cudaMemcpyHostToDevice, c->stream));
  } else {
    CK(cudaMemsetAsync(off, 0, 8, c->stream));
  }
  raw->off = off;
  raw->bytes = bytes;
  raw->n = d.n;
  return CCO_OK;
}
// JSON-escape every string of a device dictionary (two passes: lengths, scan, bytes)
static int escape_dict(cco_ctx *c, Arena &ar, const DevDict &raw, DevDict *esc) {
  long long *len, *off;
  CKR(ar.alloc(&len, raw.n + 1));
  CKR(ar.alloc(&off, raw.n + 1));
  CK(cudaMemsetAsync(len + raw.n, 0, 8, c->stream));
  if (raw.n > 0) {
    k_escape_len<<<grid_for(raw.n, 256, c->sm_count), 256, 0, c->stream>>>(raw.n, raw.off, raw.bytes, len);
    c->launches++;
  }
  CKR(exclusive_sum_i64(c, ar, len, off, raw.n + 1));
  long long total = 0;
  CK(cudaMemcpyAsync(&total, off + raw.n, 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  unsigned char *bytes;
  CKR(ar.alloc(&bytes, std::max<long long>(total, 1)));
  if (raw.n > 0) {
    k_escape_write<<<grid_for(raw.n, 256, c->sm_count), 256, 0, c->stream>>>(raw.n, raw.off, raw.bytes, off, bytes);
    c->launches++;
  }
  esc->off = off;
  esc->bytes = bytes;
  esc->n = raw.n;
  ar.release(len);
  return CCO_OK;
}

// the argument checks cco_format_es_bulk and cco_format_model_bulk share
static int check_indicators(const cco_result_t *res, int32_t n_names, const char *const *names, const cco_dictionary_t *col_ids) {
  const int n_ind = (int)res->mats.size();
  if (n_names != n_ind) return set_error(CCO_E_INVALID_ARG, "%d event names for %d indicators", n_names, n_ind);
  if (n_ind < 1 || n_ind > kMaxFormatIndicators) return set_error(CCO_E_UNSUPPORTED, "1..%d indicators", kMaxFormatIndicators);
  const int64_t row_lo = res->mats[0].row_begin, row_hi = res->mats[0].row_end;
  for (int i = 0; i < n_ind; ++i) {
    const ResultMat &m = res->mats[i];
    if (m.row_begin != row_lo || m.row_end != row_hi) return set_error(CCO_E_INVALID_ARG, "indicators cover different row ranges");
    if (!m.row_ptr || (m.row_ptr[row_hi - row_lo] > 0 && !m.col)) return set_error(CCO_E_INVALID_ARG, "indicator %d has no column array on the host", i);
    if (col_ids[i].n < m.n_cols) return set_error(CCO_E_INVALID_ARG, "column dictionary %d has %lld ids for %d columns", i, (long long)col_ids[i].n, m.n_cols);
    if (!names[i]) return set_error(CCO_E_INVALID_ARG, "null event name");
  }
  return CCO_OK;
}

// n C strings as one escaped blob on the device: string i = bytes[off[i] .. off[i + 1])
static int escape_names(cco_ctx *c, Arena &ar, int n, const char *const *names, const unsigned char **bytes, int32_t *off) {
  std::vector<int64_t> noff(n + 1, 0);
  std::string blob;
  for (int i = 0; i < n; ++i) {
    blob += names[i];
    noff[i + 1] = (int64_t)blob.size();
  }
  cco_dictionary_t nd = {n, noff.data(), blob.data()};
  DevDict nraw, nesc;
  CKR(upload_dict(c, ar, nd, &nraw));
  CK(cudaStreamSynchronize(c->stream));   // noff / blob are locals
  CKR(escape_dict(c, ar, nraw, &nesc));
  std::vector<long long> eoff(n + 1);
  CK(cudaMemcpyAsync(eoff.data(), nesc.off, sizeof(long long) * ((size_t)n + 1), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  *bytes = nesc.bytes;
  for (int i = 0; i <= n; ++i) off[i] = (int32_t)eoff[i];
  return CCO_OK;
}

// the indicator part of FormatArgs on the device: event names and column dictionaries escaped, the rows of every indicator
static int upload_indicators(cco_ctx *c, Arena &ar, const cco_result_t *res, const char *const *names, const cco_dictionary_t *col_ids,
                             FormatArgs *fa) {
  cudaStream_t s = c->stream;
  const int n_ind = (int)res->mats.size();
  const int64_t row_lo = res->mats[0].row_begin, row_hi = res->mats[0].row_end;
  fa->n_rows = (int32_t)(row_hi - row_lo);
  fa->row_id_base = row_lo;
  fa->n_ind = n_ind;
  CKR(escape_names(c, ar, n_ind, names, &fa->names, fa->name_off));
  for (int i = 0; i < n_ind; ++i) {
    const ResultMat &m = res->mats[i];
    DevDict raw;
    CKR(upload_dict(c, ar, col_ids[i], &raw));
    CKR(escape_dict(c, ar, raw, &fa->col_ids[i]));
    const long long n_my = row_hi - row_lo, nnz = m.row_ptr[n_my] - m.row_ptr[0];
    long long *d_rp;
    int32_t *d_col;
    CKR(ar.alloc(&d_rp, n_my + 1));
    CKR(ar.alloc(&d_col, std::max<long long>(nnz, 1)));
    CK(cudaMemcpyAsync(d_rp, m.row_ptr, sizeof(int64_t) * ((size_t)n_my + 1), cudaMemcpyHostToDevice, s));
    if (nnz > 0) CK(cudaMemcpyAsync(d_col, m.col + m.row_ptr[0], sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, s));
    if (m.row_ptr[0] != 0) {   // a group member's slice is rebased inside the merged arrays: bring it back to 0
      k_add_i64<<<grid_for(n_my + 1, 256, c->sm_count, 2), 256, 0, s>>>(n_my + 1, -(long long)m.row_ptr[0], d_rp);
      c->launches++;
    }
    fa->row_ptr[i] = d_rp;
    fa->col[i] = d_col;
  }
  return CCO_OK;
}

// lengths of n_docs documents -> exclusive scan -> bytes, copied into pinned memory of `owner` (the caller frees it with
// cco_host_free).  launch_len(doc_len) and launch_write(doc_off, out) enqueue the two kernels.
extern "C++" {   // a template inside the extern "C" block of the entries
template <class Len, class Write>
static int assemble_docs(cco_ctx *owner, cco_ctx *c, Arena &ar, long long n_docs, Len launch_len, Write launch_write, char **out_bytes,
                         int64_t *out_len) {
  cudaStream_t s = c->stream;
  long long *doc_len, *doc_off;
  CKR(ar.alloc(&doc_len, n_docs + 1));
  CKR(ar.alloc(&doc_off, n_docs + 1));
  CK(cudaMemsetAsync(doc_len + n_docs, 0, 8, s));
  if (n_docs > 0) {
    launch_len(doc_len);
    c->launches++;
  }
  CKR(exclusive_sum_i64(c, ar, doc_len, doc_off, n_docs + 1));
  long long total = 0;
  CK(cudaMemcpyAsync(&total, doc_off + n_docs, 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  unsigned char *d_out;
  CKR(ar.alloc(&d_out, std::max<long long>(total, 1)));
  if (n_docs > 0 && total > 0) {
    launch_write(doc_off, d_out);
    c->launches++;
  }
  char *host = (char *)owner->pinned_get((size_t)std::max<long long>(total, 1), /*for_result=*/false);
  if (!host) return set_error(CCO_E_OOM, "pinned host allocation failed");
  if (total > 0) CK(cudaMemcpyAsync(host, d_out, (size_t)total, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  *out_bytes = host;
  *out_len = total;
  return CCO_OK;
}
}  // extern "C++"

// PopModel's bucket edges: Joda's integer millisecond arithmetic over [start_ms, end_ms)
static PopArgs pop_args(int32_t mode, int64_t start_ms, int64_t end_ms, int32_t n_items) {
  PopArgs a;
  memset(&a, 0, sizeof a);
  a.n_items = n_items;
  const long long dur = end_ms - start_ms;
  if (mode == CCO_POP_POPULAR) {
    a.n_buckets = 1;
    a.edge[0] = start_ms;
    a.edge[1] = end_ms;
  } else if (mode == CCO_POP_TRENDING) {   // PopModel.scala:134-138: halfInterval = durationMillis / 2
    a.n_buckets = 2;
    a.edge[0] = start_ms;
    a.edge[1] = start_ms + dur / 2;
    a.edge[2] = end_ms;
  } else {                                  // PopModel.scala:159-164: older = dur / 3, middle = the same length, newer = the rest
    a.n_buckets = 3;
    a.edge[0] = start_ms;
    a.edge[1] = start_ms + dur / 3;
    a.edge[2] = a.edge[1] + dur / 3;
    a.edge[3] = end_ms;
  }
  return a;
}
}  // namespace cco

int cco_format_es_bulk(cco_ctx_t *ctx, const cco_result_t *res, int32_t n_names, const char *const *names,
                       const cco_dictionary_t *row_ids, const cco_dictionary_t *col_ids, char **out_bytes, int64_t *out_len) {
  if (!ctx || !res || !names || !row_ids || !col_ids || !out_bytes || !out_len) return set_error(CCO_E_INVALID_ARG, "null argument");
  CKR(check_indicators(res, n_names, names, col_ids));
  cco_ctx *c = ctx->members.empty() ? ctx : ctx->members[0];   // a group's merged model is formatted on its first GPU
  const int64_t row_hi = res->mats[0].row_end;
  if (row_ids->n < row_hi) return set_error(CCO_E_INVALID_ARG, "row dictionary has %lld ids, rows go up to %lld", (long long)row_ids->n, (long long)row_hi);
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Arena ar(s);
  nvtx_push("cco:format_es_bulk");
  struct Pop { ~Pop() { nvtx_pop(); } } pop;
  FormatArgs fa;
  memset(&fa, 0, sizeof fa);
  DevDict raw;
  CKR(upload_dict(c, ar, *row_ids, &raw));
  CKR(escape_dict(c, ar, raw, &fa.row_ids));
  CKR(upload_indicators(c, ar, res, names, col_ids, &fa));
  return assemble_docs(
      ctx, c, ar, fa.n_rows,
      [&](long long *doc_len) { k_doc_len<<<grid_for(fa.n_rows, 256, c->sm_count), 256, 0, s>>>(fa, doc_len); },
      [&](const long long *doc_off, unsigned char *out) {
        k_doc_write<<<grid_for((long long)fa.n_rows * 32, 256, c->sm_count), 256, 0, s>>>(fa, doc_off, out);
      },
      out_bytes, out_len);
}

// ---- SURVEY.md 8f-3: PopModel rank histograms -------------------------------------------------------------------------
int cco_pop_model(cco_ctx_t *ctx, int32_t mode, int64_t n_events, const int32_t *item, const int64_t *time_ms, int32_t n_items,
                  int64_t start_ms, int64_t end_ms, double *score, unsigned char *present) {
  if (!ctx || n_events < 0 || n_items < 0 || (n_events > 0 && (!item || !time_ms)) || (n_items > 0 && (!score || !present)))
    return set_error(CCO_E_INVALID_ARG, "bad argument");
  if (mode < CCO_POP_POPULAR || mode > CCO_POP_HOT) return set_error(CCO_E_INVALID_ARG, "mode must be CCO_POP_POPULAR, _TRENDING or _HOT");
  if (end_ms < start_ms) return set_error(CCO_E_INVALID_ARG, "end before start (Joda Interval would throw)");
  if (n_items == 0) return CCO_OK;
  cco_ctx *c = ctx->members.empty() ? ctx : ctx->members[0];
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  Arena ar(s);
  nvtx_push("cco:pop_model");
  struct Pop { ~Pop() { nvtx_pop(); } } pop;
  const PopArgs a = pop_args(mode, start_ms, end_ms, n_items);
  int32_t *d_item, *d_counts;
  long long *d_t;
  unsigned long long *d_tot;
  double *d_score;
  unsigned char *d_present;
  CKR(ar.alloc(&d_item, std::max<long long>(n_events, 1)));
  CKR(ar.alloc(&d_t, std::max<long long>(n_events, 1)));
  CKR(ar.alloc(&d_counts, (size_t)a.n_buckets * n_items));
  CKR(ar.alloc(&d_tot, 4));
  CKR(ar.alloc(&d_score, n_items));
  CKR(ar.alloc(&d_present, n_items));
  CK(cudaMemsetAsync(d_counts, 0, sizeof(int32_t) * (size_t)a.n_buckets * n_items, s));
  CK(cudaMemsetAsync(d_tot, 0, 32, s));
  if (n_events > 0) {
    CK(cudaMemcpyAsync(d_item, item, sizeof(int32_t) * (size_t)n_events, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_t, time_ms, sizeof(int64_t) * (size_t)n_events, cudaMemcpyHostToDevice, s));
    k_pop_count<<<grid_for(n_events, 256, c->sm_count), 256, 0, s>>>(n_events, d_item, d_t, a, d_counts, d_tot);
    c->launches++;
  }
  k_pop_score<<<grid_for(n_items, 256, c->sm_count), 256, 0, s>>>(a, mode, d_counts, d_tot, d_score, d_present);
  c->launches++;
  CK(cudaMemcpyAsync(score, d_score, sizeof(double) * (size_t)n_items, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(present, d_present, (size_t)n_items, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  return CCO_OK;
}

// ---- URModel.save document content: correlators + rank fields + item properties (cco_model.cuh) ------------------------
namespace cco {
// the host-side checks of a dictionary: offsets[0] == 0, offsets[n] >= 0, bytes present; the device checks the rest
static int check_dict_host(const cco_dictionary_t &d, const char *what, int k) {
  if (d.n < 0 || !d.offsets) return set_error(CCO_E_INVALID_ARG, "%s %d: negative size or null offsets", what, k);
  if (d.offsets[0] != 0) return set_error(CCO_E_INVALID_ARG, "%s %d: offsets[0] != 0", what, k);
  if (d.offsets[d.n] < 0) return set_error(CCO_E_INVALID_ARG, "%s %d: offsets decrease", what, k);
  if (d.offsets[d.n] > 0 && !d.bytes) return set_error(CCO_E_INVALID_ARG, "%s %d: null bytes", what, k);
  return CCO_OK;
}
}  // namespace cco

int cco_format_model_bulk(cco_ctx_t *ctx, const cco_result_t *res, int32_t n_names, const char *const *names,
                          const cco_dictionary_t *row_ids, const cco_dictionary_t *col_ids, int32_t n_rankings,
                          const cco_ranking_t *rankings, const cco_dictionary_t *prop_ids, const cco_dictionary_t *prop_json,
                          uint32_t flags, char **out_bytes, int64_t *out_len) {
  if (!ctx || !res || !names || !row_ids || !col_ids || !out_bytes || !out_len || n_rankings < 0 || (n_rankings > 0 && !rankings))
    return set_error(CCO_E_INVALID_ARG, "null argument");
  if (!prop_ids != !prop_json) return set_error(CCO_E_INVALID_ARG, "prop_ids and prop_json go together");
  if (n_rankings > kMaxRankings) return set_error(CCO_E_UNSUPPORTED, "at most %d rankings (popular, trending, hot)", kMaxRankings);
  CKR(check_indicators(res, n_names, names, col_ids));
  const ResultMat &m0 = res->mats[0];
  if (m0.row_begin != 0 || m0.row_end != m0.n_cols)
    return set_error(CCO_E_UNSUPPORTED, "the result holds rows [%lld, %lld) of %d: format the merged model, not one rank's slice",
                     (long long)m0.row_begin, (long long)m0.row_end, m0.n_cols);
  const long long n_rows = m0.n_cols;
  if (row_ids->n != n_rows) return set_error(CCO_E_INVALID_ARG, "row dictionary has %lld ids for %lld rows", (long long)row_ids->n, n_rows);
  CKR(check_dict_host(*row_ids, "row dictionary", 0));
  for (int i = 0; i < n_names; ++i) CKR(check_dict_host(col_ids[i], "column dictionary", i));
  if (prop_ids) {
    CKR(check_dict_host(*prop_ids, "property ids", 0));
    CKR(check_dict_host(*prop_json, "property fragments", 0));
    if (prop_ids->n != prop_json->n)
      return set_error(CCO_E_INVALID_ARG, "%lld property ids but %lld fragments", (long long)prop_ids->n, (long long)prop_json->n);
  }
  const char *rank_names[kMaxRankings];
  for (int r = 0; r < n_rankings; ++r) {
    const cco_ranking_t &k = rankings[r];
    if (!k.name) return set_error(CCO_E_INVALID_ARG, "ranking %d: null name", r);
    if (!strcmp(k.name, "id")) return set_error(CCO_E_INVALID_ARG, "ranking %d: the name \"id\" is the document id", r);
    for (int i = 0; i < n_names; ++i)
      if (!strcmp(k.name, names[i])) return set_error(CCO_E_INVALID_ARG, "ranking %d: name \"%s\" is an indicator name", r, k.name);
    for (int q = 0; q < r; ++q)
      if (!strcmp(k.name, rankings[q].name)) return set_error(CCO_E_INVALID_ARG, "ranking %d: name \"%s\" repeated", r, k.name);
    if (k.mode < CCO_POP_POPULAR || k.mode > CCO_POP_HOT) return set_error(CCO_E_INVALID_ARG, "ranking %d: mode must be CCO_POP_POPULAR, _TRENDING or _HOT", r);
    if (k.end_ms < k.start_ms) return set_error(CCO_E_INVALID_ARG, "ranking %d: end before start (Joda Interval would throw)", r);
    CKR(check_dict_host(k.item, "ranking", r));
    if (k.item.n > 0 && !k.time_ms) return set_error(CCO_E_INVALID_ARG, "ranking %d: null event times", r);
    if (k.item.n > 0x7fffffffLL) return set_error(CCO_E_UNSUPPORTED, "ranking %d: %lld events (at most 2^31 - 1)", r, (long long)k.item.n);
    rank_names[r] = k.name;
  }
  // one column of every id: the rows, then every ranking's event items, then the property ids
  std::vector<const cco_dictionary_t *> parts = {row_ids};
  for (int r = 0; r < n_rankings; ++r) parts.push_back(&rankings[r].item);
  if (prop_ids) parts.push_back(prop_ids);
  std::vector<long long> first(parts.size() + 1, 0), byte0(parts.size() + 1, 0);
  for (size_t k = 0; k < parts.size(); ++k) {
    first[k + 1] = first[k] + parts[k]->n;
    byte0[k + 1] = byte0[k] + parts[k]->offsets[parts[k]->n];
  }
  const long long n_all = first[parts.size()];
  if (n_all >= (1LL << 32)) return set_error(CCO_E_UNSUPPORTED, "%lld ids in all (at most 2^32 - 1)", n_all);
  const long long prop_base = prop_ids ? first[parts.size() - 1] : n_all, n_prop = prop_ids ? prop_ids->n : 0;

  cco_ctx *c = ctx->members.empty() ? ctx : ctx->members[0];   // a group's merged model is formatted on its first GPU
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  nvtx_push("cco:format_model_bulk");
  struct Pop { ~Pop() { nvtx_pop(); } } pop;
  mail_reset(c);
  Arena ar(s);
  const unsigned long long N = (unsigned long long)n_all;

  // offsets first: no id byte is read before every dictionary's offsets are known not to decrease
  long long *off_all;
  unsigned char *bytes_all;
  int *bad;
  CKR(ar.alloc(&off_all, N + 1));
  CKR(ar.alloc(&bad, 1));
  CK(cudaMemsetAsync(bad, 0x7f, sizeof(int), s));
  for (size_t k = 0; k < parts.size(); ++k) {
    const long long n = parts[k]->n;
    long long *o = off_all + first[k];
    CK(cudaMemcpyAsync(o, parts[k]->offsets, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, s));
    if (n > 0) {
      k_ingest_str_check_offsets<<<grid_for(n, 256, c->sm_count), 256, 0, s>>>(n, o, (int)k, bad);
      c->launches++;
    }
    if (byte0[k] != 0) {   // rebase onto the concatenated bytes (the next part's copy rewrites the shared last entry with the same value)
      k_add_i64<<<grid_for(n + 1, 256, c->sm_count, 2), 256, 0, s>>>(n + 1, byte0[k], o);
      c->launches++;
    }
  }
  // the other dictionaries: column ids (code 100 + i) and the fragments (code 200)
  std::vector<const cco_dictionary_t *> others;
  for (int i = 0; i < n_names; ++i) others.push_back(&col_ids[i]);
  if (prop_json) others.push_back(prop_json);
  for (size_t k = 0; k < others.size(); ++k) {
    const long long n = others[k]->n;
    if (n == 0) continue;
    long long *o;
    CKR(ar.alloc(&o, n + 1));
    CK(cudaMemcpyAsync(o, others[k]->offsets, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, s));
    k_ingest_str_check_offsets<<<grid_for(n, 256, c->sm_count), 256, 0, s>>>(n, o, (int)k < n_names ? 100 + (int)k : 200, bad);
    c->launches++;
    ar.release(o);
  }
  int first_bad = 0;
  CKR(mail_fetch(c, &first_bad, bad, sizeof(int)));
  CKR(mail_wait(c));
  if (first_bad != 0x7f7f7f7f) {
    if (first_bad >= 200) return set_error(CCO_E_INVALID_ARG, "property fragments: offsets decrease");
    if (first_bad >= 100) return set_error(CCO_E_INVALID_ARG, "column dictionary %d: offsets decrease", first_bad - 100);
    if (first_bad == 0) return set_error(CCO_E_INVALID_ARG, "row dictionary: offsets decrease");
    if (first_bad <= n_rankings) return set_error(CCO_E_INVALID_ARG, "ranking %d: offsets decrease", first_bad - 1);
    return set_error(CCO_E_INVALID_ARG, "property ids: offsets decrease");
  }
  CKR(ar.alloc(&bytes_all, std::max<long long>(byte0[parts.size()], 1)));
  for (size_t k = 0; k < parts.size(); ++k) {
    const long long nb = byte0[k + 1] - byte0[k];
    if (nb > 0) CK(cudaMemcpyAsync(bytes_all + byte0[k], parts[k]->bytes, (size_t)nb, cudaMemcpyHostToDevice, s));
  }
  DevCol all;
  all.n = n_all;
  all.off = off_all;
  all.bytes = bytes_all;
  const StrCols cols = one_column(all);

  // group equal ids; number the classes (distinct ids) in order of first appearance; rows are classes 0 .. n_rows - 1
  uint32_t *rep, *cflag, *cpos;
  int *dup;   // [0] a repeated row id, [1] a repeated property id
  CKR(ar.alloc(&rep, N));
  CKR(ar.alloc(&cflag, N + 1));
  CKR(ar.alloc(&cpos, N + 1));
  CKR(ar.alloc(&dup, 2));
  CKR(group_ids(c, ar, N, cols, (flags & CCO_FLAG_INGEST_SHORT_HASH) != 0, rep));
  CK(cudaMemsetAsync(dup, 0, 2 * sizeof(int), s));
  CK(cudaMemsetAsync(cflag + N, 0, sizeof(uint32_t), s));
  const int G = grid_for(n_all, 256, c->sm_count);
  if (N > 0) {
    k_model_class_flags<<<G, 256, 0, s>>>(N, (unsigned long long)n_rows, rep, cflag, dup);
    c->launches++;
  }
  CKR(exclusive_sum_u32(c, ar, cflag, cpos, n_all + 1));
  uint32_t n_classes = 0;
  CKR(mail_fetch(c, &n_classes, cpos + N, 4));
  CKR(mail_wait(c));
  if (n_classes > 0x7fffffffu) return set_error(CCO_E_UNSUPPORTED, "%u distinct ids (at most 2^31 - 1)", n_classes);
  uint32_t *cls_elem, *prop_of;
  CKR(ar.alloc(&cls_elem, n_classes));
  CKR(ar.alloc(&prop_of, n_classes));
  CK(cudaMemsetAsync(prop_of, 0xff, sizeof(uint32_t) * std::max<size_t>(n_classes, 1), s));
  if (N > 0) {
    k_model_class_elem<<<G, 256, 0, s>>>(N, rep, cpos, cls_elem);
    c->launches++;
  }
  if (n_prop > 0) {
    k_model_props<<<grid_for(n_prop, 256, c->sm_count), 256, 0, s>>>(n_prop, prop_base, rep, cpos, prop_of, dup + 1);
    c->launches++;
  }
  int dups[2] = {0, 0};
  CKR(mail_fetch(c, dups, dup, 2 * sizeof(int)));
  CKR(mail_wait(c));
  if (dups[0]) return set_error(CCO_E_INVALID_ARG, "two equal ids in the row dictionary");
  if (dups[1]) return set_error(CCO_E_INVALID_ARG, "two equal property ids");

  // rank histograms per class: the counting of cco_pop_model over class indices, then its scoring
  ModelArgs ma;
  memset(&ma, 0, sizeof ma);
  ma.n_rank = n_rankings;
  for (int r = 0; r < n_rankings; ++r) {
    const cco_ranking_t &k = rankings[r];
    const PopArgs pa = pop_args(k.mode, k.start_ms, k.end_ms, (int32_t)n_classes);
    int32_t *counts;
    unsigned long long *tot;
    long long *d_t;
    double *score;
    unsigned char *present;
    CKR(ar.alloc(&counts, (size_t)pa.n_buckets * n_classes));
    CKR(ar.alloc(&tot, 4));
    CKR(ar.alloc(&d_t, std::max<long long>(k.item.n, 1)));
    CKR(ar.alloc(&score, n_classes));
    CKR(ar.alloc(&present, n_classes));
    CK(cudaMemsetAsync(counts, 0, sizeof(int32_t) * std::max<size_t>((size_t)pa.n_buckets * n_classes, 1), s));
    CK(cudaMemsetAsync(tot, 0, 32, s));
    if (k.item.n > 0) {
      CK(cudaMemcpyAsync(d_t, k.time_ms, sizeof(int64_t) * (size_t)k.item.n, cudaMemcpyHostToDevice, s));
      k_rank_count<<<grid_for(k.item.n, 256, c->sm_count), 256, 0, s>>>(k.item.n, rep + first[1 + r], cpos, d_t, pa, counts, tot);
      c->launches++;
    }
    if (n_classes > 0) {
      k_pop_score<<<grid_for(n_classes, 256, c->sm_count), 256, 0, s>>>(pa, k.mode, counts, tot, score, present);
      c->launches++;
    }
    ar.release(counts);
    ar.release(d_t);
    ma.score[r] = score;
    ma.present[r] = present;
  }
  if (n_rankings > 0) CKR(escape_names(c, ar, n_rankings, rank_names, &ma.rank_names, ma.rank_name_off));

  // documents: every row, then the extra classes with a present rank or a property entry, in class order
  ma.prop_of = prop_of;
  ma.f.n_rows = (int32_t)n_rows;
  uint32_t *dflag, *dpos;
  CKR(ar.alloc(&dflag, (size_t)n_classes + 1));
  CKR(ar.alloc(&dpos, (size_t)n_classes + 1));
  CK(cudaMemsetAsync(dflag + n_classes, 0, sizeof(uint32_t), s));
  if (n_classes > 0) {
    k_model_doc_flags<<<grid_for(n_classes, 256, c->sm_count), 256, 0, s>>>(ma, n_classes, dflag);
    c->launches++;
  }
  CKR(exclusive_sum_u32(c, ar, dflag, dpos, (long long)n_classes + 1));
  uint32_t n_docs = 0;
  CKR(mail_fetch(c, &n_docs, dpos + n_classes, 4));
  CKR(mail_wait(c));
  uint32_t *doc_cls, *doc_src;
  CKR(ar.alloc(&doc_cls, n_docs));
  CKR(ar.alloc(&doc_src, n_docs));
  if (n_classes > 0) {
    k_model_doc_list<<<grid_for(n_classes, 256, c->sm_count), 256, 0, s>>>(n_classes, dflag, dpos, cls_elem, doc_cls, doc_src);
    c->launches++;
  }
  ma.n_docs = n_docs;
  ma.doc_cls = doc_cls;

  // the document ids, gathered and escaped; the fragments verbatim; the indicators as cco_format_es_bulk has them
  DevCol ids;
  std::vector<void *> unused;
  CKR(gather_dict(c, ar, cols, doc_src, n_docs, &ids, nullptr, unused));
  CKR(escape_dict(c, ar, DevDict{ids.off, ids.bytes, ids.n}, &ma.f.row_ids));
  const cco_dictionary_t no_props = {0, nullptr, nullptr};
  CKR(upload_dict(c, ar, prop_json ? *prop_json : no_props, &ma.frag));
  FormatArgs fa;
  memset(&fa, 0, sizeof fa);
  CKR(upload_indicators(c, ar, res, names, col_ids, &fa));
  fa.row_ids = ma.f.row_ids;
  ma.f = fa;
  return assemble_docs(
      ctx, c, ar, (long long)n_docs,
      [&](long long *doc_len) { k_model_doc_len<<<grid_for(n_docs, 256, c->sm_count), 256, 0, s>>>(ma, doc_len); },
      [&](const long long *doc_off, unsigned char *out) {
        k_model_doc_write<<<grid_for((long long)n_docs * 32, 256, c->sm_count), 256, 0, s>>>(ma, doc_off, out);
      },
      out_bytes, out_len);
}

void cco_free(void *p) { free(p); }

// ---- debug / parity entries ------------------------------------------------------------------------
int cco_debug_llr(cco_ctx_t *c, int64_t n, const int64_t *k11, const int64_t *k12, const int64_t *k21, const int64_t *k22,
                  uint32_t flags, double *out) {
  if (!c || n < 0 || (n > 0 && (!k11 || !k12 || !k21 || !k22 || !out))) return set_error(CCO_E_INVALID_ARG, "bad argument");
  if (n == 0) return CCO_OK;
  for (int64_t i = 0; i < n; ++i)
    if (k11[i] < 0 || k12[i] < 0 || k21[i] < 0 || k22[i] < 0)
      return set_error(CCO_E_INVALID_ARG, "negative count at %lld (Preconditions.checkArgument in LogLikelihood)", (long long)i);
  CK(cudaSetDevice(c->device));
  Arena ar(c->stream);
  long long *d[4];
  double *dout;
  const int64_t *h[4] = {k11, k12, k21, k22};
  for (int j = 0; j < 4; ++j) {
    CKR(ar.alloc(&d[j], n));
    CK(cudaMemcpyAsync(d[j], h[j], sizeof(int64_t) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  }
  CKR(ar.alloc(&dout, n));
  k_debug_llr<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(n, d[0], d[1], d[2], d[3], flags, dout);
  CK(cudaMemcpyAsync(out, dout, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaGetLastError());
  return CCO_OK;
}

int cco_debug_downsample(cco_ctx_t *c, const cco_csr_t *m, int32_t max_interactions, int32_t seed, uint32_t flags,
                         int64_t **row_ptr, int32_t **col_idx, int32_t *raw_col_counts, int32_t *new_col_counts) {
  if (!c || !m || !row_ptr || !col_idx) return set_error(CCO_E_INVALID_ARG, "null argument");
  if (c->world != 1 || !c->members.empty()) return set_error(CCO_E_UNSUPPORTED, "debug entries need a single-GPU context");
  cco_indicator_params_t prm = {max_interactions, 1, 0, 0.0};
  CKR(validate_host(1, m, &prm));
  CK(cudaSetDevice(c->device));
  mail_reset(c);
  cco_dataset *ds = nullptr;
  CKR(dataset_upload(c, 1, m, flags, &ds));
  struct DG { cco_dataset *d; ~DG() { dataset_release(d); } } dg{ds};
  Arena ar(c->stream);
  DevRaw raw;
  raw.n_rows = ds->n_users; raw.n_cols = (int32_t)ds->n_cols[0]; raw.nnz = ds->nnz[0]; raw.nnz_cap = ds->nnz[0];
  raw.rp = ds->rp[0]; raw.col = ds->col[0];
  int32_t *counts;
  CKR(ar.alloc(&counts, std::max<int32_t>(m->n_cols, 1)));
  CK(cudaMemsetAsync(counts, 0, sizeof(int32_t) * (size_t)std::max<int32_t>(m->n_cols, 1), c->stream));
  if (raw.nnz > 0 && m->n_rows > 0)
    k_col_histogram<<<grid_for(raw.nnz, 256, c->sm_count), 256, 0, c->stream>>>(0, m->n_rows, raw.rp, raw.col, raw.n_cols, counts, 1, 0);
  DevMat dm;
  CKR(downsample_device(c, ar, raw, nullptr, counts, max_interactions, seed, flags, &dm));
  std::vector<uint32_t> rp32((size_t)m->n_rows + 1);
  CK(cudaMemcpyAsync(rp32.data(), dm.rp, sizeof(uint32_t) * rp32.size(), cudaMemcpyDeviceToHost, c->stream));
  if (raw_col_counts && m->n_cols > 0)
    CK(cudaMemcpyAsync(raw_col_counts, counts, sizeof(int32_t) * (size_t)m->n_cols, cudaMemcpyDeviceToHost, c->stream));
  if (new_col_counts && m->n_cols > 0)
    CK(cudaMemcpyAsync(new_col_counts, dm.marg, sizeof(int32_t) * (size_t)m->n_cols, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaGetLastError());
  size_t nnz = rp32[m->n_rows];
  int64_t *rp = (int64_t *)malloc(sizeof(int64_t) * rp32.size());
  int32_t *ci = (int32_t *)malloc(sizeof(int32_t) * std::max<size_t>(nnz, 1));
  if (!rp || !ci) return set_error(CCO_E_OOM, "malloc failed");
  for (size_t i = 0; i < rp32.size(); ++i) rp[i] = rp32[i];
  if (nnz) CK(cudaMemcpy(ci, dm.col, sizeof(int32_t) * nnz, cudaMemcpyDeviceToHost));
  *row_ptr = rp;
  *col_idx = ci;
  return CCO_OK;
}

int cco_debug_cooccurrence(cco_ctx_t *c, const cco_csr_t *a, const cco_csr_t *b, int64_t **row_ptr, int32_t **col_idx,
                           int32_t **count) {
  if (!c || !a || !b || !row_ptr || !col_idx || !count) return set_error(CCO_E_INVALID_ARG, "null argument");
  if (c->world != 1 || !c->members.empty()) return set_error(CCO_E_UNSUPPORTED, "debug entries need a single-GPU context");
  cco_csr_t two[2] = {*a, *b};
  cco_indicator_params_t prm[2] = {{0x7fffffff, 1, 0, 0.0}, {0x7fffffff, 1, 0, 0.0}};
  CKR(validate_host(2, two, prm));
  CK(cudaSetDevice(c->device));
  mail_reset(c);
  cudaStream_t s = c->stream;
  cco_dataset *ds = nullptr;
  CKR(dataset_upload(c, 2, two, 0, &ds));
  struct DG { cco_dataset *d; ~DG() { dataset_release(d); } } dg{ds};
  Arena ar(s);
  struct CopyJoin {
    cco_ctx *c;
    ~CopyJoin() { cudaStreamSynchronize(c->copy_stream); }
  } copy_join{c};
  std::vector<DevRaw> raw(2);
  for (int i = 0; i < 2; ++i) {
    raw[i].n_rows = ds->n_users; raw[i].n_cols = (int32_t)ds->n_cols[i]; raw[i].nnz = ds->nnz[i]; raw[i].nnz_cap = ds->nnz[i];
    raw[i].rp = ds->rp[i]; raw[i].col = ds->col[i];
  }
  // identity "downsample" (m = INT_MAX) gives the device CSR + marginals
  std::vector<DevMat> dm(2);
  for (int i = 0; i < 2; ++i) {
    int32_t *counts;
    CKR(ar.alloc(&counts, std::max<int32_t>(raw[i].n_cols, 1)));
    CK(cudaMemsetAsync(counts, 0, sizeof(int32_t) * (size_t)std::max<int32_t>(raw[i].n_cols, 1), s));
    if (raw[i].nnz > 0 && raw[i].n_rows > 0)
      k_col_histogram<<<grid_for(raw[i].nnz, 256, c->sm_count), 256, 0, s>>>(0, raw[i].n_rows, raw[i].rp, raw[i].col, raw[i].n_cols, counts, 1, 0);
    CKR(downsample_device(c, ar, raw[i], nullptr, counts, 0x7fffffff, 0, 0, &dm[i]));
  }
  const int32_t n_items_a = dm[0].n_cols;
  uint32_t *at_ptr, *cursor, *marg_pad;
  int32_t *at_users, *d_max;
  CKR(ar.alloc(&at_ptr, n_items_a + 1));
  CKR(ar.alloc(&cursor, n_items_a + 1));
  CKR(ar.alloc(&marg_pad, n_items_a + 1));
  CKR(ar.alloc(&d_max, 2));
  CKR(ar.alloc(&at_users, std::max<long long>(raw[0].nnz, 1)));
  CK(cudaMemsetAsync(d_max, 0, 8, s));
  CK(cudaMemcpyAsync(marg_pad, dm[0].marg, sizeof(int32_t) * (size_t)n_items_a, cudaMemcpyDeviceToDevice, s));
  CK(cudaMemsetAsync(marg_pad + n_items_a, 0, 4, s));
  CKR(exclusive_sum_u32(c, ar, marg_pad, at_ptr, (long long)n_items_a + 1));
  CK(cudaMemcpyAsync(cursor, at_ptr, sizeof(uint32_t) * ((size_t)n_items_a + 1), cudaMemcpyDeviceToDevice, s));
  k_transpose_scatter<<<grid_for(a->n_rows * kSG, 256, c->sm_count), 256, 0, s>>>(a->n_rows, dm[0].rp, dm[0].col, cursor, at_users);
  if (n_items_a > 0) k_max_i32<<<grid_for(n_items_a, 256, c->sm_count, 2), 256, 0, s>>>(n_items_a, dm[0].marg, d_max);
  if (dm[1].n_cols > 0) k_max_i32<<<grid_for(dm[1].n_cols, 256, c->sm_count, 2), 256, 0, s>>>(dm[1].n_cols, dm[1].marg, d_max + 1);
  int32_t max_marg_ab[2] = {0, 0};
  CK(cudaMemcpyAsync(max_marg_ab, d_max, 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  ResultMat rm;
  IndicatorOut io;
  IndicatorState ist;
  struct EG { IndicatorState &x; ~EG() { if (x.packed) cudaEventDestroy(x.packed); } } eg{ist};
  cco_indicator_params_t p1 = {0x7fffffff, 1, 0, 0.0};
  auto put = [&]() {
    for (void *p : {(void *)rm.row_ptr, (void *)rm.col, (void *)rm.llr, (void *)rm.cnt})
      if (p) c->pinned_put(p);
  };
  int rc = enqueue_indicator(c, ar, at_ptr, at_users, n_items_a, dm[0].marg, max_marg_ab[0], max_marg_ab[1], dm[1], a->n_rows, false, p1,
                             0, true, nullptr, nullptr, nullptr, &ist);
  if (rc == CCO_OK) rc = finish_indicator(c, &ist, 0, 0, &rm, &io);
  cudaStreamSynchronize(c->copy_stream);
  if (rc != CCO_OK) {
    put();
    return rc;
  }
  size_t nnz = (size_t)rm.row_ptr[n_items_a];
  int64_t *rp = (int64_t *)malloc(sizeof(int64_t) * ((size_t)n_items_a + 1));
  int32_t *ci = (int32_t *)malloc(sizeof(int32_t) * std::max<size_t>(nnz, 1));
  int32_t *cn = (int32_t *)malloc(sizeof(int32_t) * std::max<size_t>(nnz, 1));
  if (!rp || !ci || !cn) {
    put();
    return set_error(CCO_E_OOM, "malloc failed");
  }
  memcpy(rp, rm.row_ptr, sizeof(int64_t) * ((size_t)n_items_a + 1));
  // cells of a row come back in table order: sort each row by column for the caller
  std::vector<std::pair<int32_t, int32_t>> tmp;
  for (int32_t r = 0; r < n_items_a; ++r) {
    size_t lo = (size_t)rp[r], hi = (size_t)rp[r + 1];
    tmp.resize(hi - lo);
    for (size_t q = lo; q < hi; ++q) tmp[q - lo] = {rm.col[q], rm.cnt[q]};
    std::sort(tmp.begin(), tmp.end());
    for (size_t q = lo; q < hi; ++q) {
      ci[q] = tmp[q - lo].first;
      cn[q] = tmp[q - lo].second;
    }
  }
  put();
  *row_ptr = rp;
  *col_idx = ci;
  *count = cn;
  return CCO_OK;
}

}  // extern "C"
