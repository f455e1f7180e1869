// cco_strings.cuh -- device kernels of cco_ingest_strings: Preparator.prepare from raw (user, item) id strings
// (Preparator.scala:111-126, 170-190 builds one BiDictionary per id space from distinct().collect()).
//
//   hashing                    -> k_ingest_str_hash (64-bit hash of every id; a warp takes the long ones)
//   grouping equal ids         -> CUB radix sort of (hash, index), k_ingest_str_run_heads + max-scan,
//                                 k_ingest_str_resolve (byte comparison against the first id of each equal-hash run);
//                                 ids that differ from their run's first id (hash collisions) are sorted by
//                                 (hash, bytes, index) and grouped by k_ingest_str_class_heads / k_ingest_str_class_rep
//   user dictionary            -> k_ingest_str_user_count, k_ingest_str_user_flags, k_ingest_str_user_tokens,
//                                 k_ingest_str_match_users (secondary-type users against the user dictionary)
//   item dictionaries          -> k_ingest_str_first_surv, k_ingest_str_item_flags, k_ingest_str_item_tokens
//   dictionary bytes           -> k_ingest_str_lengths + scan + k_ingest_str_gather
//   input check                -> k_ingest_str_check_offsets
//
// Equality of ids is byte equality; the hash only brings candidates together.  Every kernel is grid-stride over
// warps: a lane handles an id of up to kShortId bytes alone, longer ids are handled by the whole warp one after the
// other, so one very long id does not hold 31 lanes idle for its whole length.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace cco {

constexpr long long kShortId = 64;
constexpr uint32_t kNoRep = 0xffffffffu;

// one column of ids, or two columns back to back: element i < n_a is id i of column a, element n_a + j is id j of b
struct StrCols {
  long long n_a = 0;
  const long long *off_a = nullptr;
  const unsigned char *bytes_a = nullptr;
  const long long *off_b = nullptr;
  const unsigned char *bytes_b = nullptr;
  __device__ __forceinline__ void get(unsigned long long i, const unsigned char **p, long long *len) const {
    if ((long long)i < n_a) {
      const long long s = off_a[i];
      *p = bytes_a + s;
      *len = off_a[i + 1] - s;
    } else {
      i -= (unsigned long long)n_a;
      const long long s = off_b[i];
      *p = bytes_b + s;
      *len = off_b[i + 1] - s;
    }
  }
};

__device__ __forceinline__ uint64_t str_mix(uint64_t z) {
  z ^= z >> 30;
  z *= 0xbf58476d1ce4e5b9ULL;
  z ^= z >> 27;
  z *= 0x94d049bb133111ebULL;
  z ^= z >> 31;
  return z;
}
// little-endian 8-byte word w of an id, zero past its end
__device__ __forceinline__ uint64_t str_word(const unsigned char *p, long long len, long long w) {
  const long long b = w * 8;
  const int n = (int)(len - b < 8 ? len - b : 8);
  uint64_t x = 0;
  for (int k = 0; k < n; ++k) x |= (uint64_t)p[b + k] << (8 * k);
  return x;
}
// hash = mix(sum over words w of mix(word_w ^ w * golden) + len * c): a sum, so a warp can split the words of a long id
__device__ __forceinline__ uint64_t str_term(const unsigned char *p, long long len, long long w) {
  return str_mix(str_word(p, len, w) ^ ((uint64_t)w * 0x9e3779b97f4a7c15ULL));
}
__device__ __forceinline__ uint64_t str_finish(uint64_t sum, long long len, uint64_t mask) {
  return str_mix(sum + (uint64_t)len * 0xd6e8feb86659fd93ULL) & mask;
}

__device__ __forceinline__ unsigned long long warp_first_index() {
  return (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x) & ~31ULL;
}
__device__ __forceinline__ unsigned long long grid_threads() { return (unsigned long long)gridDim.x * blockDim.x; }

// Equality of (p, lp) and (q, lq) for the lanes with `want`.  Called by all 32 lanes together.
__device__ __forceinline__ bool warp_equal(bool want, const unsigned char *p, long long lp, const unsigned char *q, long long lq) {
  const int lane = threadIdx.x & 31;
  bool eq = want && lp == lq;
  const bool lng = eq && lp > kShortId;
  if (eq && !lng)
    for (long long k = 0; k < lp; ++k)
      if (p[k] != q[k]) { eq = false; break; }
  unsigned m = __ballot_sync(0xffffffffu, lng);
  while (m) {
    const int src = __ffs(m) - 1;
    m &= m - 1;
    const unsigned char *a = (const unsigned char *)__shfl_sync(0xffffffffu, (unsigned long long)p, src);
    const unsigned char *b = (const unsigned char *)__shfl_sync(0xffffffffu, (unsigned long long)q, src);
    const long long l = __shfl_sync(0xffffffffu, lp, src);
    bool diff = false;
    for (long long b0 = 0; b0 < l; b0 += 32 * 8) {
      const long long k0 = b0 + lane * 8;
      for (long long k = k0; k < k0 + 8 && k < l; ++k) diff |= a[k] != b[k];
      if (__any_sync(0xffffffffu, diff)) { diff = true; break; }
    }
    if (lane == src) eq = !diff;
  }
  return eq;
}

// hash[i] = hash of element i (masked: the tests-only short hash keeps a few bits), idx[i] = i
__global__ void k_ingest_str_hash(unsigned long long n, StrCols c, uint64_t mask, unsigned long long *__restrict__ hash,
                                  uint32_t *__restrict__ idx) {
  const int lane = threadIdx.x & 31;
  for (unsigned long long base = warp_first_index(); base < n; base += grid_threads()) {
    const unsigned long long i = base + lane;
    const unsigned char *p = nullptr;
    long long len = 0;
    const bool have = i < n;
    if (have) c.get(i, &p, &len);
    const bool lng = have && len > kShortId;
    if (have && !lng) {
      uint64_t s = 0;
      for (long long w = 0; w * 8 < len; ++w) s += str_term(p, len, w);
      hash[i] = str_finish(s, len, mask);
      idx[i] = (uint32_t)i;
    }
    unsigned m = __ballot_sync(0xffffffffu, lng);
    while (m) {
      const int src = __ffs(m) - 1;
      m &= m - 1;
      const unsigned char *q = (const unsigned char *)__shfl_sync(0xffffffffu, (unsigned long long)p, src);
      const long long ql = __shfl_sync(0xffffffffu, len, src);
      uint64_t s = 0;
      for (long long w = lane; w * 8 < ql; w += 32) s += str_term(q, ql, w);
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == src) {
        hash[i] = str_finish(s, ql, mask);
        idx[i] = (uint32_t)i;
      }
    }
  }
}

// head[k] = k where a run of equal sorted hashes starts, 0 elsewhere (an inclusive max-scan then gives each position
// the start of its run)
__global__ void k_ingest_str_run_heads(unsigned long long n, const unsigned long long *__restrict__ hs, uint32_t *__restrict__ head) {
  for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < n; k += grid_threads())
    head[k] = (k == 0 || hs[k] != hs[k - 1]) ? (uint32_t)k : 0u;
}

// Sorted position k holds element is[k]; its run of equal hashes starts at head[k], whose element is the smallest index
// of the run (the radix sort is stable).  rep[i] = that first element when the bytes are equal; otherwise i is a
// collision and goes to the list `un` for the exact pass.
__global__ void k_ingest_str_resolve(unsigned long long n, StrCols c, const uint32_t *__restrict__ is, const uint32_t *__restrict__ head,
                                     uint32_t *__restrict__ rep, uint32_t *__restrict__ un, unsigned long long *__restrict__ n_un) {
  const int lane = threadIdx.x & 31;
  for (unsigned long long base = warp_first_index(); base < n; base += grid_threads()) {
    const unsigned long long k = base + lane;
    const bool have = k < n;
    uint32_t i = 0, j = 0;
    const unsigned char *p = nullptr, *q = nullptr;
    long long lp = 0, lq = 0;
    bool cmp = false;
    if (have) {
      i = is[k];
      const uint32_t h = head[k];
      j = is[h];
      cmp = h != k;
      if (cmp) {
        c.get(i, &p, &lp);
        c.get(j, &q, &lq);
      } else {
        rep[i] = i;
      }
    }
    const bool eq = warp_equal(cmp, p, lp, q, lq);
    if (cmp) {
      if (eq) rep[i] = j;
      else {
        rep[i] = kNoRep;
        un[atomicAdd(n_un, 1ULL)] = i;
      }
    }
  }
}

// the exact order of the collision pass: (hash, bytes, length, index); equal ids end up adjacent, smallest index first
struct StrLess {
  StrCols c;
  const unsigned long long *hash;
  __device__ bool operator()(uint32_t a, uint32_t b) const {
    if (hash[a] != hash[b]) return hash[a] < hash[b];
    const unsigned char *p, *q;
    long long la, lb;
    c.get(a, &p, &la);
    c.get(b, &q, &lb);
    const long long l = la < lb ? la : lb;
    for (long long k = 0; k < l; ++k)
      if (p[k] != q[k]) return p[k] < q[k];
    if (la != lb) return la < lb;
    return a < b;
  }
};

// over the collision list sorted by StrLess: head[k] = k where a class of equal ids starts, 0 elsewhere
__global__ void k_ingest_str_class_heads(unsigned long long n, StrCols c, const uint32_t *__restrict__ un,
                                         const unsigned long long *__restrict__ hash, uint32_t *__restrict__ head) {
  const int lane = threadIdx.x & 31;
  for (unsigned long long base = warp_first_index(); base < n; base += grid_threads()) {
    const unsigned long long k = base + lane;
    const bool have = k < n;
    const unsigned char *p = nullptr, *q = nullptr;
    long long lp = 0, lq = 0;
    bool cmp = false;
    if (have && k > 0) {
      const uint32_t a = un[k - 1], b = un[k];
      cmp = hash[a] == hash[b];
      if (cmp) {
        c.get(a, &p, &lp);
        c.get(b, &q, &lq);
      }
    }
    const bool eq = warp_equal(cmp, p, lp, q, lq);
    if (have) head[k] = eq ? 0u : (uint32_t)k;
  }
}
__global__ void k_ingest_str_class_rep(unsigned long long n, const uint32_t *__restrict__ un, const uint32_t *__restrict__ head,
                                       uint32_t *__restrict__ rep) {
  for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < n; k += grid_threads())
    rep[un[k]] = un[head[k]];
}

// ---- users ----------------------------------------------------------------------------------------------------------
// primary events per distinct user (duplicates count: Preparator.scala:129-132); cnt is indexed by the first event
__global__ void k_ingest_str_user_count(unsigned long long n, const uint32_t *__restrict__ rep, uint32_t *__restrict__ cnt) {
  for (unsigned long long e = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; e < n; e += grid_threads())
    atomicAdd(&cnt[rep[e]], 1u);
}
// first[e] = e is the first appearance of its user; kept[e] = ... and the user has at least `need` primary events
__global__ void k_ingest_str_user_flags(unsigned long long n, const uint32_t *__restrict__ rep, const uint32_t *__restrict__ cnt,
                                        uint32_t need, uint32_t *__restrict__ first, uint32_t *__restrict__ kept) {
  for (unsigned long long e = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; e < n; e += grid_threads()) {
    const bool f = rep[e] == (uint32_t)e;
    first[e] = f ? 1u : 0u;
    kept[e] = f && cnt[e] >= need ? 1u : 0u;
  }
}
// primary event e: raw user id = first-appearance rank of its user, survives iff the user is kept.  Kept users also
// fill the dictionary: dict_ev[d] = first event of user d, dict_raw[d] = its raw id.
__global__ void k_ingest_str_user_tokens(unsigned long long n, const uint32_t *__restrict__ rep, const uint32_t *__restrict__ fpos,
                                         const uint32_t *__restrict__ kept, const uint32_t *__restrict__ kpos,
                                         long long *__restrict__ uraw, uint32_t *__restrict__ surv, uint32_t *__restrict__ dict_ev,
                                         uint32_t *__restrict__ dict_raw) {
  for (unsigned long long e = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; e < n; e += grid_threads()) {
    const uint32_t r = rep[e];
    uraw[e] = fpos[r];
    surv[e] = kept[r];
    if (kept[e]) {
      dict_ev[kpos[e]] = (uint32_t)e;
      dict_raw[kpos[e]] = fpos[e];
    }
  }
}
// secondary events grouped together with the user dictionary (elements [0, n_dict)): an event whose group starts in the
// dictionary gets that user's raw id; any other user gets `none`, a raw id without primary events, and is dropped
__global__ void k_ingest_str_match_users(unsigned long long n, uint32_t n_dict, const uint32_t *__restrict__ rep,
                                         const uint32_t *__restrict__ dict_raw, uint32_t none, long long *__restrict__ uraw,
                                         uint32_t *__restrict__ surv) {
  for (unsigned long long e = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; e < n; e += grid_threads()) {
    const uint32_t r = rep[n_dict + e];
    const bool m = r < n_dict;
    uraw[e] = m ? dict_raw[r] : none;
    surv[e] = m ? 1u : 0u;
  }
}

// ---- items ----------------------------------------------------------------------------------------------------------
// fs[first event of an item] = its first event with a surviving user (Preparator.scala:184: items of surviving events)
__global__ void k_ingest_str_first_surv(unsigned long long n, const uint32_t *__restrict__ rep, const uint32_t *__restrict__ surv,
                                        uint32_t *__restrict__ fs) {
  for (unsigned long long e = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; e < n; e += grid_threads())
    if (surv[e]) atomicMin(&fs[rep[e]], (uint32_t)e);
}
__global__ void k_ingest_str_item_flags(unsigned long long n, const uint32_t *__restrict__ rep, const uint32_t *__restrict__ fs,
                                        uint32_t *__restrict__ flag) {
  for (unsigned long long e = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; e < n; e += grid_threads())
    flag[e] = fs[rep[e]] == (uint32_t)e ? 1u : 0u;
}
// surviving event e: raw item id = rank of its item's first surviving appearance (dropped events: 0, never read)
__global__ void k_ingest_str_item_tokens(unsigned long long n, const uint32_t *__restrict__ rep, const uint32_t *__restrict__ surv,
                                         const uint32_t *__restrict__ fs, const uint32_t *__restrict__ flag,
                                         const uint32_t *__restrict__ ipos, int32_t *__restrict__ iraw, uint32_t *__restrict__ dict_ev) {
  for (unsigned long long e = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; e < n; e += grid_threads()) {
    iraw[e] = surv[e] ? (int32_t)ipos[fs[rep[e]]] : 0;
    if (flag[e]) dict_ev[ipos[e]] = (uint32_t)e;
  }
}

// ---- dictionary bytes -----------------------------------------------------------------------------------------------
__global__ void k_ingest_str_lengths(unsigned long long n, StrCols c, const uint32_t *__restrict__ src, long long *__restrict__ len) {
  for (unsigned long long d = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; d < n; d += grid_threads()) {
    const unsigned char *p;
    long long l;
    c.get(src[d], &p, &l);
    len[d] = l;
  }
}
__global__ void k_ingest_str_gather(unsigned long long n, StrCols c, const uint32_t *__restrict__ src, const long long *__restrict__ off,
                                    unsigned char *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  for (unsigned long long base = warp_first_index(); base < n; base += grid_threads()) {
    const unsigned long long d = base + lane;
    const unsigned char *p = nullptr;
    long long l = 0;
    const bool have = d < n;
    if (have) c.get(src[d], &p, &l);
    const bool lng = have && l > kShortId;
    if (have && !lng)
      for (long long k = 0; k < l; ++k) out[off[d] + k] = p[k];
    unsigned m = __ballot_sync(0xffffffffu, lng);
    while (m) {
      const int s = __ffs(m) - 1;
      m &= m - 1;
      const unsigned char *q = (const unsigned char *)__shfl_sync(0xffffffffu, (unsigned long long)p, s);
      const long long ql = __shfl_sync(0xffffffffu, l, s);
      unsigned char *dst = out + off[base + s];
      for (long long k = lane; k < ql; k += 32) dst[k] = q[k];
    }
  }
}

// offsets must not decrease: *bad = smallest column id with a decrease
__global__ void k_ingest_str_check_offsets(unsigned long long n, const long long *__restrict__ off, int col, int *__restrict__ bad) {
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += grid_threads())
    if (off[i + 1] < off[i]) atomicMin(bad, col);
}

}  // namespace cco
