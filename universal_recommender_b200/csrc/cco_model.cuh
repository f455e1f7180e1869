// cco_model.cuh -- the whole model document on the device (cco_format_model_bulk): URModel.save writes
// groupAll(correlators ++ propertiesRDD) (/root/reference/src/main/scala/URModel.scala:57-102), where propertiesRDD is the
// item properties full-outer-joined with one rank field per ranking (URAlgorithm.getRanksRDD, URAlgorithm.scala:351-367,
// 537-560).
//
//   one id space              -> group_ids over (row ids, every ranking's event item ids, property ids) (cco_strings.cuh);
//                                k_model_class_flags + scan numbers the distinct ids ("classes") by first appearance
//   property per class        -> k_model_props (a second property id in one class is a duplicate)
//   rank histograms per class -> k_rank_count (warp-aggregated atomics), then k_pop_score (cco_format.cuh)
//   document list             -> k_model_doc_flags + scan + k_model_doc_list
//   bytes                     -> doc ids gathered (k_ingest_str_lengths / _gather) and escaped (k_escape_*), then
//                                k_model_doc_len + scan + k_model_doc_write, one warp per document
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "cco_format.cuh"

namespace cco {

constexpr int kMaxRankings = 3;
constexpr uint32_t kNoProp = 0xffffffffu;

// Double.toString of an integral double with |v| < 2^34, as elasticsearch-hadoop writes a JDouble: "<int>.0" when
// |v| < 10^7, otherwise d.dddE<n> with the trailing zeros of the fraction stripped (at least one digit is kept).  At these
// magnitudes the shortest round-trip digits of the double are the integer's own digits.  s needs 24 bytes; returns the length.
__device__ __forceinline__ int java_double_integral(double v, char *s) {
  long long x = (long long)v;
  int n = 0;
  if (x < 0) {
    s[n++] = '-';
    x = -x;
  }
  char d[20];   // decimal digits, least significant first
  int nd = 0;
  do {
    d[nd++] = (char)('0' + x % 10);
    x /= 10;
  } while (x);
  if (nd <= 7) {
    for (int k = nd - 1; k >= 0; --k) s[n++] = d[k];
    s[n++] = '.';
    s[n++] = '0';
    return n;
  }
  s[n++] = d[nd - 1];
  s[n++] = '.';
  int lo = 0;
  while (lo < nd - 1 && d[lo] == '0') ++lo;
  if (lo == nd - 1) s[n++] = '0';
  for (int k = nd - 2; k >= lo; --k) s[n++] = d[k];
  s[n++] = 'E';
  const int e = nd - 1;   // 7 .. 10
  if (e >= 10) s[n++] = (char)('0' + e / 10);
  s[n++] = (char)('0' + e % 10);
  return n;
}

// class numbering: flag[i] = element i is the first of its id; a row (the first n_rows elements) that is not is a duplicate
__global__ void k_model_class_flags(unsigned long long n, unsigned long long n_rows, const uint32_t *__restrict__ rep,
                                    uint32_t *__restrict__ flag, int *__restrict__ dup_row) {
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
    const bool first = rep[i] == (uint32_t)i;
    flag[i] = first ? 1u : 0u;
    if (i < n_rows && !first) *dup_row = 1;
  }
}
// class c's first element
__global__ void k_model_class_elem(unsigned long long n, const uint32_t *__restrict__ rep, const uint32_t *__restrict__ cpos,
                                   uint32_t *__restrict__ cls_elem) {
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x)
    if (rep[i] == (uint32_t)i) cls_elem[cpos[i]] = (uint32_t)i;
}
// prop_of[class of property id k] = k (prop_of starts at kNoProp); a class that already has one is a duplicate property id
__global__ void k_model_props(unsigned long long n_prop, unsigned long long base, const uint32_t *__restrict__ rep,
                              const uint32_t *__restrict__ cpos, uint32_t *__restrict__ prop_of, int *__restrict__ dup_prop) {
  for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < n_prop; k += (unsigned long long)gridDim.x * blockDim.x) {
    const uint32_t c = cpos[rep[base + k]];
    if (atomicCAS(&prop_of[c], kNoProp, (uint32_t)k) != kNoProp) *dup_prop = 1;
  }
}

// The events of one ranking: event e has class cpos[rep[e]] (rep offset to the ranking's first element) and time t_ms[e].
// counts[b][class] += 1 for the bucket b that holds t (buckets are disjoint), totals[b] = events per bucket.  The ranking's
// items are Zipf-distributed, so the lanes of a warp that hit the same (bucket, class) are aggregated first
// (__match_any_sync, as k_col_histogram_flat) and only their leader adds: the hot classes take one atomic per warp.
__global__ void k_rank_count(long long n, const uint32_t *__restrict__ rep, const uint32_t *__restrict__ cpos,
                             const long long *__restrict__ t_ms, const PopArgs a, int32_t *__restrict__ counts,
                             unsigned long long *__restrict__ totals) {
  const int lane = threadIdx.x & 31;
  unsigned long long mine[3] = {0, 0, 0};
  for (long long q0 = blockIdx.x * (long long)blockDim.x + (threadIdx.x & ~31); q0 < n; q0 += (long long)gridDim.x * blockDim.x) {
    const long long q = q0 + lane;
    int b = -1;
    uint32_t c = 0;
    if (q < n) {
      const long long t = t_ms[q];
#pragma unroll
      for (int k = 0; k < 3; ++k)
        if (k < a.n_buckets && t >= a.edge[k] && t < a.edge[k + 1]) b = k;
      if (b >= 0) c = cpos[rep[q]];
    }
    const unsigned om = __ballot_sync(0xffffffffu, b >= 0);
    if (b >= 0) {
      const unsigned long long key = (unsigned long long)b * (uint32_t)a.n_items + c;
      const unsigned peers = __match_any_sync(om, key);
      if ((__ffs(peers) - 1) == lane) atomicAdd(&counts[key], __popc(peers));
#pragma unroll
      for (int k = 0; k < 3; ++k) mine[k] += k == b;
    }
  }
  for (int k = 0; k < 3; ++k) {
    unsigned long long v = mine[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0 && v) atomicAdd(&totals[k], v);
  }
}

struct ModelArgs {
  FormatArgs f;                     // f.n_rows indicator rows = the first documents; f.row_ids = escaped ids of ALL documents
  long long n_docs;
  int n_rank;
  const uint32_t *doc_cls;          // [n_docs] class of each document
  const double *score[kMaxRankings];             // [n_classes] per ranking
  const unsigned char *present[kMaxRankings];    // [n_classes] per ranking
  const unsigned char *rank_names;               // escaped, concatenated
  int32_t rank_name_off[kMaxRankings + 1];
  const uint32_t *prop_of;          // [n_classes] property index or kNoProp
  DevDict frag;                     // property fragments, verbatim
};

// class c is a document: a row, or an id with a present rank or a property entry.  flag[n_classes] is the scan's tail.
__global__ void k_model_doc_flags(const ModelArgs a, uint32_t n_classes, uint32_t *__restrict__ flag) {
  for (uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; c < n_classes; c += gridDim.x * blockDim.x) {
    bool doc = c < (uint32_t)a.f.n_rows || a.prop_of[c] != kNoProp;
    for (int r = 0; r < a.n_rank; ++r) doc = doc || a.present[r][c];
    flag[c] = doc ? 1u : 0u;
  }
}
// document dpos[c] = class c, its id = the class's first element
__global__ void k_model_doc_list(uint32_t n_classes, const uint32_t *__restrict__ flag, const uint32_t *__restrict__ dpos,
                                 const uint32_t *__restrict__ cls_elem, uint32_t *__restrict__ doc_cls, uint32_t *__restrict__ doc_src) {
  for (uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; c < n_classes; c += gridDim.x * blockDim.x)
    if (flag[c]) {
      doc_cls[dpos[c]] = c;
      doc_src[dpos[c]] = cls_elem[c];
    }
}

// Bytes of document d:  {"index":{"_id":"<id>"}}\n{"id":"<id>"  [indicator fields, rows only]  ,"<rank>":<score> per present
// rank  ,<fragment> if non-empty  }\n
__global__ void k_model_doc_len(const ModelArgs a, long long *__restrict__ doc_len) {
  for (long long d = blockIdx.x * (long long)blockDim.x + threadIdx.x; d < a.n_docs; d += (long long)gridDim.x * blockDim.x) {
    const long long idl = a.f.row_ids.off[d + 1] - a.f.row_ids.off[d];
    long long len = 17 + idl + 11 + idl + 1 + 2;
    if (d < a.f.n_rows) len += indicator_fields_len(a.f, (int)d);
    const uint32_t c = a.doc_cls[d];
    char num[24];
    for (int r = 0; r < a.n_rank; ++r)
      if (a.present[r][c]) len += (a.rank_name_off[r + 1] - a.rank_name_off[r]) + 4 + java_double_integral(a.score[r][c], num);
    const uint32_t k = a.prop_of[c];
    if (k != kNoProp) {
      const long long fl = a.frag.off[k + 1] - a.frag.off[k];
      if (fl > 0) len += 1 + fl;
    }
    doc_len[d] = len;
  }
}
__global__ void k_model_doc_write(const ModelArgs a, const long long *__restrict__ doc_off, unsigned char *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long d = warp; d < a.n_docs; d += nwarps) {
    const unsigned char *id = a.f.row_ids.bytes + a.f.row_ids.off[d];
    const long long idl = a.f.row_ids.off[d + 1] - a.f.row_ids.off[d];
    unsigned char *w = out + doc_off[d];
    warp_lit(w, "{\"index\":{\"_id\":\"", 17, lane); w += 17;
    warp_copy(w, id, idl, lane); w += idl;
    warp_lit(w, "\"}}\n{\"id\":\"", 11, lane); w += 11;
    warp_copy(w, id, idl, lane); w += idl;
    warp_lit(w, "\"", 1, lane); w += 1;
    if (d < a.f.n_rows) w = warp_indicator_fields(a.f, (int)d, w, lane);
    const uint32_t c = a.doc_cls[d];
    for (int r = 0; r < a.n_rank; ++r) {
      if (!a.present[r][c]) continue;
      const int nl = a.rank_name_off[r + 1] - a.rank_name_off[r];
      warp_lit(w, ",\"", 2, lane); w += 2;
      warp_copy(w, a.rank_names + a.rank_name_off[r], nl, lane); w += nl;
      warp_lit(w, "\":", 2, lane); w += 2;
      char num[24];
      const int ln = java_double_integral(a.score[r][c], num);
      warp_lit(w, num, ln, lane); w += ln;
    }
    const uint32_t k = a.prop_of[c];
    if (k != kNoProp) {
      const long long fl = a.frag.off[k + 1] - a.frag.off[k];
      if (fl > 0) {
        warp_lit(w, ",", 1, lane); w += 1;
        warp_copy(w, a.frag.bytes + a.frag.off[k], fl, lane); w += fl;
      }
    }
    warp_lit(w, "}\n", 2, lane);
    __syncwarp();
  }
}

}  // namespace cco
