// cco_format.cuh -- SURVEY.md 8f-2: the indicator model as the Elasticsearch bulk body, assembled on the device.
//
// Reference (what this replaces, per item of the primary event):
//   IndexedDatasetConversions.toStringMapRDD   /root/reference/src/main/scala/package.scala:82-110
//       row -> non-zeros sorted by -LLR -> column id STRINGS (the LLR values are dropped); empty rows give an empty JArray
//   URModel.save: groupAll + ("id" -> itemId)    /root/reference/src/main/scala/URModel.scala:47-84, 87-102
//   EsClient.hotSwap: saveToEs(.., "es.mapping.id" -> "id")   /root/reference/src/main/scala/EsClient.scala:300-313
// One document per primary item, one keyword-array field per event name.  As elasticsearch-hadoop sends it:
//   {"index":{"_id":"<item>"}}\n
//   {"id":"<item>","<event 0>":["<col>","<col>",...],"<event 1>":[...]}\n
// The indicator rows arrive already ordered (llr desc, col asc), so the consumer's sortBy(-llr) is a no-op and the
// formatter only concatenates: dictionary strings are JSON-escaped once, then every document is a gather of byte ranges.
// HBM-bound byte work: two passes (lengths -> exclusive scan -> bytes), one warp per document.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace cco {

struct DevDict {            // id i = bytes[off[i] .. off[i + 1])
  const long long *off;
  const unsigned char *bytes;
  long long n;
};

// JSON string escaping (RFC 8259 minimum): '"' -> \" , '\\' -> \\\\ , bytes < 0x20 -> \u00xx (lower-case hex); everything
// else (UTF-8 included) passes through.  Same rule in the CPU restatement (oracle/format_oracle.py).
__device__ __forceinline__ int json_escaped_len(unsigned char ch) { return ch == '"' || ch == '\\' ? 2 : (ch < 0x20 ? 6 : 1); }

__global__ void k_escape_len(long long n, const long long *__restrict__ off, const unsigned char *__restrict__ bytes,
                             long long *__restrict__ out_len) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    long long len = 0;
    for (long long q = off[i]; q < off[i + 1]; ++q) len += json_escaped_len(bytes[q]);
    out_len[i] = len;
  }
}
__global__ void k_escape_write(long long n, const long long *__restrict__ off, const unsigned char *__restrict__ bytes,
                               const long long *__restrict__ out_off, unsigned char *__restrict__ out) {
  const char hex[] = "0123456789abcdef";
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    long long w = out_off[i];
    for (long long q = off[i]; q < off[i + 1]; ++q) {
      const unsigned char ch = bytes[q];
      if (ch == '"' || ch == '\\') {
        out[w++] = '\\';
        out[w++] = ch;
      } else if (ch < 0x20) {
        out[w++] = '\\'; out[w++] = 'u'; out[w++] = '0'; out[w++] = '0';
        out[w++] = hex[ch >> 4];
        out[w++] = hex[ch & 15];
      } else {
        out[w++] = ch;
      }
    }
  }
}

constexpr int kMaxFormatIndicators = 16;
struct FormatArgs {
  int32_t n_rows;          // documents = rows [0, n_rows) of every indicator (a rank's slice or the whole model)
  long long row_id_base;   // global item index of row 0 (the row dictionary is global)
  int32_t n_ind;
  DevDict row_ids;                              // escaped
  DevDict col_ids[kMaxFormatIndicators];        // escaped
  const long long *row_ptr[kMaxFormatIndicators];
  const int32_t *col[kMaxFormatIndicators];
  const unsigned char *names;                   // escaped event names, concatenated
  int32_t name_off[kMaxFormatIndicators + 1];
};

// {"index":{"_id":"  = 17 bytes ; "}}\n{"id":"  = 11 ; closing quote of the id = 1 ; per field  ,"name":[  = name + 5 and ] = 1 ;
// per element two quotes + a comma between elements ; }\n = 2
__device__ __forceinline__ long long indicator_fields_len(const FormatArgs &a, int r) {
  long long len = 0;
  for (int i = 0; i < a.n_ind; ++i) {
    len += (a.name_off[i + 1] - a.name_off[i]) + 5 + 1;
    const long long s = a.row_ptr[i][r], e = a.row_ptr[i][r + 1];
    for (long long q = s; q < e; ++q) {
      const int32_t c = a.col[i][q];
      len += a.col_ids[i].off[c + 1] - a.col_ids[i].off[c] + 2;
    }
    if (e > s) len += e - s - 1;
  }
  return len;
}
__global__ void k_doc_len(const FormatArgs a, long long *__restrict__ doc_len) {
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < a.n_rows; r += gridDim.x * blockDim.x) {
    const long long g = a.row_id_base + r;
    const long long idl = a.row_ids.off[g + 1] - a.row_ids.off[g];
    doc_len[r] = 17 + idl + 11 + idl + 1 + 2 + indicator_fields_len(a, r);
  }
}

__device__ __forceinline__ void warp_copy(unsigned char *dst, const unsigned char *src, long long n, int lane) {
  for (long long i = lane; i < n; i += 32) dst[i] = src[i];
}
__device__ __forceinline__ void warp_lit(unsigned char *dst, const char *lit, int n, int lane) {
  if (lane < n) dst[lane] = (unsigned char)lit[lane];
}

// the indicator fields of row r, written by the whole warp from w on: ,"<name>":["<col>",...] per indicator
__device__ __forceinline__ unsigned char *warp_indicator_fields(const FormatArgs &a, int r, unsigned char *w, int lane) {
  for (int i = 0; i < a.n_ind; ++i) {
    const int nl = a.name_off[i + 1] - a.name_off[i];
    warp_lit(w, ",\"", 2, lane); w += 2;
    warp_copy(w, a.names + a.name_off[i], nl, lane); w += nl;
    warp_lit(w, "\":[", 3, lane); w += 3;
    const long long s = a.row_ptr[i][r], e = a.row_ptr[i][r + 1];
    // elements: the lanes first agree on every element's offset inside the array (prefix sums of 32 at a time)
    for (long long q0 = s; q0 < e; q0 += 32) {
      const long long q = q0 + lane;
      long long el = 0;
      const unsigned char *src = nullptr;
      if (q < e) {
        const int32_t c = a.col[i][q];
        src = a.col_ids[i].bytes + a.col_ids[i].off[c];
        el = a.col_ids[i].off[c + 1] - a.col_ids[i].off[c];
      }
      long long mine = q < e ? el + 2 + (q > s ? 1 : 0) : 0;   // leading comma from the second element on
      long long incl = mine;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const long long v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
      }
      const long long total = __shfl_sync(0xffffffffu, incl, 31);
      if (q < e) {
        unsigned char *p = w + (incl - mine);
        if (q > s) *p++ = ',';
        *p++ = '"';
        for (long long k = 0; k < el; ++k) p[k] = src[k];   // ids are short (a few to a few dozen bytes)
        p[el] = '"';
      }
      w += total;
    }
    warp_lit(w, "]", 1, lane); w += 1;
  }
  return w;
}

// one warp per document: the lanes copy every byte range cooperatively; the write position advances uniformly
__global__ void k_doc_write(const FormatArgs a, const long long *__restrict__ doc_off, unsigned char *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int r = warp; r < a.n_rows; r += nwarps) {
    const long long g = a.row_id_base + r;
    const unsigned char *id = a.row_ids.bytes + a.row_ids.off[g];
    const long long idl = a.row_ids.off[g + 1] - a.row_ids.off[g];
    unsigned char *w = out + doc_off[r];
    warp_lit(w, "{\"index\":{\"_id\":\"", 17, lane); w += 17;
    warp_copy(w, id, idl, lane); w += idl;
    warp_lit(w, "\"}}\n{\"id\":\"", 11, lane); w += 11;
    warp_copy(w, id, idl, lane); w += idl;
    warp_lit(w, "\"", 1, lane); w += 1;
    w = warp_indicator_fields(a, r, w, lane);
    warp_lit(w, "}\n", 2, lane);
    __syncwarp();
  }
}

// ---- SURVEY.md 8f-3: PopModel rank histograms (/root/reference/src/main/scala/PopModel.scala:113-182) -----------------------
// popular  = events per item in [start, end)                                              (calcPopular :113-122)
// trending = newer half - older half, items present in BOTH halves; nothing if the older half is empty   (:128-148)
// hot      = (newer - middle) - (middle - older) over thirds, items present in all three buckets; nothing if the older or
//            the middle third is empty                                                                  (:153-182)
// Bucket edges follow the reference's Joda arithmetic: integer millisecond division, [start, end) intervals
// (PEventStore.find: startTime inclusive, untilTime exclusive).
struct PopArgs {
  long long edge[4];   // bucket b = [edge[b], edge[b + 1])
  int n_buckets;
  int32_t n_items;
};
__global__ void k_pop_count(long long n_events, const int32_t *__restrict__ item, const long long *__restrict__ t_ms, const PopArgs a,
                            int32_t *__restrict__ counts /* [n_buckets][n_items] */, unsigned long long *__restrict__ totals) {
  unsigned long long mine[3] = {0, 0, 0};
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_events; e += (long long)gridDim.x * blockDim.x) {
    const long long t = t_ms[e];
    const int32_t j = item[e];
    if ((uint32_t)j >= (uint32_t)a.n_items) continue;
#pragma unroll
    for (int b = 0; b < 3; ++b)
      if (b < a.n_buckets && t >= a.edge[b] && t < a.edge[b + 1]) {
        atomicAdd(&counts[(size_t)b * a.n_items + j], 1);
        ++mine[b];
      }
  }
  for (int b = 0; b < 3; ++b) {
    unsigned long long v = mine[b];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&totals[b], v);
  }
}
__global__ void k_pop_score(const PopArgs a, int mode, const int32_t *__restrict__ counts, const unsigned long long *__restrict__ totals,
                            double *__restrict__ score, unsigned char *__restrict__ present) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n_items; j += gridDim.x * blockDim.x) {
    const int32_t c0 = counts[j], c1 = a.n_buckets > 1 ? counts[(size_t)a.n_items + j] : 0,
                  c2 = a.n_buckets > 2 ? counts[(size_t)2 * a.n_items + j] : 0;
    double v = 0.0;
    bool ok = false;
    if (mode == 0) {          // popular
      ok = c0 > 0;
      v = (double)c0;
    } else if (mode == 1) {   // trending: buckets = (older, newer)
      ok = totals[0] > 0 && c0 > 0 && c1 > 0;
      v = (double)c1 - (double)c0;
    } else {                  // hot: buckets = (older, middle, newer)
      ok = totals[0] > 0 && totals[1] > 0 && c0 > 0 && c1 > 0 && c2 > 0;
      v = ((double)c2 - (double)c1) - ((double)c1 - (double)c0);
    }
    score[j] = ok ? v : 0.0;
    present[j] = ok ? 1 : 0;
  }
}

}  // namespace cco
