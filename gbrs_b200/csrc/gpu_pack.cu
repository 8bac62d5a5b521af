// Device-side packer: H x CSC(N x T) incidence (host arrays)  ->  the class-major + locus-major arrays of
// include/gbrs_em.h, built ON THE GPU.  Same inputs, same outputs -- array for array, bit for bit -- as the host packer
// gbrs_pack_create (pack.cpp), which stays as its oracle and as the path for inputs this one refuses.
//
// What it replaces in the reference: the storage walk of Sparse3DMatrix (src/gbrs/emase/Sparse3DMatrix.py:26-66, the CSC
// matrices are class-id lists per locus) re-laid for the two GPU passes; the `-G` restriction of quantify
// (src/gbrs/gbrs/emase_utils.py:247-273) is applied while counting.  The host packer costs 0.2 s at 5 M classes (16
// threads) -- a hundred times the EM it feeds; here the same work is a transposition by a stable radix sort of the stored
// entries, one linear merge per class, three radix sorts of 5-10 M keys and a handful of scans (11 ms at 5 M classes incl.
// the 293 MB over PCIe):
//
//   transpose  the stored entries that survive the haplotype mask, re-laid locus-major (k_gp_col_len, scan, k_gp_gen), are
//              stable-sorted by class id (cub::DeviceRadixSort, library); rowstart from the sorted keys (k_gp_rowstart).
//   merge      per class: OR the haplotype bits of equal loci (records arrive ordered) -> pair words, pair count, smallest loci
//   order      classes of this shard by (min(pairs, 9) - 1, smallest locus, second-smallest locus), stable   cub::DeviceRadixSort (library)
//   fill       rowptr / count / pairs in the new order, pairs sorted by (gene, locus), (class, gene) runs
//   loci       per-locus entry counts (partial / full masks), padded part sizes, item counts, their scans
//   entries    pairs sorted by (locus, part, new class id) -> ent_cls / ent_pair / ent_run        cub::DeviceRadixSort
//   items      item_off, visiting order (kind, longest first), item_desc; loci deepest first, locus_desc
//   interleave lane-interleaved entry order inside every work item
//
// The library owns no device memory: every buffer comes from the caller's allocator (a PyTorch tensor per request).
#include <cuda_runtime.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "gbrs_em.h"

void gbrs_set_error(const std::string& s);  // em_kernels.cu

#define GP_CUDA(call)                                                                                \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess) {                                                                         \
      gbrs_set_error(std::string("gbrs_pack_device: ") + #call + ": " + cudaGetErrorString(e_));     \
      return GBRS_E_CUDA;                                                                            \
    }                                                                                                \
  } while (0)

namespace {

constexpr int kGpThreads = 256;
constexpr uint32_t kLoc = 0xFFFFFFu;

inline int gp_grid(int64_t threads, int cap = 148 * 16) {
  int64_t b = (threads + kGpThreads - 1) / kGpThreads;
  if (b > cap) b = cap;
  return (int) (b < 1 ? 1 : b);
}

struct Columns {            // the H CSC matrices on the device
  const int64_t* indptr;    // [H][T + 1]
  const uint32_t* indices;  // all haplotypes back to back (class ids, narrowed to 32 bits)
  int64_t hoff[GBRS_HPAD];  // first entry of haplotype h in `indices`
  const uint8_t* hapmask;   // [T] or null
  int32_t T, H;
  int64_t N;
};

__global__ void __launch_bounds__(kGpThreads) k_gp_narrow(const int64_t* __restrict__ in, uint32_t* __restrict__ out, int64_t n,
                                                         int64_t N, int* bad) {
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
    const int64_t v = in[i];
    if (v < 0 || v >= N) *bad = 1;
    out[i] = (uint32_t) v;
  }
}

// ---- transposition by sorting: the stored entries, re-laid locus-major, are stable-sorted by class id ----------------
// column lengths in [locus][haplotype] order after the haplotype mask
__global__ void __launch_bounds__(kGpThreads) k_gp_col_len(const Columns c, uint32_t* __restrict__ len) {
  const int64_t n_cols = (int64_t) c.H * c.T;
  for (int64_t q = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; q < n_cols; q += (int64_t) gridDim.x * blockDim.x) {
    const int t = (int) (q / c.H), h = (int) (q - (int64_t) t * c.H);
    const int64_t* ip = c.indptr + (int64_t) h * (c.T + 1) + t;
    const bool keep = !c.hapmask || ((c.hapmask[t] >> h) & 1);
    len[q] = keep ? (uint32_t) (ip[1] - ip[0]) : 0u;
  }
}
// one warp per (locus, haplotype) column: key = class id, value = (locus << 3 | haplotype), written at the column's place
// in locus-major order -- a stable sort by class then leaves every class' records ordered by (locus, haplotype)
__global__ void __launch_bounds__(kGpThreads) k_gp_gen(const Columns c, const uint32_t* __restrict__ colstart,
                                                      uint32_t* __restrict__ keys, uint32_t* __restrict__ vals, int* bad) {
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t) gridDim.x * blockDim.x) >> 5, n_cols = (int64_t) c.H * c.T;
  for (int64_t q = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; q < n_cols; q += n_warps) {
    const uint32_t o = colstart[q], n = colstart[q + 1] - o;
    if (n == 0) continue;
    const int t = (int) (q / c.H), h = (int) (q - (int64_t) t * c.H);
    const uint32_t* src = c.indices + c.hoff[h] + c.indptr[(int64_t) h * (c.T + 1) + t];
    const uint32_t v = ((uint32_t) t << 3) | (uint32_t) h;
    for (uint32_t i = lane; i < n; i += 32) {
      uint32_t cls = src[i];
      if ((int64_t) cls >= c.N) { *bad = 1; cls = 0u; }
      keys[o + i] = cls;
      vals[o + i] = v;
    }
  }
}
// rowstart[c] = first record of class c in the sorted list (n for the classes behind the last one; rowstart[N] = n)
__global__ void __launch_bounds__(kGpThreads) k_gp_rowstart(const uint32_t* __restrict__ keys, int64_t n, int64_t N,
                                                           uint32_t* __restrict__ rowstart) {
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += (int64_t) gridDim.x * blockDim.x) {
    const int64_t prev = i > 0 ? (int64_t) keys[i - 1] : -1, cur = i < n ? (int64_t) keys[i] : N;
    for (int64_t x = prev + 1; x <= cur; ++x) rowstart[x] = (uint32_t) i;
  }
}

// per class: records (locus << 3 | hap) -> pair words (locus | mask << 24), compacted at the front of the class' segment;
// the records of a class come ordered by (locus, haplotype) from the transposition by sorting
__global__ void __launch_bounds__(kGpThreads) k_gp_merge(int64_t N, const uint32_t* __restrict__ rowstart,
                                                        uint32_t* __restrict__ rec,
                                                        uint32_t* __restrict__ npair, uint32_t* __restrict__ minloc,
                                                        uint32_t* __restrict__ secloc) {
  for (int64_t c = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; c < N; c += (int64_t) gridDim.x * blockDim.x) {
    const int n = (int) (rowstart[c + 1] - rowstart[c]);
    uint32_t* a = rec + rowstart[c];
    if (n == 0) { npair[c] = 0; minloc[c] = 0xFFFFFFFFu; secloc[c] = 0u; continue; }
    int k = 0;
    for (int i = 0; i < n;) {
      const uint32_t t = a[i] >> 3;
      uint32_t m = 0;
      for (; i < n && (a[i] >> 3) == t; ++i) m |= 1u << (a[i] & 7u);
      a[k++] = t | (m << 24);
    }
    npair[c] = (uint32_t) k;
    minloc[c] = a[0] & kLoc;
    secloc[c] = k > 1 ? (a[1] & kLoc) : 0u;  // second-smallest locus (> 0 when there is one): the minor key of the class order
  }
}

// shard boundaries balanced by nnz: class c belongs to shard min(R - 1, rowstart[c] * R / total)   (pack.cpp step 2)
__global__ void k_gp_shard(const uint32_t* __restrict__ rowstart, int64_t N, int R, int rank, int64_t* lohi) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const uint64_t total = rowstart[N];
  auto shard_of = [&](int64_t c) -> int {
    if (total == 0) return 0;
    const uint64_t r = (uint64_t) rowstart[c] * (uint64_t) R / total;
    return (int) (r < (uint64_t) (R - 1) ? r : (uint64_t) (R - 1));
  };
  auto first_with = [&](int want_ge) {  // smallest c with shard_of(c) >= want_ge (N if none)
    int64_t a = 0, b = N;
    while (a < b) {
      const int64_t m = (a + b) >> 1;
      if (shard_of(m) >= want_ge) b = m; else a = m + 1;
    }
    return a;
  };
  int64_t lo = 0, hi = N;
  if (R > 1) {
    lo = first_with(rank);
    hi = first_with(rank + 1);
    if (hi < lo) hi = lo;
  }
  lohi[0] = lo;
  lohi[1] = hi;
}

__global__ void __launch_bounds__(kGpThreads) k_gp_order_keys(int64_t N, const int64_t* __restrict__ lohi,
                                                             const uint32_t* __restrict__ npair,
                                                             const uint32_t* __restrict__ minloc, uint32_t* __restrict__ key,
                                                             uint32_t* __restrict__ val, unsigned long long* __restrict__ stats) {
  // stats: [0] non-empty classes over all shards, [1] max pairs per class in this shard
  unsigned long long nonempty = 0, maxk = 0;
  for (int64_t c = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; c < N; c += (int64_t) gridDim.x * blockDim.x) {
    const uint32_t k = npair[c];
    nonempty += k > 0;
    const bool mine = k > 0 && c >= lohi[0] && c < lohi[1];
    if (mine && k > maxk) maxk = k;
    const uint32_t bucket = (k < (uint32_t) GBRS_KMAX + 1u ? k : (uint32_t) GBRS_KMAX + 1u) - 1u;
    key[c] = mine ? ((bucket << 24) | minloc[c]) : 0xFFFFFFFFu;
    val[c] = (uint32_t) c;
  }
  for (int o = 16; o > 0; o >>= 1) {
    nonempty += __shfl_xor_sync(0xFFFFFFFFu, nonempty, o);
    const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, maxk, o);
    maxk = other > maxk ? other : maxk;
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(stats, nonempty);
    atomicMax(stats + 1, maxk);
  }
}

// bucket boundaries from the sorted keys: first position whose key >= (b << 24); [10] = number of valid classes
__global__ void k_gp_buckets(const uint32_t* __restrict__ sorted_key, int64_t N, int64_t* bucket_class0) {
  const int b = threadIdx.x;
  if (b > GBRS_KMAX + 1) return;
  const uint32_t want = b <= GBRS_KMAX ? ((uint32_t) b << 24) : 0xFFFFFFFFu;
  int64_t lo = 0, hi = N;
  while (lo < hi) {
    const int64_t m = (lo + hi) >> 1;
    if (sorted_key[m] >= want) hi = m; else lo = m + 1;
  }
  bucket_class0[b] = lo;
}

__global__ void __launch_bounds__(kGpThreads) k_gp_gather_u32(int64_t n, const uint32_t* __restrict__ order,
                                                             const uint32_t* __restrict__ src, uint32_t* __restrict__ dst) {
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) dst[i] = src[order[i]];
}

// per new class: copy its pair words, sort by (gene, locus), number its (class, gene) runs, carry the count over
__global__ void __launch_bounds__(kGpThreads) k_gp_fill_classes(int64_t n_classes, const uint32_t* __restrict__ order,
                                                               const uint32_t* __restrict__ rowstart,
                                                               const uint32_t* __restrict__ rec, const uint32_t* __restrict__ rowptr,
                                                               const int32_t* __restrict__ gene_of, const double* __restrict__ count_in,
                                                               uint32_t* __restrict__ pairs, uint32_t* __restrict__ ric,
                                                               uint32_t* __restrict__ nruns, double* __restrict__ count_out) {
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n_classes; i += (int64_t) gridDim.x * blockDim.x) {
    const uint32_t c = order[i];
    const uint32_t* src = rec + rowstart[c];
    uint32_t* dst = pairs + rowptr[i];
    const int k = (int) (rowptr[i + 1] - rowptr[i]);
    auto keyof = [&](uint32_t w) { return ((uint64_t) (uint32_t) gene_of[w & kLoc] << 24) | (w & kLoc); };
    for (int j = 0; j < k; ++j) {  // insertion sort while copying (input ascending in locus: genes mostly ascending too)
      const uint32_t w = src[j];
      const uint64_t key = keyof(w);
      int q = j - 1;
      for (; q >= 0 && keyof(dst[q]) > key; --q) dst[q + 1] = dst[q];
      dst[q + 1] = w;
    }
    uint32_t runs = k > 0 ? 1u : 0u;
    uint32_t* r = ric + rowptr[i];
    if (k > 0) r[0] = 0;
    for (int j = 1; j < k; ++j) {
      runs += gene_of[dst[j] & kLoc] != gene_of[dst[j - 1] & kLoc];
      r[j] = runs - 1;
    }
    nruns[i] = runs;
    count_out[i] = count_in ? count_in[c] : 1.0;
  }
}

__global__ void __launch_bounds__(kGpThreads) k_gp_locus_counts(int64_t n_pairs, const uint32_t* __restrict__ pairs, uint32_t full,
                                                               uint32_t* __restrict__ lcnt, uint32_t* __restrict__ lpart_raw) {
  for (int64_t p = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; p < n_pairs; p += (int64_t) gridDim.x * blockDim.x) {
    const uint32_t w = pairs[p];
    atomicAdd(lcnt + (w & kLoc), 1u);
    if ((w >> 24) != full) atomicAdd(lpart_raw + (w & kLoc), 1u);
  }
}

struct ItemRule {  // pack.cpp step 6
  int64_t item_len, long_len;
  __host__ __device__ int64_t len_of(int64_t len) const {
    if (len <= 8 * item_len) return item_len;
    const int64_t n = (len + long_len - 1) / long_len;
    return ((len + n - 1) / n + 31) / 32 * 32;
  }
  __host__ __device__ int64_t items_of(int64_t len) const { return len ? (len + len_of(len) - 1) / len_of(len) : 0; }
};

__global__ void __launch_bounds__(kGpThreads) k_gp_locus_geometry(int T, ItemRule rule, const uint32_t* __restrict__ lcnt,
                                                                 const uint32_t* __restrict__ lpart_raw, uint32_t* __restrict__ lpart,
                                                                 uint32_t* __restrict__ ppart, uint32_t* __restrict__ lsize,
                                                                 uint32_t* __restrict__ nitems) {
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < T; t += gridDim.x * blockDim.x) {
    const int64_t cnt = lcnt[t];
    const bool split = cnt > 8 * rule.item_len;
    const int64_t part = split ? (int64_t) lpart_raw[t] : cnt;
    const int64_t pp = (part + 3) / 4 * 4, pf = (cnt - part + 3) / 4 * 4;
    lpart[t] = (uint32_t) part;
    ppart[t] = (uint32_t) pp;
    lsize[t] = (uint32_t) (pp + pf);
    nitems[t] = (uint32_t) (rule.items_of(pp) + rule.items_of(pf));
  }
}

__global__ void __launch_bounds__(kGpThreads) k_gp_entry_keys(int64_t n_classes, const uint32_t* __restrict__ rowptr,
                                                             const uint32_t* __restrict__ pairs, const uint32_t* __restrict__ lcnt,
                                                             ItemRule rule, uint32_t full, unsigned long long* __restrict__ key,
                                                             uint32_t* __restrict__ val) {
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n_classes; i += (int64_t) gridDim.x * blockDim.x) {
    for (uint32_t p = rowptr[i]; p < rowptr[i + 1]; ++p) {
      const uint32_t w = pairs[p], t = w & kLoc;
      const unsigned long long part = ((int64_t) lcnt[t] > 8 * rule.item_len && (w >> 24) == full) ? 1ull : 0ull;
      key[p] = ((unsigned long long) t << 32) | (part << 31) | (unsigned long long) i;
      val[p] = p;
    }
  }
}

template <typename E>
__global__ void __launch_bounds__(kGpThreads) k_gp_fill_pad(int64_t n, E* a, E* b, E* c, E va, E vb, E vc) {
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
    a[i] = va;
    b[i] = vb;
    c[i] = vc;
  }
}

template <typename E>
__global__ void __launch_bounds__(kGpThreads) k_gp_fill_entries(int64_t n_pairs, const unsigned long long* __restrict__ key,
                                                               const uint32_t* __restrict__ val, const uint32_t* __restrict__ pairs,
                                                               const uint32_t* __restrict__ lptr, const uint32_t* __restrict__ lstart,
                                                               const uint32_t* __restrict__ lpart, const uint32_t* __restrict__ ppart,
                                                               const uint32_t* __restrict__ runptr, const uint32_t* __restrict__ ric,
                                                               E* __restrict__ ent_cls, E* __restrict__ ent_pair, E* __restrict__ ent_run) {
  constexpr int SH = 8 * (int) sizeof(E) - 8;
  for (int64_t j = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; j < n_pairs; j += (int64_t) gridDim.x * blockDim.x) {
    const unsigned long long k = key[j];
    const uint32_t t = (uint32_t) (k >> 32), part = (uint32_t) ((k >> 31) & 1u), i = (uint32_t) (k & 0x7FFFFFFFu);
    const uint32_t p = val[j];
    const E m = (E) (pairs[p] >> 24) << SH;
    const int64_t pos = (int64_t) lptr[t] + (part ? ppart[t] : 0u) + (j - (int64_t) lstart[t] - (part ? lpart[t] : 0u));
    ent_cls[pos] = (E) i | m;
    ent_pair[pos] = (E) p | m;
    ent_run[pos] = (E) (runptr[i] + ric[p]) | m;
  }
}

// item_off / item_full of every locus' items (pack.cpp step 6)
__global__ void __launch_bounds__(kGpThreads) k_gp_items(int T, ItemRule rule, const uint32_t* __restrict__ lptr,
                                                        const uint32_t* __restrict__ ppart, const uint32_t* __restrict__ lsize,
                                                        const uint32_t* __restrict__ item_ptr, uint32_t* __restrict__ item_off,
                                                        uint8_t* __restrict__ item_full) {
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < T; t += gridDim.x * blockDim.x) {
    uint32_t it = item_ptr[t];
    const int64_t np = ppart[t], nf = (int64_t) lsize[t] - np;
    const int64_t ilp = rule.len_of(np), ilf = rule.len_of(nf);
    for (int64_t o = 0; o < np; o += ilp) { item_full[it] = 0; item_off[it++] = (uint32_t) (lptr[t] + o); }
    for (int64_t o = 0; o < nf; o += ilf) { item_full[it] = 1; item_off[it++] = (uint32_t) (lptr[t] + np + o); }
  }
}

__global__ void __launch_bounds__(kGpThreads) k_gp_item_keys(int64_t n_items, int64_t item_len, const uint32_t* __restrict__ item_off,
                                                            const uint8_t* __restrict__ item_full, uint32_t* __restrict__ key,
                                                            uint32_t* __restrict__ val) {
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += (int64_t) gridDim.x * blockDim.x) {
    const uint32_t len = item_off[i + 1] - item_off[i];
    const uint32_t kind = ((int64_t) len > item_len ? 0u : 2u) + item_full[i];
    key[i] = (kind << 28) | (0x0FFFFFFFu - len);  // kind ascending, then longest first; the sort is stable in the item id
    val[i] = (uint32_t) i;
  }
}

__global__ void __launch_bounds__(kGpThreads) k_gp_item_desc(int64_t n_items, const uint32_t* __restrict__ sorted_key,
                                                            const uint32_t* __restrict__ sorted_item,
                                                            const uint32_t* __restrict__ item_off, const uint8_t* __restrict__ item_full,
                                                            uint32_t* __restrict__ item_desc, unsigned long long* n_long,
                                                            unsigned long long* __restrict__ cls /* [5] size classes */) {
  unsigned long long mine = 0, c[5] = {0, 0, 0, 0, 0};  // short partial: all, > 8 words, > 4 words; short full: > 8, > 4
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += (int64_t) gridDim.x * blockDim.x) {
    const uint32_t it = sorted_item[i];
    const uint32_t b = item_off[it], e = item_off[it + 1], kind = sorted_key[i] >> 28, f = item_full[it];
    item_desc[4 * i + 0] = b;
    item_desc[4 * i + 1] = e;
    item_desc[4 * i + 2] = it;
    item_desc[4 * i + 3] = f;
    mine += kind < 2u;
    if (kind >= 2u) {
      c[0] += !f;
      c[f ? 3 : 1] += e - b > 8u;
      c[f ? 4 : 2] += e - b > 4u;
    }
  }
  if (mine) atomicAdd(n_long, mine);
  for (int k = 0; k < 5; ++k)
    if (c[k]) atomicAdd(cls + k, c[k]);
}

// the trailer of item_desc (see k_column_reduce): positions where the short items change kind / size class
__global__ void k_gp_item_trailer(int64_t n_items, const unsigned long long* __restrict__ n_long,
                                  const unsigned long long* __restrict__ cls, uint32_t* __restrict__ item_desc) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const unsigned long long nl = *n_long, f0 = nl + cls[0];
  uint32_t* tr = item_desc + 4 * n_items;
  tr[0] = (uint32_t) (nl + cls[1]);
  tr[1] = (uint32_t) (nl + cls[2]);
  tr[2] = (uint32_t) f0;
  tr[3] = (uint32_t) (f0 + cls[3]);
  tr[4] = (uint32_t) (f0 + cls[4]);
  tr[5] = tr[6] = tr[7] = 0u;
}

__global__ void __launch_bounds__(kGpThreads) k_gp_locus_keys(int T, const uint32_t* __restrict__ nitems, uint32_t* __restrict__ key,
                                                             uint32_t* __restrict__ val) {
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < T; t += gridDim.x * blockDim.x) {
    key[t] = 0xFFFFFFFFu - nitems[t];
    val[t] = (uint32_t) t;
  }
}

__global__ void __launch_bounds__(kGpThreads) k_gp_locus_desc(int T, const uint32_t* __restrict__ sorted_locus,
                                                             const uint32_t* __restrict__ item_ptr, uint32_t* __restrict__ locus_desc,
                                                             unsigned long long* n_deep) {
  unsigned long long mine = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < T; i += gridDim.x * blockDim.x) {
    const uint32_t t = sorted_locus[i];
    locus_desc[4 * i + 0] = t;
    locus_desc[4 * i + 1] = item_ptr[t];
    locus_desc[4 * i + 2] = item_ptr[t + 1];
    locus_desc[4 * i + 3] = 0;
    mine += item_ptr[t + 1] - item_ptr[t] > (uint32_t) GBRS_DEEP_LOCUS_ITEMS;
  }
  if (mine) atomicAdd(n_deep, mine);
}

// lane-interleaved entry order inside every work item (pack.cpp step 6b), out of place: one thread per entry word
template <typename E>
__global__ void __launch_bounds__(kGpThreads) k_gp_interleave(int64_t n_items, int64_t item_len, const uint32_t* __restrict__ item_off,
                                                             const E* __restrict__ a0, const E* __restrict__ b0, const E* __restrict__ c0,
                                                             E* __restrict__ a1, E* __restrict__ b1, E* __restrict__ c1) {
  const int lane = threadIdx.x & 31;
  const int64_t n_warps = ((int64_t) gridDim.x * blockDim.x) >> 5;
  for (int64_t it = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; it < n_items; it += n_warps) {
    const int64_t b = item_off[it], e = item_off[it + 1];
    const int64_t B = (e - b > item_len) ? 128 : 32;
    for (int64_t k = b; k < e; k += B) {
      const int64_t m = (B < e - k) ? B : e - k, nq = m / 4;
      for (int64_t r = lane; r < m; r += 32) {
        const int64_t dst = k + 4 * (r % nq) + r / nq;
        a1[dst] = a0[k + r];
        b1[dst] = b0[k + r];
        c1[dst] = c0[k + r];
      }
    }
  }
}

struct Arena {  // every request goes to the caller's allocator
  gbrs_alloc_fn fn;
  void* user;
  bool failed = false;
  template <typename T>
  T* get(int64_t n, const char* tag) {
    void* p = fn((n > 0 ? n : 1) * (int64_t) sizeof(T), tag, user);
    if (!p) failed = true;
    return static_cast<T*>(p);
  }
};

template <typename In, typename Out>
int inclusive_scan_into(Arena& A, const In* in, Out* out, int64_t n, cudaStream_t s) {
  size_t bytes = 0;
  GP_CUDA(cub::DeviceScan::InclusiveSum(nullptr, bytes, in, out, n));
  void* tmp = A.get<uint8_t>((int64_t) bytes, "tmp:scan");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  GP_CUDA(cub::DeviceScan::InclusiveSum(tmp, bytes, in, out, n, s));
  return GBRS_OK;
}

template <typename K, typename V>
int sort_pairs(Arena& A, const K* kin, K* kout, const V* vin, V* vout, int64_t n, int end_bit, cudaStream_t s) {
  size_t bytes = 0;
  GP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, kin, kout, vin, vout, n, 0, end_bit));
  void* tmp = A.get<uint8_t>((int64_t) bytes, "tmp:sort");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  GP_CUDA(cub::DeviceRadixSort::SortPairs(tmp, bytes, kin, kout, vin, vout, n, 0, end_bit, s));
  return GBRS_OK;
}

template <typename T>
int read_back(const T* dev, T* host, int64_t n, cudaStream_t s) {
  GP_CUDA(cudaMemcpyAsync(host, dev, sizeof(T) * (size_t) n, cudaMemcpyDeviceToHost, s));
  GP_CUDA(cudaStreamSynchronize(s));
  return GBRS_OK;
}

template <typename E>
int build_entries(Arena& A, cudaStream_t s, int64_t n_pairs, int64_t n_entries, int64_t n_items, int64_t n_classes, int64_t n_runs,
                  int64_t item_len, const unsigned long long* skey, const uint32_t* sval, const uint32_t* pairs,
                  const uint32_t* lptr, const uint32_t* lstart, const uint32_t* lpart, const uint32_t* ppart,
                  const uint32_t* runptr, const uint32_t* ric, const uint32_t* item_off, gbrs_device_pack* out) {
  constexpr int SH = 8 * (int) sizeof(E) - 8;
  (void) SH;
  E* a = A.get<E>(n_entries, "tmp:ent_cls");
  E* b = A.get<E>(n_entries, "tmp:ent_pair");
  E* c = A.get<E>(n_entries, "tmp:ent_run");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  if (n_entries > 0) {
    k_gp_fill_pad<E><<<gp_grid(n_entries), kGpThreads, 0, s>>>(n_entries, a, b, c, (E) n_classes, (E) n_pairs, (E) n_runs);
    if (n_pairs > 0)
      k_gp_fill_entries<E><<<gp_grid(n_pairs), kGpThreads, 0, s>>>(n_pairs, skey, sval, pairs, lptr, lstart, lpart, ppart, runptr, ric, a,
                                                                 b, c);
  }
  E* a1 = A.get<E>(n_entries, "ent_cls");
  E* b1 = A.get<E>(n_entries, "ent_pair");
  E* c1 = A.get<E>(n_entries, "ent_run");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  if (n_items > 0)
    k_gp_interleave<E><<<gp_grid(n_items * 32), kGpThreads, 0, s>>>(n_items, item_len, item_off, a, b, c, a1, b1, c1);
  GP_CUDA(cudaGetLastError());
  out->ent_cls = a1;
  out->ent_pair = b1;
  out->ent_run = c1;
  return GBRS_OK;
}

}  // namespace

extern "C" int gbrs_pack_device(const gbrs_pack_input* in, gbrs_alloc_fn alloc, void* user, void* stream, gbrs_pack_info* info_out,
                                gbrs_device_pack* out) {
  if (!in || !alloc || !info_out || !out) { gbrs_set_error("gbrs_pack_device: null argument"); return GBRS_E_ARG; }
  const int T = in->T, H = in->H;
  const int64_t N = in->N;
  if (T <= 0 || N < 0 || H <= 0 || !in->indptr || !in->indices || (in->index_bytes != 4 && in->index_bytes != 8) ||
      in->shard_count < 1 || in->shard_rank < 0 || in->shard_rank >= in->shard_count) {
    gbrs_set_error("gbrs_pack_device: bad shape / shard / index width"); return GBRS_E_ARG;
  }
  if (H > GBRS_HPAD || T >= (1 << 24) || N >= (int64_t(1) << 31)) {
    gbrs_set_error("gbrs_pack_device: H > 8, T >= 2^24 or N >= 2^31 (use gbrs_pack_create)"); return GBRS_E_LIMIT;
  }
  if (in->values) { gbrs_set_error("gbrs_pack_device: stored values are not supported (use gbrs_pack_create)"); return GBRS_E_LIMIT; }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { gbrs_set_error("gbrs_pack_device: no CUDA device (there is no CPU fallback)"); return GBRS_E_CUDA; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Arena A{alloc, user};
  std::memset(out, 0, sizeof(*out));
  std::memset(info_out, 0, sizeof(*info_out));
  const int64_t item_len = in->item_len > 0 ? (in->item_len + 7) / 8 * 8 : 64;
  const char* lf_env = std::getenv("GBRS_LONG_FACTOR");
  const ItemRule rule{item_len, (lf_env ? std::max(8, std::atoi(lf_env)) : 32) * item_len};
  const uint32_t full = (1u << H) - 1u;

  // ---- inputs to the device ------------------------------------------------------------------------------------------
  Columns col{};
  col.T = T; col.H = H; col.N = N;
  int64_t nnz_in = 0;
  for (int h = 0; h < H; ++h) {
    if (!in->indptr[h] || in->indptr[h][0] != 0 || (!in->indices[h] && in->indptr[h][T] > 0)) {
      gbrs_set_error("gbrs_pack_device: bad CSC arrays"); return GBRS_E_ARG;
    }
    col.hoff[h] = nnz_in;
    nnz_in += in->indptr[h][T];
  }
  if (nnz_in >= (int64_t(1) << 32)) { gbrs_set_error("gbrs_pack_device: more than 2^32 stored entries (use gbrs_pack_create)"); return GBRS_E_LIMIT; }
  int64_t* d_indptr = A.get<int64_t>((int64_t) H * (T + 1), "tmp:indptr");
  uint32_t* d_indices = A.get<uint32_t>(nnz_in, "tmp:indices");
  int* d_bad = A.get<int>(4, "tmp:bad");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  GP_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int) * 4, s));
  for (int h = 0; h < H; ++h) {
    GP_CUDA(cudaMemcpyAsync(d_indptr + (int64_t) h * (T + 1), in->indptr[h], sizeof(int64_t) * (size_t) (T + 1), cudaMemcpyHostToDevice, s));
    const int64_t n = in->indptr[h][T];
    if (n == 0) continue;
    if (in->index_bytes == 4) {
      GP_CUDA(cudaMemcpyAsync(d_indices + col.hoff[h], in->indices[h], sizeof(uint32_t) * (size_t) n, cudaMemcpyHostToDevice, s));
    } else {
      int64_t* wide = A.get<int64_t>(n, "tmp:indices64");
      if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
      GP_CUDA(cudaMemcpyAsync(wide, in->indices[h], sizeof(int64_t) * (size_t) n, cudaMemcpyHostToDevice, s));
      k_gp_narrow<<<gp_grid(n), kGpThreads, 0, s>>>(wide, d_indices + col.hoff[h], n, N, d_bad);
    }
  }
  col.indptr = d_indptr;
  col.indices = d_indices;
  if (in->locus_hapmask) {
    uint8_t* d_mask = A.get<uint8_t>(T, "tmp:hapmask");
    if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
    GP_CUDA(cudaMemcpyAsync(d_mask, in->locus_hapmask, (size_t) T, cudaMemcpyHostToDevice, s));
    col.hapmask = d_mask;
  }
  // gene tables (host: T is small), kept by the caller like every other output
  std::vector<int32_t> gene_of(T);
  for (int t = 0; t < T; ++t) {
    gene_of[t] = in->gene_of ? in->gene_of[t] : t;
    if (gene_of[t] < 0) { gbrs_set_error("gbrs_pack_device: negative gene id"); return GBRS_E_ARG; }
  }
  const int32_t n_gene_ids = 1 + *std::max_element(gene_of.begin(), gene_of.end());
  std::vector<uint32_t> gene_ptr((size_t) n_gene_ids + 1, 0), gene_loci((size_t) T, 0);
  for (int t = 0; t < T; ++t) ++gene_ptr[gene_of[t] + 1];
  for (int g = 0; g < n_gene_ids; ++g) gene_ptr[g + 1] += gene_ptr[g];
  {
    std::vector<uint32_t> cur(gene_ptr.begin(), gene_ptr.end() - 1);
    for (int t = 0; t < T; ++t) gene_loci[cur[gene_of[t]]++] = (uint32_t) t;
  }
  int32_t* d_gene_of = A.get<int32_t>(T, "gene_of");
  uint32_t* d_gene_ptr = A.get<uint32_t>(n_gene_ids + 1, "gene_ptr");
  uint32_t* d_gene_loci = A.get<uint32_t>(T, "gene_loci");
  double* d_count_in = in->count ? A.get<double>(N, "tmp:count") : nullptr;
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  GP_CUDA(cudaMemcpyAsync(d_gene_of, gene_of.data(), sizeof(int32_t) * (size_t) T, cudaMemcpyHostToDevice, s));
  GP_CUDA(cudaMemcpyAsync(d_gene_ptr, gene_ptr.data(), sizeof(uint32_t) * gene_ptr.size(), cudaMemcpyHostToDevice, s));
  GP_CUDA(cudaMemcpyAsync(d_gene_loci, gene_loci.data(), sizeof(uint32_t) * (size_t) T, cudaMemcpyHostToDevice, s));
  if (d_count_in) GP_CUDA(cudaMemcpyAsync(d_count_in, in->count, sizeof(double) * (size_t) N, cudaMemcpyHostToDevice, s));

  // ---- transposition: CSC columns -> class rows --------------------------------------------------------------------------
  uint32_t* rowstart = A.get<uint32_t>(N + 1, "tmp:rowstart");
  uint32_t* npair = A.get<uint32_t>(N + 1, "tmp:npair");
  uint32_t* minloc = A.get<uint32_t>(N + 1, "tmp:minloc");
  uint32_t* secloc = A.get<uint32_t>(N + 1, "tmp:secloc");
  uint32_t* rec = A.get<uint32_t>(nnz_in, "tmp:rec");
  int64_t* d_lohi = A.get<int64_t>(2, "tmp:lohi");
  unsigned long long* d_stats = A.get<unsigned long long>(8, "tmp:stats");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  GP_CUDA(cudaMemsetAsync(rowstart, 0, sizeof(uint32_t), s));
  GP_CUDA(cudaMemsetAsync(d_stats, 0, sizeof(unsigned long long) * 8, s));
  const int col_grid = gp_grid((int64_t) H * T * 32);
  // the entries that survive the mask, re-laid locus-major (column starts by a scan over the T x H column lengths), are
  // stable-sorted by class id (library radix sort over the bits of N); the records of a class then arrive ordered by
  // (locus, haplotype) and merging them is one linear pass -- no atomics, no per-class sorts
  const int64_t n_cols = (int64_t) H * T;
  int64_t n_kept = 0;
  for (int t = 0; t < T; ++t)
    for (int h = 0; h < H; ++h)
      if (!in->locus_hapmask || ((in->locus_hapmask[t] >> h) & 1)) n_kept += in->indptr[h][t + 1] - in->indptr[h][t];
  uint32_t* collen = A.get<uint32_t>(n_cols + 1, "tmp:collen");
  uint32_t* colstart = A.get<uint32_t>(n_cols + 1, "tmp:colstart");
  uint32_t* keys = A.get<uint32_t>(n_kept, "tmp:keys");
  uint32_t* keys2 = A.get<uint32_t>(n_kept, "tmp:keys2");
  uint32_t* vals = A.get<uint32_t>(n_kept, "tmp:vals");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  GP_CUDA(cudaMemsetAsync(colstart, 0, sizeof(uint32_t), s));
  k_gp_col_len<<<gp_grid(n_cols), kGpThreads, 0, s>>>(col, collen);
  if (int rc = inclusive_scan_into(A, collen, colstart + 1, n_cols, s)) return rc;
  k_gp_gen<<<col_grid, kGpThreads, 0, s>>>(col, colstart, keys, vals, d_bad);
  int bits = 1;
  while ((int64_t(1) << bits) < N) ++bits;
  if (n_kept > 0)
    if (int rc = sort_pairs(A, keys, keys2, vals, rec, n_kept, bits, s)) return rc;
  k_gp_rowstart<<<gp_grid(n_kept + 1), kGpThreads, 0, s>>>(keys2, n_kept, N, rowstart);
  if (N > 0) k_gp_merge<<<gp_grid(N), kGpThreads, 0, s>>>(N, rowstart, rec, npair, minloc, secloc);
  k_gp_shard<<<1, 32, 0, s>>>(rowstart, N, in->shard_count, in->shard_rank, d_lohi);

  // ---- class order ---------------------------------------------------------------------------------------------------
  uint32_t* okey = A.get<uint32_t>(N + 1, "tmp:okey");
  uint32_t* oval = A.get<uint32_t>(N + 1, "tmp:oval");
  uint32_t* okey2 = A.get<uint32_t>(N + 1, "tmp:okey2");
  uint32_t* order = A.get<uint32_t>(N + 1, "tmp:order");
  int64_t* d_buckets = A.get<int64_t>(GBRS_KMAX + 2, "tmp:buckets");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  if (N > 0) {
    k_gp_order_keys<<<gp_grid(N), kGpThreads, 0, s>>>(N, d_lohi, npair, minloc, okey, oval, d_stats);
    // (width, smallest locus, second-smallest locus, class id): two stable sorts, minor key first.  Classes sharing their two
    // smallest loci end up next to each other, so a warp of the row pass reads fewer distinct table rows and the entries of a
    // locus gather runs of consecutive weights in the column pass.
    uint32_t* sec_sorted = A.get<uint32_t>(N + 1, "tmp:sec_sorted");
    uint32_t* val1 = A.get<uint32_t>(N + 1, "tmp:val1");
    uint32_t* okey_g = A.get<uint32_t>(N + 1, "tmp:okey_g");
    if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
    if (int rc = sort_pairs(A, secloc, sec_sorted, oval, val1, N, 24, s)) return rc;
    k_gp_gather_u32<<<gp_grid(N), kGpThreads, 0, s>>>(N, val1, okey, okey_g);
    if (int rc = sort_pairs(A, okey_g, okey2, val1, order, N, 32, s)) return rc;
  }
  k_gp_buckets<<<1, 32, 0, s>>>(okey2, N, d_buckets);
  GP_CUDA(cudaGetLastError());
  int64_t h_buckets[GBRS_KMAX + 2], h_lohi[2];
  unsigned long long h_stats[8];
  int h_bad[4];
  uint32_t h_total = 0, h_lo_cum = 0, h_hi_cum = 0;
  if (int rc = read_back(d_buckets, h_buckets, GBRS_KMAX + 2, s)) return rc;
  if (int rc = read_back(d_lohi, h_lohi, 2, s)) return rc;
  if (int rc = read_back(d_stats, h_stats, 8, s)) return rc;
  if (int rc = read_back(d_bad, h_bad, 4, s)) return rc;
  if (int rc = read_back(rowstart + N, &h_total, 1, s)) return rc;
  if (int rc = read_back(rowstart + h_lohi[0], &h_lo_cum, 1, s)) return rc;
  if (int rc = read_back(rowstart + h_lohi[1], &h_hi_cum, 1, s)) return rc;
  if (h_bad[0]) { gbrs_set_error("gbrs_pack_device: class index out of range"); return GBRS_E_ARG; }
  const int64_t n_classes = h_buckets[GBRS_KMAX + 1];

  // ---- class-major arrays in the new order ----------------------------------------------------------------------------
  uint32_t* rowptr = A.get<uint32_t>(n_classes + 1, "rowptr");
  uint32_t* runptr = A.get<uint32_t>(n_classes + 1, "runptr");
  double* count = A.get<double>(n_classes, "count");
  uint32_t* class_id = A.get<uint32_t>(n_classes, "class_id");
  uint32_t* npair_new = A.get<uint32_t>(n_classes + 1, "tmp:npair_new");
  uint32_t* nruns = A.get<uint32_t>(n_classes + 1, "tmp:nruns");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  GP_CUDA(cudaMemsetAsync(rowptr, 0, sizeof(uint32_t), s));
  GP_CUDA(cudaMemsetAsync(runptr, 0, sizeof(uint32_t), s));
  uint32_t n_pairs32 = 0, n_runs32 = 0;
  if (n_classes > 0) {
    // the first n_classes entries of the order are this shard's non-empty classes: their input ids are the class ids
    GP_CUDA(cudaMemcpyAsync(class_id, order, sizeof(uint32_t) * (size_t) n_classes, cudaMemcpyDeviceToDevice, s));
    k_gp_gather_u32<<<gp_grid(n_classes), kGpThreads, 0, s>>>(n_classes, order, npair, npair_new);
    if (int rc = inclusive_scan_into(A, npair_new, rowptr + 1, n_classes, s)) return rc;
    if (int rc = read_back(rowptr + n_classes, &n_pairs32, 1, s)) return rc;
  }
  const int64_t n_pairs = n_pairs32;
  uint32_t* pairs = A.get<uint32_t>(n_pairs, "pairs");
  uint32_t* ric = A.get<uint32_t>(n_pairs, "tmp:ric");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  if (n_classes > 0) {
    k_gp_fill_classes<<<gp_grid(n_classes), kGpThreads, 0, s>>>(n_classes, order, rowstart, rec, rowptr, d_gene_of, d_count_in, pairs, ric,
                                                                nruns, count);
    if (int rc = inclusive_scan_into(A, nruns, runptr + 1, n_classes, s)) return rc;
    if (int rc = read_back(runptr + n_classes, &n_runs32, 1, s)) return rc;
  }
  const int64_t n_runs = n_runs32;

  // ---- loci ------------------------------------------------------------------------------------------------------------
  uint32_t* lcnt = A.get<uint32_t>(T + 1, "tmp:lcnt");
  uint32_t* lpart_raw = A.get<uint32_t>(T + 1, "tmp:lpart_raw");
  uint32_t* lpart = A.get<uint32_t>(T + 1, "tmp:lpart");
  uint32_t* ppart = A.get<uint32_t>(T + 1, "tmp:ppart");
  uint32_t* lsize = A.get<uint32_t>(T + 1, "tmp:lsize");
  uint32_t* nitems = A.get<uint32_t>(T + 1, "tmp:nitems");
  uint32_t* lptr = A.get<uint32_t>(T + 1, "tmp:lptr");
  uint32_t* lstart = A.get<uint32_t>(T + 1, "tmp:lstart");
  uint32_t* item_ptr = A.get<uint32_t>(T + 1, "tmp:item_ptr");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  GP_CUDA(cudaMemsetAsync(lcnt, 0, sizeof(uint32_t) * (size_t) (T + 1), s));
  GP_CUDA(cudaMemsetAsync(lpart_raw, 0, sizeof(uint32_t) * (size_t) (T + 1), s));
  GP_CUDA(cudaMemsetAsync(lptr, 0, sizeof(uint32_t), s));
  GP_CUDA(cudaMemsetAsync(lstart, 0, sizeof(uint32_t), s));
  GP_CUDA(cudaMemsetAsync(item_ptr, 0, sizeof(uint32_t), s));
  if (n_pairs > 0) k_gp_locus_counts<<<gp_grid(n_pairs), kGpThreads, 0, s>>>(n_pairs, pairs, full, lcnt, lpart_raw);
  k_gp_locus_geometry<<<gp_grid(T), kGpThreads, 0, s>>>(T, rule, lcnt, lpart_raw, lpart, ppart, lsize, nitems);
  if (int rc = inclusive_scan_into(A, lsize, lptr + 1, T, s)) return rc;
  if (int rc = inclusive_scan_into(A, lcnt, lstart + 1, T, s)) return rc;
  if (int rc = inclusive_scan_into(A, nitems, item_ptr + 1, T, s)) return rc;
  uint32_t n_entries32 = 0, n_items32 = 0;
  if (int rc = read_back(lptr + T, &n_entries32, 1, s)) return rc;
  if (int rc = read_back(item_ptr + T, &n_items32, 1, s)) return rc;
  const int64_t n_entries = n_entries32, n_items = n_items32;

  // ---- locus-major entries ----------------------------------------------------------------------------------------------
  unsigned long long* ekey = A.get<unsigned long long>(n_pairs, "tmp:ekey");
  unsigned long long* ekey2 = A.get<unsigned long long>(n_pairs, "tmp:ekey2");
  uint32_t* eval = A.get<uint32_t>(n_pairs, "tmp:eval");
  uint32_t* eval2 = A.get<uint32_t>(n_pairs, "tmp:eval2");
  uint32_t* item_off = A.get<uint32_t>(n_items + 1, "tmp:item_off");
  uint8_t* item_full = A.get<uint8_t>(n_items + 1, "tmp:item_full");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  if (n_pairs > 0) {
    k_gp_entry_keys<<<gp_grid(n_classes), kGpThreads, 0, s>>>(n_classes, rowptr, pairs, lcnt, rule, full, ekey, eval);
    if (int rc = sort_pairs(A, ekey, ekey2, eval, eval2, n_pairs, 56, s)) return rc;
  }
  k_gp_items<<<gp_grid(T), kGpThreads, 0, s>>>(T, rule, lptr, ppart, lsize, item_ptr, item_off, item_full);
  GP_CUDA(cudaMemcpyAsync(item_off + n_items, &n_entries32, sizeof(uint32_t), cudaMemcpyHostToDevice, s));
  const bool force64 = std::getenv("GBRS_FORCE_ENTRY64") != nullptr;
  const int entry_bytes = (!force64 && std::max({n_classes, n_pairs, n_runs}) + 1 < (int64_t(1) << 24)) ? 4 : 8;
  int rc_e = entry_bytes == 4
                 ? build_entries<uint32_t>(A, s, n_pairs, n_entries, n_items, n_classes, n_runs, item_len, ekey2, eval2, pairs,
                                           lptr, lstart, lpart, ppart, runptr, ric, item_off, out)
                 : build_entries<unsigned long long>(A, s, n_pairs, n_entries, n_items, n_classes, n_runs, item_len, ekey2,
                                                     eval2, pairs, lptr, lstart, lpart, ppart, runptr, ric, item_off, out);
  if (rc_e) return rc_e;

  // ---- items and loci in visiting order ---------------------------------------------------------------------------------
  uint32_t* ikey = A.get<uint32_t>(n_items + 1, "tmp:ikey");
  uint32_t* ikey2 = A.get<uint32_t>(n_items + 1, "tmp:ikey2");
  uint32_t* ival = A.get<uint32_t>(n_items + 1, "tmp:ival");
  uint32_t* ival2 = A.get<uint32_t>(n_items + 1, "tmp:ival2");
  uint32_t* item_desc = A.get<uint32_t>((n_items + 2) * 4, "item_desc");  // + the two-descriptor trailer
  unsigned long long* d_cls = A.get<unsigned long long>(8, "tmp:item_classes");
  uint32_t* tkey = A.get<uint32_t>(T, "tmp:tkey");
  uint32_t* tkey2 = A.get<uint32_t>(T, "tmp:tkey2");
  uint32_t* tval = A.get<uint32_t>(T, "tmp:tval");
  uint32_t* tval2 = A.get<uint32_t>(T, "tmp:tval2");
  uint32_t* locus_desc = A.get<uint32_t>((int64_t) T * 4, "locus_desc");
  if (A.failed) { gbrs_set_error("gbrs_pack_device: allocation failed"); return GBRS_E_NOMEM; }
  GP_CUDA(cudaMemsetAsync(d_cls, 0, sizeof(unsigned long long) * 8, s));
  if (n_items > 0) {
    k_gp_item_keys<<<gp_grid(n_items), kGpThreads, 0, s>>>(n_items, item_len, item_off, item_full, ikey, ival);
    if (int rc = sort_pairs(A, ikey, ikey2, ival, ival2, n_items, 32, s)) return rc;
    k_gp_item_desc<<<gp_grid(n_items), kGpThreads, 0, s>>>(n_items, ikey2, ival2, item_off, item_full, item_desc, d_stats + 2, d_cls);
  }
  k_gp_item_trailer<<<1, 32, 0, s>>>(n_items, d_stats + 2, d_cls, item_desc);
  k_gp_locus_keys<<<gp_grid(T), kGpThreads, 0, s>>>(T, nitems, tkey, tval);
  if (int rc = sort_pairs(A, tkey, tkey2, tval, tval2, T, 32, s)) return rc;
  k_gp_locus_desc<<<gp_grid(T), kGpThreads, 0, s>>>(T, tval2, item_ptr, locus_desc, d_stats + 3);
  GP_CUDA(cudaGetLastError());
  if (int rc = read_back(d_stats, h_stats, 8, s)) return rc;

  out->rowptr = rowptr;
  out->pairs = pairs;
  out->count = count;
  out->runptr = runptr;
  out->class_id = class_id;
  out->item_desc = item_desc;
  out->locus_desc = locus_desc;
  out->gene_of = d_gene_of;
  out->gene_ptr = d_gene_ptr;
  out->gene_loci = d_gene_loci;
  gbrs_pack_info& I = *info_out;
  I.n_classes = n_classes;
  I.n_pairs = n_pairs;
  I.n_runs = n_runs;
  I.n_items = n_items;
  I.n_entries = n_entries;
  I.n_long_items = (int64_t) h_stats[2];
  I.nnz = (int64_t) h_hi_cum - (int64_t) h_lo_cum;
  I.nnz_total = h_total;
  I.n_classes_total = (int64_t) h_stats[0];
  I.entry_bytes = entry_bytes;
  I.n_gene_ids = n_gene_ids;
  I.max_pairs_per_class = (int32_t) h_stats[1];
  I.n_deep_loci = (int32_t) h_stats[3];
  for (int b = 0; b <= GBRS_KMAX + 1; ++b) {
    I.bucket_class0[b] = b <= GBRS_KMAX ? std::min<int64_t>(h_buckets[b], n_classes) : n_classes;
  }
  {
    // bucket_pair0[b] = rowptr[bucket_class0[b]]
    for (int b = 0; b <= GBRS_KMAX + 1; ++b) {
      uint32_t v = 0;
      if (int rc = read_back(rowptr + I.bucket_class0[b], &v, 1, s)) return rc;
      I.bucket_pair0[b] = v;
    }
  }
  return GBRS_OK;
}
