// sm_100a kernels + C-ABI launchers of the multiway EM quantifier.  See include/gbrs_em.h for the contract and
// DESIGN.md for the layout / roofline discussion.  Reference lines are cited per kernel (paths under /root/reference).
//
// One EM update (EMfactory.update_allelic_expression, src/gbrs/emase/EMfactory.py:214-232) is
//
//   row pass     k_weights_m*     per class:  normaliser(s) of the model's hierarchy from theta  ->  weight(s)
//   column pass  k_column_reduce  per locus work item:  sum of the weights of the classes hitting it, per haplotype
//   k_locus_acc                   acc[t][h] = theta[t][h] * W[t][h]                (= sum_n count[n] * P[n,t,h])
//   -- cross-rank sum of acc when the classes are row-sharded --
//   k_locus_update                theta' = acc / efflen, isoform totals, block partial sums
//   k_converge                    TPM-scaled L1 change, stop decision, ping-pong flip (EMfactory.py:267-279)
//
// Both passes are gathers over an incidence matrix stored twice (class-major / locus-major), so there are no atomics
// and the result is bit-reproducible run to run.  The posterior P is never materialised.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "gbrs_em.h"

// NVTX ranges around the phases of an update (row pass / column pass / locus kernel + exchange / stop test): visible in
// Nsight Systems timelines; a no-op without an attached tool.  Header-only NVTX 3 (no link dependency).
#ifndef GBRS_SIMT_EMULATION
#include <nvtx3/nvToolsExt.h>
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};
#else
struct NvtxRange {
  explicit NvtxRange(const char*) {}
};
#endif

// ---------------------------------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
void gbrs_set_error(const std::string& s) { g_last_error = s; }
extern "C" const char* gbrs_last_error(void) { return g_last_error.c_str(); }
extern "C" int gbrs_abi_version(void) { return GBRS_EM_ABI_VERSION; }

#define GBRS_CUDA(call)                                                                              \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess) {                                                                         \
      gbrs_set_error(std::string(#call) + ": " + cudaGetErrorString(e_));                            \
      return GBRS_E_CUDA;                                                                            \
    }                                                                                                \
  } while (0)

#define GBRS_LAUNCH_CHECK(name)                                                                      \
  do {                                                                                               \
    cudaError_t e_ = cudaGetLastError();                                                             \
    if (e_ != cudaSuccess) {                                                                         \
      gbrs_set_error(std::string("launch ") + name + ": " + cudaGetErrorString(e_));                 \
      return GBRS_E_CUDA;                                                                            \
    }                                                                                                \
  } while (0)

namespace {

#ifndef GBRS_THREADS
#define GBRS_THREADS 256
#endif
constexpr int kThreads = GBRS_THREADS;  // threads per block of every grid-stride kernel
#ifndef GBRS_COL_MINBLOCKS
#define GBRS_COL_MINBLOCKS 4  // resident blocks per SM the column pass is compiled for (64 registers at 256 threads)
#endif
constexpr uint32_t kLocusMask = 0xFFFFFFu;
constexpr int kStampSlot = GBRS_PART_SLOTS - 8;  // k_locus_xchg: phase time stamps of block 0 (diagnostics, bench.py)

int g_sm_count = 0;
int sm_count() {
  if (g_sm_count == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) g_sm_count = 148;
  }
  return g_sm_count;
}

inline int grid_for(int64_t threads_needed, int blocks_per_sm = 8) {
  int64_t b = (threads_needed + kThreads - 1) / kThreads;
  int64_t cap = (int64_t) sm_count() * blocks_per_sm;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int) b;
}

// Persistent grid: exactly as many blocks as are resident at once (SMs x occupancy of this kernel), so that the
// grid-stride loops run in a single full wave instead of 1.33 ragged ones.
template <typename Kern>
int resident_grid(Kern kern, int64_t threads_needed) {
  static std::unordered_map<const void*, int> cache;
  const void* key = reinterpret_cast<const void*>(kern);
  auto it = cache.find(key);
  int occ;
  if (it == cache.end()) {
    occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kThreads, 0) != cudaSuccess || occ < 1) occ = 4;
    cache[key] = occ;
  } else {
    occ = it->second;
  }
  return grid_for(threads_needed, occ);
}

// ---------------------------------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double2 ldg2(const double* p) { return __ldg(reinterpret_cast<const double2*>(p)); }

// sum of the haplotype slots selected by `m` of one 64-byte locus line
__device__ __forceinline__ double masked_sum8(const double* __restrict__ line, uint32_t m) {
  const double2 a = ldg2(line), b = ldg2(line + 2), c = ldg2(line + 4), e = ldg2(line + 6);
  double s = 0.0;
  s += (m & 1u) ? a.x : 0.0;
  s += (m & 2u) ? a.y : 0.0;
  s += (m & 4u) ? b.x : 0.0;
  s += (m & 8u) ? b.y : 0.0;
  s += (m & 16u) ? c.x : 0.0;
  s += (m & 32u) ? c.y : 0.0;
  s += (m & 64u) ? e.x : 0.0;
  s += (m & 128u) ? e.y : 0.0;
  return s;
}

__device__ __forceinline__ void load8(const double* __restrict__ line, double (&v)[8]) {
  const double2 a = ldg2(line), b = ldg2(line + 2), c = ldg2(line + 4), e = ldg2(line + 6);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = e.x; v[7] = e.y;
}

// a[h] += w for every haplotype slot h whose bit is set in m.  ptxas turns both `if (bit) a += w` and
// `a += bit ? w : 0` (and even PTX-level predicated add.f64) into DADD + two 32-bit selects per slot.  Multiplying by a
// 0.0 / 1.0 whose high word is built from the bit costs LOP3 + IMAD + IMAD.MOV (zero low word) + DFMA, and
// fma(w, 1.0, a) == a + w exactly.  Measured on B200 (C2, column pass, profiles/r1_column_pass_variants.txt): this form
// 34.2 us; selecting both words of w with R2P predicates (3 instructions per slot, all on the ALU pipe) 41.6 us;
// selecting only the high word (2 per slot, masked-out terms become denormals) 53.5 us.  Fewer instructions lose here
// because the multiplier form spreads its work over the ALU, FMA and FP64 pipes.
__device__ __forceinline__ void masked_add8(double (&a)[8], double w, uint32_t m) {
#pragma unroll
  for (int h = 0; h < 8; ++h) {
    // (m & 2^h) is 0 or 2^h; times (0x3FF00000 >> h) gives the high word of 0.0 or 1.0 in two integer instructions
    const uint32_t hi = (m & (1u << h)) * (0x3FF00000u >> h);
    a[h] = fma(w, __hiloint2double((int) hi, 0), a[h]);
  }
}

// c / s without the library division's slow path: reciprocal seed + two Newton steps + one residual correction
// (<= 1 ulp; s == 0, a denormal s -- rcp.approx flushes it -- or non-finite input yields inf/NaN, which the convergence
// kernel turns into GBRS_E_NUMERIC.  A guard that re-divides with the IEEE division cost the row pass 3-4 us and was dropped).
__device__ __forceinline__ double fast_div(double c, double s) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(s));
  r = fma(fma(-s, r, 1.0), r, r);
  r = fma(fma(-s, r, 1.0), r, r);
  const double q = c * r;
  return fma(fma(-s, q, c), r, q);
}

// Sum over the 8 lanes of an aligned lane group; every lane gets the total.  Fixed order => deterministic.
__device__ __forceinline__ double group8_sum(double v) {
  v += __shfl_xor_sync(0xFFFFFFFFu, v, 4);
  v += __shfl_xor_sync(0xFFFFFFFFu, v, 2);
  v += __shfl_xor_sync(0xFFFFFFFFu, v, 1);
  return v;
}

// Transposing reduction: each of the 8 lanes of a group holds a[0..8); afterwards lane j holds sum over lanes of a[j].
__device__ __forceinline__ double group8_transpose_sum(const double (&a)[8], int lane8) {
  double b[4], c[2];
  const bool hi4 = lane8 & 4, hi2 = lane8 & 2, hi1 = lane8 & 1;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const double send = hi4 ? a[i] : a[i + 4];
    const double keep = hi4 ? a[i + 4] : a[i];
    b[i] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, 4);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const double send = hi2 ? b[i] : b[i + 2];
    const double keep = hi2 ? b[i + 2] : b[i];
    c[i] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, 2);
  }
  const double send = hi1 ? c[0] : c[1];
  const double keep = hi1 ? c[1] : c[0];
  return keep + __shfl_xor_sync(0xFFFFFFFFu, send, 1);
}

// Block-wide sum in a fixed order (warp shuffle tree, then warp 0 over the per-warp values).  All threads must call.
__device__ __forceinline__ double block_sum(double v, double* smem /* [32] */) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  // only warp 0 reads the per-warp values: it overwrites smem[0] with the total below, which the other warps must not
  // be reading at that moment (they discarded the value, but the access itself was unordered)
  double r = (warp == 0 && lane < nw) ? smem[lane] : 0.0;
  if (warp == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, o);
    if (lane == 0) smem[0] = r;
  }
  __syncthreads();
  r = smem[0];
  return r;
}

__device__ __forceinline__ const double* theta_cur(const gbrs_em_dev& d) {
  return d.theta + (size_t) d.ctrl[GBRS_CTRL_PARITY] * d.T * GBRS_HPAD;
}

// ---------------------------------------------------------------------------------------------------------------------
// Fused cross-rank exchange over NVLink peer memory (row-sharded runs, up to 8 ranks of one NVSwitch domain).
// Every rank owns one symmetric buffer, peer-mapped into all ranks (`xchg_peer[r]`):
//     [0, 64T)   acc_local   this rank's local numerator (written by k_locus_acc)
//     [64T,128T) acc_total   the numerator summed over ranks (written by the owners of each slice, k_xchg_reduce)
//     then       ready[8], done[8]   u32 epoch flags, written remotely by the rank they are indexed by
// `xchg_mc` (optional) is the NVSwitch multicast mapping of the same buffers.
// Two-shot all-reduce inside our own kernels: k_locus_acc publishes acc_local and raises ready[me] = e on every peer;
// k_xchg_reduce waits for all ready flags, sums ITS slice of the loci over the ranks in rank order with peer loads,
// stores the total into every rank's acc_total with peer stores and raises done[me] = e everywhere; k_locus_update
// waits for all done flags and carries on locally.  In an EM update the reduce step runs at the head of the
// k_locus_update launch itself (k_locus_update<true, true>), and with a multicast mapping the switch does the adding
// and the broadcasting (xchg_reduce_slice<true>).  Each element is summed by exactly one rank, so all ranks see
// bit-identical totals and take identical stop decisions.  Waits are bounded: a missing peer raises the error flag
// instead of hanging the GPU.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ double2 ld_relaxed_sys_f64x2(const double* p) {
  double2 v;
  asm volatile("ld.relaxed.sys.global.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys_f64x2(double* p, double2 v) {
  asm volatile("st.relaxed.sys.global.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ double* xchg_acc_local(const gbrs_em_dev& d, int r) { return static_cast<double*>(d.xchg_peer[r]); }
__device__ __forceinline__ double* xchg_acc_total(const gbrs_em_dev& d, int r) {
  return static_cast<double*>(d.xchg_peer[r]) + (size_t) d.T * GBRS_HPAD;
}
__device__ __forceinline__ uint32_t* xchg_flags(const gbrs_em_dev& d, int r, int which /* 0 ready, 1 done */) {
  return reinterpret_cast<uint32_t*>(static_cast<double*>(d.xchg_peer[r]) + 2 * (size_t) d.T * GBRS_HPAD) + which * 8;
}
// thread 0 of the block waits until every rank's flag has reached epoch e; the block then proceeds together
__device__ __forceinline__ void xchg_wait_all(const gbrs_em_dev& d, int which, uint32_t e) {
  if (threadIdx.x == 0) {
    const uint32_t* f = xchg_flags(d, d.xchg_rank, which);
    for (int r = 0; r < d.n_ranks; ++r) {
      long spins = 0;
      while ((int32_t) (ld_acquire_sys(f + r) - e) < 0) {
        if (++spins > (1L << 24)) { d.ctrl[GBRS_CTRL_ERROR] = 3; break; }
        __nanosleep(100);
      }
    }
  }
  __syncthreads();
}
// called by every block at the end of a kernel: when the whole grid is through, raise flag[me] = e on every rank
__device__ __forceinline__ void xchg_signal_all(const gbrs_em_dev& d, int which, uint32_t e, int ticket_slot) {
  __syncthreads();
  if (threadIdx.x == 0) {
    // every block orders its own writes before its ticket at gpu scope; the last block, having observed all tickets,
    // issues the one system-scope fence before the flags (release cumulativity) -- a system fence per block costs
    // ~15 us over the ~900 blocks of the locus kernel
    __threadfence();
    const int ticket = atomicAdd(d.ctrl + ticket_slot, 1);
    if (ticket == (int) gridDim.x - 1) {
      d.ctrl[ticket_slot] = 0;
      if (which == 1) d.ctrl[GBRS_CTRL_XEPOCH] = (int32_t) e;  // the exchange e is complete on this rank's side
      // one system-scope fence, then the flags as plain system-scope stores issued back to back (a releasing store
      // per peer would wait for the previous one to be performed: ~2 us each over NVLink)
      __threadfence_system();
      for (int r = 0; r < d.n_ranks; ++r) st_relaxed_sys_u32(xchg_flags(d, r, which) + d.xchg_rank, e);
    }
  }
}

// In-switch reduction / multicast store on the NVSwitch multicast mapping of the symmetric buffers (NVLS): one load
// returns the sum over all ranks of the addressed element, one store writes every rank's copy.
__device__ __forceinline__ double multimem_ld_reduce_add(const double* mc) {
  double v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.f64 %0, [%1];" : "=d"(v) : "l"(mc) : "memory");
  return v;
}
__device__ __forceinline__ void multimem_st(double* mc, double v) {
  asm volatile("multimem.st.relaxed.sys.global.f64 [%0], %1;" ::"l"(mc), "d"(v) : "memory");
}

// This rank's slice of the T*8 numerator (in units of double2): summed over the ranks and stored into every rank's
// acc_total.  NVLS = false: peer loads, all issued first (one NVLink round trip instead of n_ranks serial ones), then
// the sum in rank order.  NVLS = true: the switch adds (multimem.ld_reduce) and broadcasts (multimem.st); a rank moves
// 2 x 1/R of the numerator instead of 2 x (R-1)/R.  Either way every element is reduced by exactly one rank and the
// same bits reach every rank, so all ranks take identical stop decisions.
template <bool NVLS>
__device__ __forceinline__ void xchg_reduce_slice(const gbrs_em_dev& d) {
  const int64_t n2 = (int64_t) d.T * GBRS_HPAD / 2;
  const int64_t per = (n2 + d.n_ranks - 1) / d.n_ranks;
  const int64_t lo = per * d.xchg_rank, hi = lo + per < n2 ? lo + per : n2;
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t i = lo + (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += stride) {
    if (NVLS) {
      double* mc_local = static_cast<double*>(d.xchg_mc);
      double* mc_total = mc_local + (size_t) d.T * GBRS_HPAD;
      const double x = multimem_ld_reduce_add(mc_local + 2 * i), y = multimem_ld_reduce_add(mc_local + 2 * i + 1);
      multimem_st(mc_total + 2 * i, x);
      multimem_st(mc_total + 2 * i + 1, y);
    } else {
      double2 v[8];
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < d.n_ranks) v[r] = ld_relaxed_sys_f64x2(xchg_acc_local(d, r) + 2 * i);
      double2 s = make_double2(0.0, 0.0);
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < d.n_ranks) {
          s.x += v[r].x;
          s.y += v[r].y;
        }
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < d.n_ranks) st_relaxed_sys_f64x2(xchg_acc_total(d, r) + 2 * i, s);
    }
  }
}

// stand-alone reduce (prepare): k_locus_update follows as a kernel of its own
__global__ void __launch_bounds__(kThreads) k_xchg_reduce(const __grid_constant__ gbrs_em_dev d) {
  const uint32_t e = (uint32_t) d.ctrl[GBRS_CTRL_XEPOCH] + 1u;
  xchg_wait_all(d, 0, e);
  if (d.xchg_mc) xchg_reduce_slice<true>(d);
  else xchg_reduce_slice<false>(d);
  xchg_signal_all(d, 1, e, GBRS_CTRL_TICKET + 2);
}

// ---------------------------------------------------------------------------------------------------------------------
// row pass, model 4:  w[n] = count[n] / sum_{(t,h) in n} theta[t][h]
// reference: multiply(theta, READ) + normalize_reads(READ)   EMfactory.py:204-208, AlignmentPropertyMatrix.py:335-342
// UNIT = true is the prepare() variant with theta == 1 on the pattern (EMfactory.py:95): w[n] = count[n] / nnz[n].
// ---------------------------------------------------------------------------------------------------------------------
// Subset-sum tables: for every locus the 16 subset sums of haplotype slots 0-3 and the 16 subset sums of slots 4-7,
//   sub[t][m]      = sum_{h<4,  bit h of m}  theta[t][h]        m = 0..15
//   sub[t][16 + m] = sum_{h>=4, bit h-4 of m} theta[t][h]
// so that the masked sum of a (class, locus) pair is two 8-byte loads and one add instead of a 64-byte line and eight
// predicated adds: the row pass is instruction-issue bound, not bandwidth bound, and this removes ~80% of its
// instructions.  One warp per locus, lane = table slot; 256-byte coalesced store.  Rebuilt once per EM update (20 MB
// at 80k loci, L2 resident).
__global__ void __launch_bounds__(kThreads) k_subset_tables(const gbrs_em_dev d) {
  const double* __restrict__ th = theta_cur(d);
  const int lane = threadIdx.x & 31, half = lane >> 4, m = lane & 15;
  const int64_t nwarps = ((int64_t) gridDim.x * blockDim.x) >> 5;
  for (int64_t t = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < d.T; t += nwarps) {
    const double2 a = *reinterpret_cast<const double2*>(th + (size_t) t * GBRS_HPAD + 4 * half);
    const double2 b = *reinterpret_cast<const double2*>(th + (size_t) t * GBRS_HPAD + 4 * half + 2);
    double s = 0.0;
    s += (m & 1) ? a.x : 0.0;
    s += (m & 2) ? a.y : 0.0;
    s += (m & 4) ? b.x : 0.0;
    s += (m & 8) ? b.y : 0.0;
    d.subsets[(size_t) t * 32 + lane] = s;
  }
}

__device__ __forceinline__ double pair_sum(const double* __restrict__ sub, uint32_t w) {
  const double* row = sub + (size_t) (w & kLocusMask) * 32;
  return __ldg(row + ((w >> 24) & 15u)) + __ldg(row + 16 + (w >> 28));
}

// Fixed-width part (classes with K <= GBRS_KMAX pairs, stored contiguously per width, so no row pointers): one thread
// per class, UNR classes per thread; all pair words are loaded first, then all table loads are issued together
// (memory-level parallelism), then the adds.  Classes are ordered by smallest locus within a width, so the lanes of a
// warp mostly read the same few table rows.
__host__ __device__ constexpr int unr_of(int K) { return K <= 2 ? 4 : (K <= 4 ? 2 : 1); }

struct RowPlan {                     // host-computed: work units ordered from the widest fixed bucket down to width 1
  int64_t unit_end[GBRS_KMAX];       // unit_end[i] = one past the last unit (= 32 * unr classes) of width GBRS_KMAX - i
};

template <int K, bool UNIT, bool ZA>
__device__ __forceinline__ void row_classes_m4(const gbrs_em_dev& d, int64_t class0, int64_t class_end,
                                               int64_t bucket_class0, int64_t bucket_pair0) {
  constexpr int UNR = unr_of(K);
  const int lane = threadIdx.x & 31;
  uint32_t w[UNR][K];
  int64_t n[UNR];
  double cnt[UNR];
#pragma unroll
  for (int u = 0; u < UNR; ++u) {
    n[u] = class0 + u * 32 + lane;
    const bool valid = n[u] < class_end;
    const uint32_t* __restrict__ pw = d.pairs + bucket_pair0 + (valid ? (n[u] - bucket_class0) : 0) * K;
#pragma unroll
    for (int p = 0; p < K; ++p) w[u][p] = valid ? __ldcs(pw + p) : 0u;
    cnt[u] = valid ? __ldcs(d.count + n[u]) : 0.0;
  }
  double s[UNR];
  if (UNIT) {
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      int c = 0;
#pragma unroll
      for (int p = 0; p < K; ++p) c += __popc(w[u][p] >> 24);
      s[u] = (double) c;
    }
  } else {
    double lo[UNR][K], hi[UNR][K];
#pragma unroll
    for (int u = 0; u < UNR; ++u)
#pragma unroll
      for (int p = 0; p < K; ++p) {
        const double* row = d.subsets + (size_t) (w[u][p] & kLocusMask) * 32;
        lo[u][p] = __ldg(row + ((w[u][p] >> 24) & 15u));
        hi[u][p] = __ldg(row + 16 + (w[u][p] >> 28));
      }
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      double a = 0.0;
#pragma unroll
      for (int p = 0; p < K; ++p) a += lo[u][p] + hi[u][p];
      s[u] = a;
    }
  }
#pragma unroll
  for (int u = 0; u < UNR; ++u)
    if (n[u] < class_end) d.weights[n[u]] = (ZA && cnt[u] == 0.0) ? 0.0 : fast_div(cnt[u], s[u]);
}

// One launch per width range [KLO, KHI]: the narrow classes (four out of five have at most three pairs) are not compiled for
// the register needs of the widest, so more of them are resident and more loads are in flight.
#ifndef GBRS_ROW_MINBLOCKS
#define GBRS_ROW_MINBLOCKS 1  // resident blocks per SM the model-4 row pass is compiled for (1: no register cap)
#endif
// ZA (descriptor flag zero_count_absent): a class of count 0 is absent -- weight 0 without a division, so a class whose
// entries all have theta 0 does not turn into 0 / 0 (bootstrap replicates drop classes).  The default instantiation
// (ZA = false) is the row pass of every ordinary update, unchanged.
template <bool UNIT, int KLO, int KHI, bool ZA = false>
__global__ void __launch_bounds__(kThreads, GBRS_ROW_MINBLOCKS) k_weights_m4(const __grid_constant__ gbrs_em_dev d,
                                                          const __grid_constant__ RowPlan plan) {
  if (!UNIT && d.ctrl[GBRS_CTRL_DONE]) return;
  const int64_t nwarps = ((int64_t) gridDim.x * blockDim.x) >> 5;
  const int64_t total_units = plan.unit_end[KHI - KLO];
  int i = 0;  // bucket index only ever advances along the warp's grid-stride walk
  int64_t unit0 = 0, unit1 = plan.unit_end[0];
  for (int64_t u = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < total_units; u += nwarps) {
    while (u >= unit1) {
      unit0 = unit1;
      unit1 = plan.unit_end[++i];
    }
    const int k = KHI - i;
    const int64_t c0 = d.bucket_class0[k - 1], c1 = d.bucket_class0[k], p0 = d.bucket_pair0[k - 1];
    const int cpu = 32 * unr_of(k);
    const int64_t class0 = c0 + (u - unit0) * cpu;
#define GBRS_ROW_CASE(K) \
  case K:                \
    if constexpr (K >= KLO && K <= KHI) row_classes_m4<K, UNIT, ZA>(d, class0, c1, c0, p0); \
    break;
    switch (k) {
      GBRS_ROW_CASE(1) GBRS_ROW_CASE(2) GBRS_ROW_CASE(3) GBRS_ROW_CASE(4)
      GBRS_ROW_CASE(5) GBRS_ROW_CASE(6) GBRS_ROW_CASE(7) GBRS_ROW_CASE(8)
      default: break;
    }
#undef GBRS_ROW_CASE
  }
}

// Classes with more than GBRS_KMAX pairs: one thread per class over the CSR row.
template <bool UNIT, bool ZA = false>
__global__ void __launch_bounds__(kThreads) k_weights_m4_long(const gbrs_em_dev d) {
  if (!UNIT && d.ctrl[GBRS_CTRL_DONE]) return;
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t n = d.bucket_class0[GBRS_KMAX] + (int64_t) blockIdx.x * blockDim.x + threadIdx.x; n < d.n_classes; n += stride) {
    const uint32_t b = __ldg(d.rowptr + n), e = __ldg(d.rowptr + n + 1);
    double s = 0.0;
    for (uint32_t p = b; p < e; ++p) {
      const uint32_t w = __ldg(d.pairs + p);
      if (UNIT) s += (double) __popc(w >> 24);
      else s += pair_sum(d.subsets, w);
    }
    const double c = __ldg(d.count + n);
    d.weights[n] = (ZA && c == 0.0) ? 0.0 : c / s;
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// per-gene totals for models 1-3:  gene_hap[g][h] = sum_{t in g} theta[t][h]  ( = theta * t2t_mat, EMfactory.py:167 ),
// gamma[t] = sum_h gene_hap[g(t)][h]  ( = (theta * t2t_mat).sum(axis=0), EMfactory.py:173/188/200 ).  8 lanes per gene.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_gene_totals(const gbrs_em_dev d) {
  if (d.ctrl[GBRS_CTRL_DONE]) return;
  const double* __restrict__ th = theta_cur(d);
  const int lane8 = threadIdx.x & 7;
  const int64_t ngroups = ((int64_t) gridDim.x * blockDim.x) >> 3;
  const int64_t rounds = (d.n_gene_ids + ngroups - 1) / ngroups;
  int64_t g = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  for (int64_t r = 0; r < rounds; ++r, g += ngroups) {
    double s = 0.0;
    uint32_t b = 0, e = 0;
    if (g < d.n_gene_ids) { b = __ldg(d.gene_ptr + g); e = __ldg(d.gene_ptr + g + 1); }
    for (uint32_t i = b; i < e; ++i) s += th[(size_t) __ldg(d.gene_loci + i) * GBRS_HPAD + lane8];
    const double tot = group8_sum(s);
    if (g < d.n_gene_ids) {
      d.gene_hap[g * GBRS_HPAD + lane8] = s;
      for (uint32_t i = b + lane8; i < e; i += 8) d.gamma[__ldg(d.gene_loci + i)] = tot;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// row pass, model 3 (Gene -> Isoform*Allele, EMfactory.py:192-203): one weight per (class, gene) run
//   u[r] = count[n] * Gamma_r / (sum_{r' of n} Gamma_r') / D_r,   D_r = sum_{(t,h) in n, t in gene r} theta[t][h]
// Runs whose D_r is 0 drop out (eliminate_zeros before the GROUP division, AlignmentPropertyMatrix.py:350-352).
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_weights_m3(const gbrs_em_dev d, int64_t first_class) {
  if (d.ctrl[GBRS_CTRL_DONE]) return;
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t n = first_class + (int64_t) blockIdx.x * blockDim.x + threadIdx.x; n < d.n_classes; n += stride) {
    const uint32_t b = __ldg(d.rowptr + n), e = __ldg(d.rowptr + n + 1);
    const double c = __ldg(d.count + n);
    double total = 0.0;
    // pass 1: sum of gene totals over the runs that are alive
    for (uint32_t p = b; p < e;) {
      const int32_t g = __ldg(d.gene_of + (__ldg(d.pairs + p) & kLocusMask));
      double D = 0.0, gam = 0.0;
      for (; p < e; ++p) {
        const uint32_t w = __ldg(d.pairs + p), t = w & kLocusMask;
        if (__ldg(d.gene_of + t) != g) break;
        D += pair_sum(d.subsets, w);
        gam = d.gamma[t];
      }
      if (D != 0.0) total += gam;
    }
    // pass 2: weights
    uint32_t run = __ldg(d.runptr + n);
    for (uint32_t p = b; p < e; ++run) {
      const int32_t g = __ldg(d.gene_of + (__ldg(d.pairs + p) & kLocusMask));
      double D = 0.0, gam = 0.0;
      for (; p < e; ++p) {
        const uint32_t w = __ldg(d.pairs + p), t = w & kLocusMask;
        if (__ldg(d.gene_of + t) != g) break;
        D += pair_sum(d.subsets, w);
        gam = d.gamma[t];
      }
      d.weights[run] = (D != 0.0) ? c * gam / total / D : 0.0;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// row pass, model 2 (Gene -> Isoform -> Allele, EMfactory.py:176-191): one weight per (class, locus) pair
//   u[p] = count[n] * (Gamma_r / sum_r' Gamma_r') * (I_t / S_r) / x_p
//   x_p = sum_{h in mask_p} theta[t][h],  I_t = sum_h theta[t][h] (all h),  S_r = sum_{p in r, x_p != 0} I_t
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_weights_m2(const gbrs_em_dev d, int64_t first_class) {
  if (d.ctrl[GBRS_CTRL_DONE]) return;
  const double* __restrict__ iso = d.iso + (size_t) d.ctrl[GBRS_CTRL_PARITY] * d.T;
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t n = first_class + (int64_t) blockIdx.x * blockDim.x + threadIdx.x; n < d.n_classes; n += stride) {
    const uint32_t b = __ldg(d.rowptr + n), e = __ldg(d.rowptr + n + 1);
    const double c = __ldg(d.count + n);
    double total = 0.0;
    for (uint32_t p = b; p < e;) {
      const int32_t g = __ldg(d.gene_of + (__ldg(d.pairs + p) & kLocusMask));
      double S = 0.0, gam = 0.0;
      for (; p < e; ++p) {
        const uint32_t w = __ldg(d.pairs + p), t = w & kLocusMask;
        if (__ldg(d.gene_of + t) != g) break;
        if (pair_sum(d.subsets, w) != 0.0) S += iso[t];
        gam = d.gamma[t];
      }
      if (S != 0.0) total += gam;
    }
    for (uint32_t p = b; p < e;) {
      const int32_t g = __ldg(d.gene_of + (__ldg(d.pairs + p) & kLocusMask));
      double S = 0.0, gam = 0.0;
      uint32_t q = p;
      for (; q < e; ++q) {
        const uint32_t w = __ldg(d.pairs + q), t = w & kLocusMask;
        if (__ldg(d.gene_of + t) != g) break;
        if (pair_sum(d.subsets, w) != 0.0) S += iso[t];
        gam = d.gamma[t];
      }
      const double wg = (S != 0.0) ? c * gam / total / S : 0.0;
      for (; p < q; ++p) {
        const uint32_t w = __ldg(d.pairs + p), t = w & kLocusMask;
        const double x = pair_sum(d.subsets, w);
        d.weights[p] = (x != 0.0) ? wg * iso[t] / x : 0.0;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Fixed-width row passes for models 3 and 2 (classes with K <= GBRS_KMAX pairs, no row pointers): one thread per class,
// all K pair words, masked sums (two subset-table loads each), gene ids and gene totals are fetched up front; the run
// structure (pairs of one gene are adjacent) is resolved in registers with K^2 compares.  Same arithmetic as the
// generic kernels above, which remain in use for the wide classes.
// ---------------------------------------------------------------------------------------------------------------------
template <int K, int MODEL>
__device__ __forceinline__ void row_class_m23(const gbrs_em_dev& d, const double* __restrict__ iso, int64_t n,
                                              const uint32_t* __restrict__ pw, uint32_t pair0) {
  uint32_t w[K];
#pragma unroll
  for (int p = 0; p < K; ++p) w[p] = __ldg(pw + p);
  const double c = __ldg(d.count + n);
  double x[K], gam[K], it[K];
  int32_t g[K];
#pragma unroll
  for (int p = 0; p < K; ++p) {
    const uint32_t t = w[p] & kLocusMask;
    const double* row = d.subsets + (size_t) t * 32;
    x[p] = __ldg(row + ((w[p] >> 24) & 15u)) + __ldg(row + 16 + (w[p] >> 28));
    g[p] = __ldg(d.gene_of + t);
    gam[p] = d.gamma[t];
    it[p] = (MODEL == 2) ? iso[t] : 0.0;
  }
  // per pair: the group sum of its run.  model 3: D = sum x; model 2: S = sum of isoform totals over alive pairs
  double grp[K];
#pragma unroll
  for (int p = 0; p < K; ++p) {
    double a = 0.0;
#pragma unroll
    for (int q = 0; q < K; ++q) {
      const double term = (MODEL == 3) ? x[q] : ((x[q] != 0.0) ? it[q] : 0.0);
      a += (g[q] == g[p]) ? term : 0.0;
    }
    grp[p] = a;
  }
  double total = 0.0;
#pragma unroll
  for (int p = 0; p < K; ++p) {
    const bool start = (p == 0) || (g[p] != g[p - 1]);
    total += (start && grp[p] != 0.0) ? gam[p] : 0.0;
  }
  if (MODEL == 3) {
    uint32_t run = __ldg(d.runptr + n);
#pragma unroll
    for (int p = 0; p < K; ++p) {
      const bool start = (p == 0) || (g[p] != g[p - 1]);
      if (start) {
        if (p > 0) ++run;
        d.weights[run] = (grp[p] != 0.0) ? c * gam[p] / total / grp[p] : 0.0;
      }
    }
  } else {
#pragma unroll
    for (int p = 0; p < K; ++p) {
      const double wg = (grp[p] != 0.0) ? c * gam[p] / total / grp[p] : 0.0;
      d.weights[pair0 + p] = (x[p] != 0.0) ? wg * it[p] / x[p] : 0.0;
    }
  }
}

template <int MODEL, int KLO, int KHI>
__global__ void __launch_bounds__(kThreads) k_weights_m23_fixed(const __grid_constant__ gbrs_em_dev d) {
  if (d.ctrl[GBRS_CTRL_DONE]) return;
  const double* __restrict__ iso = d.iso + (size_t) d.ctrl[GBRS_CTRL_PARITY] * d.T;
  const int64_t first = d.bucket_class0[KLO - 1], end = d.bucket_class0[KHI];
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  // classes are visited widest first (end - 1 down to first): the expensive ones must not form the tail
  for (int64_t j = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; j < end - first; j += stride) {
    const int64_t n = end - 1 - j;
    int k = KHI;
    while (n < d.bucket_class0[k - 1]) --k;
    const uint32_t pair0 = (uint32_t) (d.bucket_pair0[k - 1] + (n - d.bucket_class0[k - 1]) * k);
    const uint32_t* __restrict__ pw = d.pairs + pair0;
#define GBRS_M23_CASE(K) \
  case K:                \
    if constexpr (K >= KLO && K <= KHI) row_class_m23<K, MODEL>(d, iso, n, pw, pair0); \
    break;
    switch (k) {
      GBRS_M23_CASE(1) GBRS_M23_CASE(2) GBRS_M23_CASE(3) GBRS_M23_CASE(4)
      GBRS_M23_CASE(5) GBRS_M23_CASE(6) GBRS_M23_CASE(7) GBRS_M23_CASE(8)
      default: break;
    }
#undef GBRS_M23_CASE
  }
}

template <int MODEL, int KLO, int KHI>
int launch_m23_fixed(const gbrs_em_dev* d, cudaStream_t s) {
  const int64_t n = d->bucket_class0[KHI] - d->bucket_class0[KLO - 1];
  if (n > 0) {
    k_weights_m23_fixed<MODEL, KLO, KHI><<<resident_grid(k_weights_m23_fixed<MODEL, KLO, KHI>, n), kThreads, 0, s>>>(*d);
    GBRS_LAUNCH_CHECK("k_weights_m23_fixed");
  }
  return GBRS_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// row pass, model 1 (Gene -> Allele -> Isoform, EMfactory.py:160-175): eight weights per (class, gene) run
//   u[r][h] = count[n] * (Gamma_r / sum_r' Gamma_r') * (hg[g][h] / Hs_r) / Dh_r[h]
//   Dh_r[h] = sum_{p in r, h in mask_p} theta[t_p][h],  Hs_r = sum_{h: Dh_r[h] != 0} hg[g][h],  hg = gene_hap
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_weights_m1(const gbrs_em_dev d, int64_t first_class) {
  if (d.ctrl[GBRS_CTRL_DONE]) return;
  const double* __restrict__ th = theta_cur(d);
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t n = first_class + (int64_t) blockIdx.x * blockDim.x + threadIdx.x; n < d.n_classes; n += stride) {
    const uint32_t b = __ldg(d.rowptr + n), e = __ldg(d.rowptr + n + 1);
    const double c = __ldg(d.count + n);
    double total = 0.0;
    for (uint32_t p = b; p < e;) {
      const int32_t g = __ldg(d.gene_of + (__ldg(d.pairs + p) & kLocusMask));
      double any = 0.0, gam = 0.0;
      for (; p < e; ++p) {
        const uint32_t w = __ldg(d.pairs + p), t = w & kLocusMask;
        if (__ldg(d.gene_of + t) != g) break;
        any += masked_sum8(th + (size_t) t * GBRS_HPAD, w >> 24);
        gam = d.gamma[t];
      }
      if (any != 0.0) total += gam;
    }
    uint32_t run = __ldg(d.runptr + n);
    for (uint32_t p = b; p < e; ++run) {
      const int32_t g = __ldg(d.gene_of + (__ldg(d.pairs + p) & kLocusMask));
      double Dh[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      double gam = 0.0;
      for (; p < e; ++p) {
        const uint32_t w = __ldg(d.pairs + p), t = w & kLocusMask, m = w >> 24;
        if (__ldg(d.gene_of + t) != g) break;
        double v[8];
        load8(th + (size_t) t * GBRS_HPAD, v);
#pragma unroll
        for (int h = 0; h < 8; ++h) Dh[h] += ((m >> h) & 1u) ? v[h] : 0.0;
        gam = d.gamma[t];
      }
      double hg[8];
      load8(d.gene_hap + (size_t) g * GBRS_HPAD, hg);
      double Hs = 0.0;
#pragma unroll
      for (int h = 0; h < 8; ++h) Hs += (Dh[h] != 0.0) ? hg[h] : 0.0;
      const double wg = (Hs != 0.0) ? c * gam / total / Hs : 0.0;
      double* out = d.weights + (size_t) run * GBRS_HPAD;
#pragma unroll
      for (int h = 0; h < 8; ++h) out[h] = (Dh[h] != 0.0) ? wg * hg[h] / Dh[h] : 0.0;
    }
  }
}

// Model 1, narrow classes (1..3 pairs: four classes out of five), one thread per class, no row pointers and no
// data-dependent loops: the pair words, then the theta lines / gene ids / gene totals of all pairs, then the per-haplotype
// gene totals of the runs are each one round of independent loads; the run structure (pairs of one gene are adjacent) is
// resolved in registers.  Same sums in the same order as k_weights_m1, which keeps the wider classes.
template <int K>
__device__ __forceinline__ void row_class_m1_thread(const gbrs_em_dev& d, const double* __restrict__ th, int64_t n) {
  const uint32_t pair0 = (uint32_t) (d.bucket_pair0[K - 1] + (n - d.bucket_class0[K - 1]) * K);
  uint32_t w[K];
#pragma unroll
  for (int p = 0; p < K; ++p) w[p] = __ldg(d.pairs + pair0 + p);
  const double c = __ldg(d.count + n);
  uint32_t run = __ldg(d.runptr + n);
  int32_t g[K];
  double gam[K], x[K][8];
#pragma unroll
  for (int p = 0; p < K; ++p) {
    const uint32_t t = w[p] & kLocusMask, m = w[p] >> 24;
    g[p] = __ldg(d.gene_of + t);
    gam[p] = d.gamma[t];
    double v[8];
    load8(th + (size_t) t * GBRS_HPAD, v);
#pragma unroll
    for (int h = 0; h < 8; ++h) x[p][h] = ((m >> h) & 1u) ? v[h] : 0.0;
  }
  double hg[K][8];
#pragma unroll
  for (int p = 0; p < K; ++p) load8(d.gene_hap + (size_t) g[p] * GBRS_HPAD, hg[p]);
  // per run start p: Dh[h] over the pairs of the run (in pair order), Hs over the haplotypes that are alive
  double Dh[K][8], Hs[K];
  bool start[K], alive[K];
  double total = 0.0;
#pragma unroll
  for (int p = 0; p < K; ++p) {
    start[p] = (p == 0) || (g[p] != g[p - 1]);
    double hs = 0.0;
    bool any = false;
#pragma unroll
    for (int h = 0; h < 8; ++h) {
      double a = 0.0;
#pragma unroll
      for (int q = 0; q < K; ++q) a += (g[q] == g[p]) ? x[q][h] : 0.0;
      Dh[p][h] = a;
      hs += (a != 0.0) ? hg[p][h] : 0.0;
      any = any || (a != 0.0);
    }
    Hs[p] = hs;
    alive[p] = any;
    total += (start[p] && any) ? gam[p] : 0.0;
  }
#pragma unroll
  for (int p = 0; p < K; ++p) {
    if (!start[p]) continue;
    if (p > 0) ++run;
    const double wg = (Hs[p] != 0.0) ? c * gam[p] / total / Hs[p] : 0.0;
    double* out = d.weights + (size_t) run * GBRS_HPAD;
#pragma unroll
    for (int h = 0; h < 8; h += 2) {
      const double o0 = (Dh[p][h] != 0.0) ? wg * hg[p][h] / Dh[p][h] : 0.0;
      const double o1 = (Dh[p][h + 1] != 0.0) ? wg * hg[p][h + 1] / Dh[p][h + 1] : 0.0;
      *reinterpret_cast<double2*>(out + h) = make_double2(o0, o1);
    }
  }
  (void) alive;
}

constexpr int kM1Narrow = 3;
template <int K>  // one launch per width: a class of one pair is not compiled for the registers three pairs need
__global__ void __launch_bounds__(kThreads) k_weights_m1_narrow(const __grid_constant__ gbrs_em_dev d) {
  if (d.ctrl[GBRS_CTRL_DONE]) return;
  const double* __restrict__ th = theta_cur(d);
  const int64_t first = d.bucket_class0[K - 1], end = d.bucket_class0[K];
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t n = first + (int64_t) blockIdx.x * blockDim.x + threadIdx.x; n < end; n += stride)
    row_class_m1_thread<K>(d, th, n);
}

template <int K>
int launch_m1_narrow(const gbrs_em_dev* d, cudaStream_t s) {
  const int64_t n = d->bucket_class0[K] - d->bucket_class0[K - 1];
  if (n > 0) {
    k_weights_m1_narrow<K><<<resident_grid(k_weights_m1_narrow<K>, n), kThreads, 0, s>>>(*d);
    GBRS_LAUNCH_CHECK("k_weights_m1_narrow");
  }
  return GBRS_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// column pass: for every work item (<= item_len consecutive locus-major entries of ONE locus) the per-haplotype sum of
// the weights of its entries.  8 lanes per item; lane j ends up holding haplotype j and writes wit[item][j].
// reference: APM.sum(axis=READ)  AlignmentPropertyMatrix.py:288-298 (count-weighted column reduce), without the
// per-haplotype matrix copy.  VEC = 1: scalar weight per index; VEC = 8: one weight per haplotype (model 1).
// ---------------------------------------------------------------------------------------------------------------------
// CH steps of one lane of the column pass: step q covers the four entry words at p0 + 4 * LANES * q.  A step beyond the
// item's end reads the item's first quad again with the masks stripped, which adds nothing.
template <typename E, int LANES, bool FULL, int CH>
__device__ __forceinline__ void column_steps(const E* __restrict__ ents, const double* __restrict__ wts, uint32_t b,
                                             uint32_t e, uint32_t p0, double (&a)[8]) {
  uint32_t msk[CH][4];
  E idx[CH][4];
#pragma unroll
  for (int q = 0; q < CH; ++q) {
    const uint32_t p = p0 + 4 * LANES * q;
    const bool in = p < e;
    const E* src = ents + (in ? p : b);
    if (sizeof(E) == 4) {
      const uint4 v = __ldcs(reinterpret_cast<const uint4*>(src));
      const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) { idx[q][i] = w4[i] & 0xFFFFFFu; msk[q][i] = in ? (w4[i] >> 24) : 0u; }
    } else {
      const ulonglong2 v0 = __ldcs(reinterpret_cast<const ulonglong2*>(src));
      const ulonglong2 v1 = __ldcs(reinterpret_cast<const ulonglong2*>(src) + 1);
      const unsigned long long w4[4] = {v0.x, v0.y, v1.x, v1.y};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        idx[q][i] = w4[i] & 0x00FFFFFFFFFFFFFFull;
        msk[q][i] = in ? (uint32_t) (w4[i] >> 56) : 0u;
      }
    }
  }
  double w[CH][4];
#pragma unroll
  for (int q = 0; q < CH; ++q)
#pragma unroll
    for (int i = 0; i < 4; ++i) w[q][i] = __ldg(wts + idx[q][i]);
#pragma unroll
  for (int q = 0; q < CH; ++q) {
    if (FULL) {
      // padding words (and re-read quads) must not count: their mask is empty
      a[0] += (msk[q][0] ? w[q][0] : 0.0) + (msk[q][1] ? w[q][1] : 0.0);
      a[0] += (msk[q][2] ? w[q][2] : 0.0) + (msk[q][3] ? w[q][3] : 0.0);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) masked_add8(a, w[q][i], msk[q][i]);
    }
  }
}

// LANES = 8: four short items per warp (one per aligned 8-lane group); LANES = 32: one long item per warp; LANES = 2 / 1
// (VEC = 1 only): sixteen items of at most two quads / thirty-two items of one quad per warp -- a locus hit by a handful of
// classes is one item of a few entries, and half of all items are that small: on eight lanes they left seven idle.
// FULL: every entry of the item hits all H haplotypes -- a plain sum, broadcast to the H slots, no masking.
template <typename E, int VEC, int LANES, bool FULL>
__device__ __forceinline__ void column_item(const gbrs_em_dev& d, const E* __restrict__ ents, int64_t item, uint32_t b,
                                            uint32_t e) {
  constexpr int SH = 8 * (int) sizeof(E) - 8;
  constexpr E IDX = (E(1) << SH) - 1;
  const double* __restrict__ wts = d.weights;
  const int lane = threadIdx.x & 31, lane8 = lane & 7, lanex = lane & (LANES - 1);
  double a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (VEC == 1 && LANES <= 2) {
    // one quad per lane, no loop; the lane (pair) keeps all eight haplotype sums and stores them itself
    column_steps<E, LANES, FULL, 1>(ents, wts, b, e, b + 4 * lanex, a);
    if (FULL) {
      if (LANES == 2) a[0] += __shfl_xor_sync(0xFFFFFFFFu, a[0], 1);
#pragma unroll
      for (int h = 1; h < 8; ++h) a[h] = h < d.H ? a[0] : 0.0;
    } else if (LANES == 2) {
#pragma unroll
      for (int h = 0; h < 8; ++h) a[h] += __shfl_xor_sync(0xFFFFFFFFu, a[h], 1);
    }
    if (item >= 0) {
      double2* out = reinterpret_cast<double2*>(d.wit + item * GBRS_HPAD);
      if (LANES == 1) {
        out[0] = make_double2(a[0], a[1]); out[1] = make_double2(a[2], a[3]);
        out[2] = make_double2(a[4], a[5]); out[3] = make_double2(a[6], a[7]);
      } else if (lanex == 0) {
        out[0] = make_double2(a[0], a[1]); out[1] = make_double2(a[2], a[3]);
      } else {
        out[2] = make_double2(a[4], a[5]); out[3] = make_double2(a[6], a[7]);
      }
    }
    return;
  }
  if (VEC == 1) {
    // Items start at a multiple of 4 entries and are padded with empty words, so every lane fetches four consecutive
    // entries per step (one 128-bit load for 32-bit words, two for 64-bit words); two steps and their eight weight
    // gathers are in flight per lane before the adds.  When no item this warp is working on is longer than one step
    // (most short items are: the shallow loci), a single step without the loop does.
    const uint32_t longest = __reduce_max_sync(0xFFFFFFFFu, e - b);
    if (longest <= 4u * LANES) {
      column_steps<E, LANES, FULL, 1>(ents, wts, b, e, b + 4 * lanex, a);
    } else {
      for (uint32_t p0 = b + 4 * lanex; p0 < e; p0 += 4 * LANES * 2) column_steps<E, LANES, FULL, 2>(ents, wts, b, e, p0, a);
    }
  } else {
    // Model 1: eight weights per index (one per haplotype).  Lane h of an 8-lane group owns haplotype h and the whole
    // group walks the same entries: the entry words are one broadcast load, the eight weights of an entry one coalesced
    // 64-byte access (a lane gathering the full 64-byte line by itself cost four 16-byte requests per entry, each a
    // wavefront of its own: 223 us at C2), and no transposing reduction is needed at the end.
    constexpr int G = LANES >= 8 ? LANES / 8 : 1;  // lane groups sharing the item: each takes every G-th quad of entries
    const int grp = lanex >> 3;
    double acc0 = 0.0, acc1 = 0.0;
    auto quad = [&](uint32_t p, double& acc) {
      E w4[4];
      if (sizeof(E) == 4) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(ents + p));
        w4[0] = (E) v.x; w4[1] = (E) v.y; w4[2] = (E) v.z; w4[3] = (E) v.w;
      } else {
        const ulonglong2 v0 = __ldg(reinterpret_cast<const ulonglong2*>(ents + p));
        const ulonglong2 v1 = __ldg(reinterpret_cast<const ulonglong2*>(ents + p) + 1);
        w4[0] = (E) v0.x; w4[1] = (E) v0.y; w4[2] = (E) v1.x; w4[3] = (E) v1.y;
      }
      double x[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) x[i] = __ldg(wts + (size_t) (w4[i] & IDX) * GBRS_HPAD + lane8);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t bit = ((uint32_t) (w4[i] >> SH) >> lane8) & 1u;
        acc = fma(x[i], __hiloint2double(bit ? 0x3FF00000 : 0, 0), acc);
      }
    };
    uint32_t p = b + 4 * grp;
    for (; p + 4 * G < e; p += 8 * G) {  // two quads (eight gathers) in flight
      quad(p, acc0);
      quad(p + 4 * G, acc1);
    }
    if (p < e) quad(p, acc0);
    a[0] = acc0 + acc1;
  }
  double tot;
  if (VEC == 8) {
    tot = a[0];  // lane h already holds haplotype h of its group's share
  } else if (FULL && VEC == 1) {
    tot = group8_sum(a[0]);
  } else {
    tot = group8_transpose_sum(a, lane8);
  }
  if (LANES == 32) {
    tot += __shfl_xor_sync(0xFFFFFFFFu, tot, 8);
    tot += __shfl_xor_sync(0xFFFFFFFFu, tot, 16);
  }
  if (FULL && VEC == 1 && lane8 >= d.H) tot = 0.0;
  if (item >= 0 && lanex < 8) d.wit[item * GBRS_HPAD + lane8] = tot;
}

// Warp work slots over the visiting order of item_desc: [long partial | long full | short partial | short full], every part
// longest first.  A long item takes a whole warp; short items of more than two quads take eight lanes (four per warp), of
// two quads two lanes (sixteen per warp), of one quad one lane (thirty-two per warp).  The packers append the positions where
// the short parts change kind / size class as a two-descriptor trailer behind the n_items descriptors:
//   trailer[0] = {first short partial item of <= 8 words, of <= 4 words, first short full item, first short full of <= 8 words}
//   trailer[1] = {first short full item of <= 4 words, 0, 0, 0}
// Every slot holds items of one kind only, so a warp never mixes masked and plain sums.
template <typename E, int VEC>
__global__ void __launch_bounds__(kThreads, GBRS_COL_MINBLOCKS) k_column_reduce(const __grid_constant__ gbrs_em_dev d,
                                                             const E* __restrict__ ents, bool honour_done) {
  if (honour_done && d.ctrl[GBRS_CTRL_DONE]) return;
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = ((int64_t) gridDim.x * blockDim.x) >> 5;
  const uint4* __restrict__ desc = reinterpret_cast<const uint4*>(d.item_desc);
  const uint4 tr0 = __ldg(desc + d.n_items), tr1 = __ldg(desc + d.n_items + 1);
  constexpr int NSEG = 7;
  // segment starts in items, items per warp slot (model 1 keeps eight lanes per short item: lane h owns haplotype h)
  const int64_t seg_item[NSEG + 1] = {0, d.n_long_items, tr0.x, tr0.y, tr0.z, tr0.w, tr1.x, d.n_items};
  constexpr int per[NSEG] = {1, 4, VEC == 1 ? 16 : 4, VEC == 1 ? 32 : 4, 4, VEC == 1 ? 16 : 4, VEC == 1 ? 32 : 4};
  int64_t seg_slot[NSEG + 1];
  seg_slot[0] = 0;
#pragma unroll
  for (int k = 0; k < NSEG; ++k) seg_slot[k + 1] = seg_slot[k] + (seg_item[k + 1] - seg_item[k] + per[k] - 1) / per[k];
  const int64_t total_slots = seg_slot[NSEG];
  // descriptor position of the item this lane works on in slot ws (-1: none) and the slot's segment
  auto locate = [&](int64_t ws, int& seg) -> int64_t {
    seg = 0;
#pragma unroll
    for (int k = 1; k < NSEG; ++k) seg += ws >= seg_slot[k];
    int64_t pos = -1;
#pragma unroll
    for (int k = 0; k < NSEG; ++k)
      if (seg == k) {
        const int64_t i = seg_item[k] + (ws - seg_slot[k]) * per[k] + (lane / (32 / per[k]));
        pos = i < seg_item[k + 1] ? i : -1;
      }
    return pos;
  };
  const uint4 none = make_uint4(0u, 0u, 0xFFFFFFFFu, 0u);
  int64_t ws = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int seg = 0, seg_nx = 0;
  uint4 nx = none;  // descriptor of the item this lane handles in the coming iteration
  if (ws < total_slots) {
    const int64_t pos = locate(ws, seg_nx);
    if (pos >= 0) nx = __ldg(desc + pos);
  }
  for (; ws < total_slots; ws += nwarps) {
    const uint4 cur = nx;
    seg = seg_nx;
    {  // fetch the descriptor of the following slot now
      const int64_t wn = ws + nwarps;
      nx = none;
      if (wn < total_slots) {
        const int64_t pos = locate(wn, seg_nx);
        if (pos >= 0) nx = __ldg(desc + pos);
      }
    }
    const int64_t item = cur.z == 0xFFFFFFFFu ? -1 : (int64_t) cur.z;
    const uint32_t b = cur.x, e = cur.y;
    switch (seg) {  // (uniform over the warp)
      case 0:
        if (cur.w & 1u) column_item<E, VEC, 32, true>(d, ents, item, b, e);
        else column_item<E, VEC, 32, false>(d, ents, item, b, e);
        break;
      case 1: column_item<E, VEC, 8, false>(d, ents, item, b, e); break;
      case 2: column_item<E, VEC, VEC == 1 ? 2 : 8, false>(d, ents, item, b, e); break;
      case 3: column_item<E, VEC, VEC == 1 ? 1 : 8, false>(d, ents, item, b, e); break;
      case 4: column_item<E, VEC, 8, true>(d, ents, item, b, e); break;
      case 5: column_item<E, VEC, VEC == 1 ? 2 : 8, true>(d, ents, item, b, e); break;
      default: column_item<E, VEC, VEC == 1 ? 1 : 8, true>(d, ents, item, b, e); break;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Fused model-4 update over TILES (include/gbrs_em.h, tile_pack.cpp): E-step weights and the count-weighted column
// reduce of a contiguous range of classes without leaving the SM.
//   reference: normalize_reads(READ) AlignmentPropertyMatrix.py:335-342 + sum(READ) :288-298 (and the theta multiply of
//   EMfactory.py:204-208), i.e. everything between two theta updates except the division by the effective length.
// One thread block walks tiles handed out by a device-side work counter (costliest first).  The tile's inputs are
// streamed straight from its blob (every section is read once, fully coalesced: planes and sliced-ELL entries are laid out
// lane-major); what the passes share lives in shared memory (~25 KB per block, so eight blocks fit an SM): the subset-sum
// rows of the tile's loci, the class weights, the item and bucket sums.  The blob of the block's NEXT tile is prefetched
// into L2 while the current one is worked on.  Per tile:
//   phase 0 subset-sum table rows of the tile's loci -> shared (UNIT / prepare(): popcounts, so the normaliser is nnz)
//   phase 1 four neighbouring classes per thread: s = sum over their pair words of tab[l][m & 15] + tab[l][16 + (m >> 4)];
//           w = count / s -> shared
//   phase 2 one lane per work item (<= 16 local class ids of one (locus, nibble bucket)), 32 items per slice: isum = sum
//           of w[id], all gathers of a slice in flight before the adds
//   phase 3 a: the item sums of a bucket, added in item order;  b: one thread per (local locus, haplotype) adds the bucket
//           sums that contain the haplotype -> one 64-byte partial per (tile, locus) slot; k_locus_acc adds a locus'
//           slots in slot order.
// No atomics on the data path and a fixed summation order everywhere: bit-reproducible.  The per-haplotype masking of
// the two-pass column pass (4 instructions per (entry, haplotype)) is replaced by bucket sums: a partial mask costs one
// add per non-zero nibble, and the 15 + 15 + 1 bucket sums of a locus are expanded to haplotypes once per tile.
// ---------------------------------------------------------------------------------------------------------------------
#ifndef GBRS_TILE_THREADS
#define GBRS_TILE_THREADS 128
#endif
#ifndef GBRS_TILE_MINBLOCKS
#define GBRS_TILE_MINBLOCKS 8  // resident blocks per SM the tile kernel is compiled for (register budget)
#endif
constexpr int kTileThreads = GBRS_TILE_THREADS;
constexpr int kTabStride = 33;  // doubles per locus row of the shared subset table (odd: rows start on different banks)

// Every WARP owns one tile at a time and a private slice of shared memory; nothing is shared between the warps of a block,
// so there is no block barrier anywhere: a warp stalled on its loads never holds another one up.
struct TileSmem {  // byte offsets inside a warp's slice of dynamic shared memory; identical on host and device
  uint32_t w, tab, isum, slots, per_warp;
};
__host__ __device__ inline TileSmem tile_smem_layout(const gbrs_em_dev& d) {
  auto up = [](uint32_t x) { return (x + 15u) & ~15u; };
  TileSmem L;
  uint32_t o = 0;
  L.w = o; o = up(o + 8u * (uint32_t) (d.tile_max_classes + 4));  // + the always-zero slot padding ids point at
  L.tab = o; o = up(o + 8u * (uint32_t) (kTabStride * d.tile_max_loci));  // subset table (phases 0-1), then bucket sums
  L.isum = o; o = up(o + 8u * (uint32_t) (d.tile_max_items + 1));
  L.slots = o; o = up(o + 4u * (uint32_t) d.tile_max_loci);
  L.per_warp = (o + 127u) & ~127u;
  return L;
}

__device__ __forceinline__ void tile_prefetch_l2(const void* p, uint32_t bytes) {
#ifndef GBRS_SIMT_EMULATION
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
#endif
}

// sum of the weights of the entries of one lane's work item in a slice of padded length N: the N index words of the lane
// are N coalesced 64-byte rows of the slice; all gathers are in flight before the adds (fixed tree: (0+1)+(2+3) ...)
template <int N>
__device__ __forceinline__ double tile_slice_sum(const uint16_t* __restrict__ e, const double* __restrict__ w) {
  uint32_t idx[N];
#pragma unroll
  for (int i = 0; i < N; ++i) idx[i] = (uint32_t) __ldcs(e + 32 * i);
  double v[N];
#pragma unroll
  for (int i = 0; i < N; ++i) v[i] = w[idx[i]];
#pragma unroll
  for (int st = 1; st < N; st <<= 1)
#pragma unroll
    for (int i = 0; i + st < N; i += 2 * st) v[i] += v[i + st];
  return v[0];
}

// KC consecutive pair planes of four neighbouring classes (quad q): all plane words are loaded first, then all
// 2 * 4 * KC table values, then the adds -- one memory round trip per stage instead of one per plane.
template <int KC>
__device__ __forceinline__ void tile_quad_planes(const uint16_t* __restrict__ pw, const uint32_t* plane_words,
                                                 uint32_t& off, int q, const double* __restrict__ tab, double (&s)[4]) {
  uint2 v[KC];
#pragma unroll
  for (int i = 0; i < KC; ++i) {
    v[i] = __ldcs(reinterpret_cast<const uint2*>(pw + off + 4 * q));  // padding words (locus 0, empty mask) add 0.0
    off += plane_words[i];
  }
  double x[KC][4][2];
#pragma unroll
  for (int i = 0; i < KC; ++i) {
    const uint32_t wd[4] = {v[i].x & 0xFFFFu, v[i].x >> 16, v[i].y & 0xFFFFu, v[i].y >> 16};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const double* row = tab + (wd[u] >> 8) * kTabStride;
      x[i][u][0] = row[wd[u] & 15u];
      x[i][u][1] = row[16 + ((wd[u] >> 4) & 15u)];
    }
  }
#pragma unroll
  for (int i = 0; i < KC; ++i)
#pragma unroll
    for (int u = 0; u < 4; ++u) s[u] += x[i][u][0] + x[i][u][1];
}

template <bool UNIT>
__global__ void __launch_bounds__(kTileThreads, GBRS_TILE_MINBLOCKS) k_tile_em(const __grid_constant__ gbrs_em_dev d,
                                                                                const __grid_constant__ TileSmem L) {
#ifdef GBRS_SIMT_EMULATION
  static unsigned char smem[232448] __attribute__((aligned(128)));
#else
  extern __shared__ __align__(128) unsigned char smem[];
#endif
  if (!UNIT && d.ctrl[GBRS_CTRL_DONE]) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char* const mine = smem + (size_t) warp * L.per_warp;
  double* const w = reinterpret_cast<double*>(mine + L.w);
  double* const tab = reinterpret_cast<double*>(mine + L.tab);
  double* const bsum = tab;  // [local locus][32] bucket sums: the table is dead by then
  double* const isum = reinterpret_cast<double*>(mine + L.isum);
  uint32_t* const slot_of = reinterpret_cast<uint32_t*>(mine + L.slots);
  const int n_tiles = (int) d.n_tiles;
  const int n_warps = (int) (gridDim.x * (blockDim.x >> 5));
  // tiles are listed costliest first and dealt round-robin to the warps of the grid: every warp gets one tile of each
  // cost tier (no work counter: the next tile is known at once, so its descriptor and blob can be requested early)
  int cur = (int) (blockIdx.x + gridDim.x * warp);  // consecutive tiles go to different SMs
  if (cur >= n_tiles) return;
  uint32_t dword = lane < GBRS_TD_WORDS ? __ldg(d.tile_desc + (size_t) cur * GBRS_TD_WORDS + lane) : 0u;
  for (;;) {
    const int nxt = cur + n_warps;
    // the next tile: descriptor word into a register now, its blob towards L2 as soon as the descriptor is here
    const uint32_t next_dword = (nxt < n_tiles && lane < GBRS_TD_WORDS) ? __ldg(d.tile_desc + (size_t) nxt * GBRS_TD_WORDS + lane) : 0u;
    auto field = [&](int k) { return __shfl_sync(0xFFFFFFFFu, dword, k); };
    const unsigned char* const blob = d.tile_blob + (size_t) field(0) * 16;
    const uint32_t f1 = field(1), f2 = field(2), f3 = field(3);
    const int nc = (int) (f1 & 0xFFFFu), nl = (int) (f1 >> 16);
    const int n_planes = (int) (f2 & 0xFFFFu), n_runs = (int) (f2 >> 16);
    const int n_items = (int) (f3 & 0xFFFFu), n_slices = (int) (f3 >> 16);
    const unsigned char* const part_b = blob + field(4);
    const uint32_t full = field(5);
    const uint32_t* loci = reinterpret_cast<const uint32_t*>(blob + GBRS_TH_WORDS * 4);
    const uint32_t* slots = reinterpret_cast<const uint32_t*>(blob + field(8));
    const uint16_t* nplane = reinterpret_cast<const uint16_t*>(blob + field(9));
    const double* cnt = reinterpret_cast<const double*>(blob + field(10));
    const uint16_t* pw = reinterpret_cast<const uint16_t*>(blob + field(11));

    // ---- phase 0: table rows and slots of the tile's loci -----------------------------------------------------------
    if (lane == 0) w[nc] = 0.0;  // the slot padding entries point at
    for (int i = lane; i < nl * 16; i += 32) {  // 16 bytes of a 256-byte row per lane
      const int l = i >> 4, c = i & 15;
      double2 v;
      if (UNIT) v = make_double2((double) __popc((2 * c) & 15), (double) __popc((2 * c + 1) & 15));
      else v = ldg2(d.subsets + (size_t) __ldg(loci + l) * 32 + 2 * c);
      tab[l * kTabStride + 2 * c] = v.x;
      tab[l * kTabStride + 2 * c + 1] = v.y;
    }
    for (int l = lane; l < nl; l += 32) slot_of[l] = __ldg(slots + l);
    __syncwarp();

    // ---- phase 1: class weights, four neighbouring classes per lane (one 64-bit load per plane) ----------------------
    for (int q = lane; 4 * q < nc; q += 32) {
      double s[4] = {0.0, 0.0, 0.0, 0.0};
      const double2 c01 = __ldcs(reinterpret_cast<const double2*>(cnt + 4 * q));  // (the count section is padded)
      const double2 c23 = __ldcs(reinterpret_cast<const double2*>(cnt + 4 * q) + 1);
      uint32_t off = 0;
      int p0 = 0;
      while (p0 < n_planes) {
        // sizes of up to four planes at once; planes the quad's widest class (its first) has no word in end the walk
        uint32_t words[4];
        int kc = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t np = p0 + i < n_planes ? (uint32_t) __ldg(nplane + p0 + i) : 0u;
          words[i] = (np + 3u) & ~3u;
          kc += np > (uint32_t) (4 * q);
        }
        switch (kc) {
          case 0: break;
          case 1: tile_quad_planes<1>(pw, words, off, q, tab, s); break;
          case 2: tile_quad_planes<2>(pw, words, off, q, tab, s); break;
          case 3: tile_quad_planes<3>(pw, words, off, q, tab, s); break;
          default: tile_quad_planes<4>(pw, words, off, q, tab, s); break;
        }
        if (kc < 4) break;
        p0 += 4;
      }
      const double c[4] = {c01.x, c01.y, c23.x, c23.y};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = 4 * q + u;
        if (j < nc) w[j] = fast_div(c[u], s[u]);
      }
    }
    __syncwarp();  // the weights are complete, the table is no longer read
    if (nxt < n_tiles) {
      const uint32_t b0 = __shfl_sync(0xFFFFFFFFu, next_dword, 0), b7 = __shfl_sync(0xFFFFFFFFu, next_dword, 7);
      if (lane == 0) tile_prefetch_l2(d.tile_blob + (size_t) b0 * 16, b7);
    }

    // ---- phase 2: item sums, one slice (32 items, sliced-ELL entries) at a time ----------------------------------------
    for (int i = lane; i < nl * 32; i += 32) bsum[i] = 0.0;
    {
      const uint32_t* slices = reinterpret_cast<const uint32_t*>(part_b);
      const uint16_t* pos = reinterpret_cast<const uint16_t*>(part_b + field(12));
      const uint16_t* ents = reinterpret_cast<const uint16_t*>(part_b + field(15));
      for (int sidx = 0; sidx < n_slices; ++sidx) {
        const uint32_t sw = __ldg(slices + sidx);
        const int vpos = sidx * 32 + lane;
        const uint32_t at = vpos < n_items ? (uint32_t) __ldg(pos + vpos) : 0xFFFFFFFFu;
        const uint16_t* e = ents + (sw >> 5) + lane;
        double a;
        switch (sw & 31u) {
          case 1: a = tile_slice_sum<1>(e, w); break;
          case 2: a = tile_slice_sum<2>(e, w); break;
          case 3: a = tile_slice_sum<3>(e, w); break;
          case 4: a = tile_slice_sum<4>(e, w); break;
          case 6: a = tile_slice_sum<6>(e, w); break;
          case 8: a = tile_slice_sum<8>(e, w); break;
          case 12: a = tile_slice_sum<12>(e, w); break;
          default: a = tile_slice_sum<16>(e, w); break;
        }
        if (at != 0xFFFFFFFFu) isum[at] = a;  // item sums are kept in key order
      }
    }
    __syncwarp();
    // ---- phase 3a: bucket sums: the item sums of one key, in item order ------------------------------------------------
    {
      const uint16_t* run_key = reinterpret_cast<const uint16_t*>(part_b + field(13));
      const uint16_t* run_first = reinterpret_cast<const uint16_t*>(part_b + field(14));
      for (int r = lane; r < n_runs; r += 32) {
        int i = (int) __ldg(run_first + r);
        const int last = (int) __ldg(run_first + r + 1);
        const uint32_t key = (uint32_t) __ldg(run_key + r);
        double a0 = isum[i], a1 = 0.0, a2 = 0.0, a3 = 0.0;
        for (++i; i + 3 < last; i += 4) {
          a0 += isum[i];
          a1 += isum[i + 1];
          a2 += isum[i + 2];
          a3 += isum[i + 3];
        }
        for (; i < last; ++i) a0 += isum[i];
        bsum[key] = (a0 + a1) + (a2 + a3);
      }
    }
    __syncwarp();

    // ---- phase 3b: buckets -> haplotypes -> the tile's slots ---------------------------------------------------------------
    for (int q = lane; q < nl * 8; q += 32) {
      const int l = q >> 3, h = q & 7;
      const double* b = bsum + l * 32 + (h >> 2) * 16;
      const int bit = h & 3;
      double W = ((full >> h) & 1u) ? bsum[l * 32] : 0.0;
      // the eight nibble values that contain bit `bit`, ascending
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int hi = k >> bit << (bit + 1), lo = k & ((1 << bit) - 1);
        W += b[hi | (1 << bit) | lo];
      }
      d.tile_partial[(size_t) slot_of[l] * GBRS_HPAD + h] = W;
    }
    __syncwarp();  // bucket sums, item sums, weights and slots are free for the next tile
    if (nxt >= n_tiles) break;
    cur = nxt;
    dword = next_dword;
  }
}

// Subset-sum table rows of one locus from the 8 lanes holding its theta' (same sums, same order as k_subset_tables):
// lane h fills slots [4h, 4h + 4) = half (h >> 2), masks 4 * (h & 3) + q, q = 0..3 (bits 0, 1 enumerate; bits 2, 3
// are fixed by h & 3).  All 32 lanes must call (warp shuffles).
__device__ __forceinline__ void write_subset_rows(const gbrs_em_dev& d, int64_t t, int h, double v, bool valid) {
  const int base = (threadIdx.x & 31) & ~7, half4 = base + (h & 4);
  const double v0 = __shfl_sync(0xFFFFFFFFu, v, half4), v1 = __shfl_sync(0xFFFFFFFFu, v, half4 + 1);
  const double v2 = __shfl_sync(0xFFFFFFFFu, v, half4 + 2), v3 = __shfl_sync(0xFFFFFFFFu, v, half4 + 3);
  if (valid) {
    const double t2 = (h & 1) ? v2 : 0.0, t3 = (h & 2) ? v3 : 0.0;
    double* row = d.subsets + (size_t) t * 32 + 4 * h;
    *reinterpret_cast<double2*>(row) = make_double2(((0.0 + 0.0) + t2) + t3, ((v0 + 0.0) + t2) + t3);
    *reinterpret_cast<double2*>(row + 2) = make_double2(((0.0 + v1) + t2) + t3, ((v0 + v1) + t2) + t3);
  }
}

// acc[t][h] = theta[t][h] * sum_{items of t} wit[item][h]   ( = sum_n count[n] * P[n,t,h] ).  UNIT: theta == 1 (prepare).
// `wit` holds a locus' partial sums in consecutive 64-byte slots (column-pass items, or tile partials) and locus_desc lists
// the loci deepest first.  A locus with more than GBRS_DEEP_LOCUS_ITEMS slots is summed by a whole warp (lane group g takes
// slots g, g + 4, ... with four loads in flight, the groups are combined by two xor-shuffles: a fixed order); the others
// take eight lanes, four loci per warp.  The serial eight-lane walk of a 128-slot locus used to cost 32 dependent L2 round
// trips -- a 10 us floor under this kernel whatever the rest did.
// FUSE (single rank only): also theta' = acc / efflen, iso' and the block partial of sum(iso'), i.e. k_locus_update.
// Once the loop has stopped, k_converge has already flipped the ping-pong, so the theta that produced the weights in
// `wit` is the *other* buffer: a single rank simply skips, a row-sharded rank recomputes the identical local numerator
// from it (the in-place cross-rank sum that follows must always start from the local values).
// The walk both numerator kernels share: every warp takes work slots (one deep locus, or four others) round-robin,
// consecutive slots going to different blocks, and calls f(t, h, W, valid) with W = the sum of the locus' slots for
// haplotype lane h.  All 32 lanes call f in every round of their warp (f may use warp collectives); `valid` marks the
// eight lanes that finish a locus.  32-bit index arithmetic throughout: T * 8 < 2^27.
// `pre0` / `pre1` (may be null): per-(locus, haplotype) tables (theta, effective lengths) whose value for the slot's locus is
// requested together with the partial sums instead of after them -- one memory round trip less per round.
template <class F>
__device__ __forceinline__ void locus_walk(const gbrs_em_dev& d, const double* __restrict__ pre0,
                                           const double* __restrict__ pre1, F&& f) {
  const int lane = threadIdx.x & 31, h = lane & 7, grp = lane >> 3;
  const int T = d.T, n_deep = d.n_deep_loci;
  const int total_slots = n_deep + ((T - n_deep + 3) >> 2);
  const int nwarps = (int) (blockDim.x >> 5) * (int) gridDim.x;
  const uint4* __restrict__ descs = reinterpret_cast<const uint4*>(d.locus_desc);
  const double* __restrict__ wit = d.wit + h;
  int ws = (int) (threadIdx.x >> 5) * (int) gridDim.x + (int) blockIdx.x;
  auto fetch = [&](int w) {  // descriptor of this lane group's locus in slot w (.w != 0: none)
    const int di = w < n_deep ? w : n_deep + ((w - n_deep) << 2) + grp;
    return (w < total_slots && di < T) ? __ldg(descs + di) : make_uint4(0u, 0u, 0u, 0xFFFFFFFFu);
  };
  uint4 nx = fetch(ws);  // requested one round ahead
  for (; ws < total_slots; ws += nwarps) {
    const uint4 ld = nx;
    nx = fetch(ws + nwarps);
    const bool deep = ws < n_deep, have = ld.w == 0u;
    const uint32_t e = ld.z;  // (0 without a locus: the loops below do nothing)
    const bool fin = have && (!deep || grp == 0);  // the eight lanes that finish the locus
    const int po = (int) ld.x * GBRS_HPAD + h;
    const double p0 = (pre0 && fin) ? pre0[po] : 0.0, p1 = (pre1 && fin) ? pre1[po] : 0.0;
    double W = 0.0;
    if (deep) {
      uint32_t it = ld.y + (uint32_t) grp;
      for (; it + 12 < e; it += 16) {
        const double w0 = wit[(size_t) it * GBRS_HPAD], w1 = wit[(size_t) (it + 4) * GBRS_HPAD];
        const double w2 = wit[(size_t) (it + 8) * GBRS_HPAD], w3 = wit[(size_t) (it + 12) * GBRS_HPAD];
        W += (w0 + w1) + (w2 + w3);
      }
      for (; it < e; it += 4) W += wit[(size_t) it * GBRS_HPAD];
      W += __shfl_xor_sync(0xFFFFFFFFu, W, 8);
      W += __shfl_xor_sync(0xFFFFFFFFu, W, 16);
    } else {
      uint32_t it = ld.y;
      if (it + 1 == e) {  // the commonest case: one slot
        W = wit[(size_t) it * GBRS_HPAD];
      } else {
        for (; it + 3 < e; it += 4) {
          const double w0 = wit[(size_t) it * GBRS_HPAD], w1 = wit[(size_t) (it + 1) * GBRS_HPAD];
          const double w2 = wit[(size_t) (it + 2) * GBRS_HPAD], w3 = wit[(size_t) (it + 3) * GBRS_HPAD];
          W += (w0 + w1) + (w2 + w3);
        }
        for (; it < e; ++it) W += wit[(size_t) it * GBRS_HPAD];
      }
    }
    f((int) ld.x, h, W, fin, p0, p1);
  }
}

template <bool UNIT, bool FUSE>
__global__ void __launch_bounds__(kThreads, 1536 / kThreads) k_locus_acc(const gbrs_em_dev d, bool honour_done) {
  __shared__ double red[32];
  if (blockIdx.x == 0 && threadIdx.x == 0) d.ctrl[GBRS_CTRL_TILE_NEXT] = 0;
  const bool done = !UNIT && d.ctrl[GBRS_CTRL_DONE];
  if (done && (honour_done || FUSE)) return;
  const int par = d.ctrl[GBRS_CTRL_PARITY];
  const double* __restrict__ th = d.theta + (size_t) (done ? (par ^ 1) : par) * d.T * GBRS_HPAD;
  double* __restrict__ dst = d.theta + (size_t) (par ^ 1) * d.T * GBRS_HPAD;
  double* __restrict__ iso = d.iso + (size_t) (par ^ 1) * d.T;
  double* __restrict__ out = (!FUSE && d.xchg_enabled) ? xchg_acc_local(d, d.xchg_rank) : d.acc;
  double mine = 0.0;
  locus_walk(d, UNIT ? nullptr : th, FUSE ? d.efflen : nullptr, [&](int t, int h, double W, bool valid, double th_o, double len_o) {
    const int o = t * GBRS_HPAD + h;
    double a = 0.0;
    if (valid) {
      a = UNIT ? ((h < d.H) ? W : 0.0) : th_o * W;
      out[o] = a;
    }
    if (FUSE) {
      double v = 0.0;
      if (valid) {
        v = fast_div(a, len_o);
        dst[o] = v;
      }
      const double s = group8_sum(v);
      if (valid && h == 0) {
        iso[t] = s;
        mine += s;
      }
      write_subset_rows(d, t, h, v, valid);
    }
  });
  if (FUSE) {
    const double bs = block_sum(mine, red);
    if (threadIdx.x == 0) d.part[blockIdx.x] = bs;
  } else if (d.xchg_enabled) {
    xchg_signal_all(d, 0, (uint32_t) d.ctrl[GBRS_CTRL_XEPOCH] + 1u, GBRS_CTRL_TICKET + 1);
  }
}

// theta' = acc / efflen (EMfactory.py:228-232), iso'[t] = sum_h theta'[t][h], block partial sums of iso'.
// FROM_ACC = false: only (re)compute iso / partials of the current theta (after prepare / set_theta / pseudocount).
// REDUCE (row-sharded EM updates with the fused exchange): the cross-rank reduction of this rank's slice runs at the
// head of the same launch -- wait for every rank's local numerator, reduce + broadcast the slice, raise `done`, wait
// for every rank's `done`, then update -- instead of a kernel of its own.  All blocks of the grid must be resident at
// once (the launcher sizes the grid by the occupancy API): blocks waiting for `done` would otherwise keep blocks that
// still have to reduce from ever starting.
template <bool FROM_ACC, bool REDUCE = false>
__global__ void __launch_bounds__(kThreads) k_locus_update(const __grid_constant__ gbrs_em_dev d) {
  __shared__ double red[32];
  const bool xchg = FROM_ACC && d.xchg_enabled;
  if (REDUCE) {
    const uint32_t e = (uint32_t) d.ctrl[GBRS_CTRL_XEPOCH] + 1u;  // every block reads it before the last one bumps it
    xchg_wait_all(d, 0, e);
    if (d.xchg_mc) xchg_reduce_slice<true>(d);
    else xchg_reduce_slice<false>(d);
    xchg_signal_all(d, 1, e, GBRS_CTRL_TICKET + 2);
    xchg_wait_all(d, 1, e);
  } else if (xchg) {
    // fused exchange, two launches: k_xchg_reduce (same stream, just before) has set XEPOCH to the epoch of this
    // exchange; the totals are complete once every rank has raised its done flag for it
    xchg_wait_all(d, 1, (uint32_t) d.ctrl[GBRS_CTRL_XEPOCH]);
  }
  if (FROM_ACC && d.ctrl[GBRS_CTRL_DONE]) return;
  const int par = d.ctrl[GBRS_CTRL_PARITY];
  const double* __restrict__ src =
      FROM_ACC ? (xchg ? xchg_acc_total(d, d.xchg_rank) : d.acc) : d.theta + (size_t) par * d.T * GBRS_HPAD;
  double* __restrict__ dst = d.theta + (size_t) (par ^ 1) * d.T * GBRS_HPAD;
  double* __restrict__ iso = d.iso + (size_t) (FROM_ACC ? (par ^ 1) : par) * d.T;
  const int lane8 = threadIdx.x & 7;
  const int total = d.T * GBRS_HPAD;
  const int stride = (int) (gridDim.x * blockDim.x);
  const int rounds = (total + stride - 1) / stride;
  int i = (int) (blockIdx.x * blockDim.x + threadIdx.x);
  double mine = 0.0;
  for (int r = 0; r < rounds; ++r, i += stride) {
    double v = 0.0;
    const bool valid = i < total;
    if (valid) {
      v = xchg ? __ldcg(src + i) : src[i];  // totals written by peers: never through a stale L1 line
      if (FROM_ACC) {
        if (xchg) d.acc[i] = v;  // keep the summed numerator where the reports read it
        v = fast_div(v, d.efflen[i]);
        dst[i] = v;
      }
    }
    const double s = group8_sum(v);
    if (valid && lane8 == 0) {
      iso[i >> 3] = s;
      mine += s;
    }
    if (FROM_ACC) write_subset_rows(d, i >> 3, lane8, v, valid);  // theta' tables for the next row pass
  }
  const double bs = block_sum(mine, red);
  if (threadIdx.x == 0) d.part[blockIdx.x] = bs;
}

// ---------------------------------------------------------------------------------------------------------------------
// Row-sharded update, push form (xchg_enabled == 2; the default between ranks): ONE launch does the local numerator, the
// cross-rank sum and the update.  Every rank's symmetric buffer holds
//     recv  [R][slice]  doubles: recv[s] = rank s' contribution to the loci THIS rank owns (slice = its share of T * 8)
//     total [T * 8]     doubles: the summed numerator, written slice by slice by the owning ranks
//     ready [8], done [8] u32 epoch flags
//   A  numerator of the local shard; every value is stored straight into its OWNER's recv[me] with a peer store while
//      the kernel is still computing (no publish + peer-load round trip); when the whole grid is through: ready[me] = e
//      on every rank
//   B  wait for all ready flags; the owner adds its slice over the ranks in rank order -- local loads -- and stores the
//      totals into every rank's `total` (peer stores); when the grid is through: done[me] = e everywhere
//   C  wait for all done flags; theta' = total / efflen, isoform totals, subset tables, block partials (as k_locus_update)
// Each element is summed by exactly one rank in a fixed order: all ranks see the same bits and take the same stop
// decision.  All blocks must be resident (they wait for each other through the tickets): the launcher sizes the grid by
// the occupancy API.  Waits are bounded by a wall-clock limit (%globaltimer); on a timeout the error flag (3) and the stop
// flag are raised and every block leaves -- nothing continues on partial sums.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void st_relaxed_sys_f64(double* p, double v) {
  asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
// 16-byte multicast store (a store moves bits: the f32 vector form carries two doubles; multimem has no f64 vector form)
__device__ __forceinline__ void multimem_st_f64x2(double* mc, double2 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(__int_as_float(__double2loint(v.x))),
               "f"(__int_as_float(__double2hiint(v.x))), "f"(__int_as_float(__double2loint(v.y))),
               "f"(__int_as_float(__double2hiint(v.y)))
               : "memory");
}
// ---- tag form (xchg_enabled == 3): every double carries its own "arrived" flag ---------------------------------------
// The numerator is non-negative (counts >= 0, theta >= 0), so the sign bit of every transported double is free: exchange
// number e writes it as e & 1 and a reader simply polls the ELEMENT until the bit has the value of its epoch.  An 8-byte
// store is indivisible, so there is nothing to order: no ready / done flags, no grid-wide tickets, no system fences, no
// extra bytes on the wire -- the owner starts adding a locus the moment its last contribution lands, and the update of
// a locus starts the moment its total lands, while the rest of the grid is still computing.  Every element of recv and
// total is rewritten in every exchange, so the previous exchange always leaves the opposite bit behind; the zero-filled
// buffer (epoch 0) is "not arrived" for the first exchange (e = 1).
constexpr unsigned long long kTagBit = 1ull << 63;
__device__ __forceinline__ unsigned long long ld_relaxed_sys_b64(const double* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys_b64(double* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.b64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ ulonglong2 ld_relaxed_sys_b64x2(const double* p) {
  ulonglong2 v;
  asm volatile("ld.relaxed.sys.global.v2.b64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_sys_b64x2(double* p, ulonglong2 v) {
  asm volatile("st.relaxed.sys.global.v2.b64 [%0], {%1, %2};" ::"l"(p), "l"(v.x), "l"(v.y) : "memory");
}
__device__ __forceinline__ void multimem_st_b64x2(double* mc, ulonglong2 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc),
               "f"(__int_as_float((int) (uint32_t) v.x)), "f"(__int_as_float((int) (uint32_t) (v.x >> 32))),
               "f"(__int_as_float((int) (uint32_t) v.y)), "f"(__int_as_float((int) (uint32_t) (v.y >> 32)))
               : "memory");
}
__device__ __forceinline__ unsigned long long tag_bits(double a, unsigned long long tag) {
  return ((unsigned long long) __double_as_longlong(a) & ~kTagBit) | tag;
}
__device__ __forceinline__ double untag(unsigned long long v) { return __longlong_as_double((long long) (v & ~kTagBit)); }
// Bounded wait of one thread: after 256 fruitless polls it looks at the clock and at the error flag; once failed (timeout
// or another thread's failure) it never waits again, raises error 3 + the stop flag and lets the kernel run out on zeros.
struct TagWait {
  unsigned long long t0 = 0ull;
  unsigned spins = 0u;
  bool failed = false;
  __device__ __forceinline__ bool give_up(const gbrs_em_dev& d) {
    if (failed) return true;
    // back off between polls: a warp spinning flat out on system-scope loads takes issue slots and L2 request slots from
    // the blocks of the same SM that are still computing, and from the peers' stores that are trying to land
    __nanosleep(spins < 8u ? 32u : 128u);
    if ((++spins & 255u) != 0u) return false;
    const unsigned long long now = globaltimer_ns();
    if (t0 == 0ull) t0 = now;
    const unsigned long long limit = (unsigned long long) (d.xchg_timeout_ms > 0 ? d.xchg_timeout_ms : 20000) * 1000000ull;
    if (now - t0 > limit || *reinterpret_cast<volatile int32_t*>(d.ctrl + GBRS_CTRL_ERROR) == 3) {
      failed = true;
      d.ctrl[GBRS_CTRL_ERROR] = 3;
      d.ctrl[GBRS_CTRL_DONE] = 1;
      return true;
    }
    return false;
  }
};
__device__ __forceinline__ double tag_wait1(const gbrs_em_dev& d, const double* p, unsigned long long tag, TagWait& tw) {
  unsigned long long v = ld_relaxed_sys_b64(p);
  while ((v & kTagBit) != tag) {
    if (tw.give_up(d)) return 0.0;
    v = ld_relaxed_sys_b64(p);
  }
  return untag(v);
}
__host__ __device__ inline int64_t push_slice_len(const gbrs_em_dev& d) {  // doubles per owner, even
  return ((((int64_t) d.T * GBRS_HPAD + d.n_ranks - 1) / d.n_ranks) + 1) & ~(int64_t) 1;
}
__device__ __forceinline__ double* push_recv(const gbrs_em_dev& d, int owner, int src) {
  return static_cast<double*>(d.xchg_peer[owner]) + (size_t) src * push_slice_len(d);
}
__device__ __forceinline__ double* push_total(const gbrs_em_dev& d, int r) {
  return static_cast<double*>(d.xchg_peer[r]) + (size_t) d.n_ranks * push_slice_len(d);
}
__device__ __forceinline__ uint32_t* push_flags(const gbrs_em_dev& d, int r, int which /* 0 ready, 1 done */) {
  return reinterpret_cast<uint32_t*>(push_total(d, r) + (size_t) d.T * GBRS_HPAD) + which * 8;
}
// thread 0 waits until every rank's flag has reached epoch e; false (for the whole block) on a timeout
__device__ __forceinline__ bool push_wait(const gbrs_em_dev& d, int which, uint32_t e, int* s_fail) {
  if (threadIdx.x == 0) {
    const uint32_t* f = push_flags(d, d.xchg_rank, which);
    const unsigned long long t0 = globaltimer_ns();
    const unsigned long long limit = (unsigned long long) (d.xchg_timeout_ms > 0 ? d.xchg_timeout_ms : 20000) * 1000000ull;
    int fail = 0;
    for (int r = 0; r < d.n_ranks && !fail; ++r) {
      unsigned spins = 0;
      while ((int32_t) (ld_acquire_sys(f + r) - e) < 0) {
        if ((++spins & 255u) == 0u &&
            (globaltimer_ns() - t0 > limit || *reinterpret_cast<volatile int32_t*>(d.ctrl + GBRS_CTRL_ERROR) == 3)) {
          fail = 1;
          break;
        }
        __nanosleep(40);
      }
    }
    if (fail) {
      d.ctrl[GBRS_CTRL_ERROR] = 3;
      d.ctrl[GBRS_CTRL_DONE] = 1;
    }
    *s_fail = fail;
  }
  __syncthreads();
  return *s_fail == 0;
}
// every block calls it when it is through with a phase: the last one raises flag[me] = e on every rank
__device__ __forceinline__ void push_signal(const gbrs_em_dev& d, int which, uint32_t e, int ticket_slot) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();  // this block's stores (also the peer stores) are ordered before its ticket
    const int ticket = atomicAdd(d.ctrl + ticket_slot, 1);
    if (ticket == (int) gridDim.x - 1) {
      d.ctrl[ticket_slot] = 0;
      if (which == 1) d.ctrl[GBRS_CTRL_XEPOCH] = (int32_t) e;
      __threadfence_system();  // one system-scope fence for the whole grid, then the flags back to back
      for (int r = 0; r < d.n_ranks; ++r) st_relaxed_sys_u32(push_flags(d, r, which) + d.xchg_rank, e);
    }
  }
}

template <bool UNIT, bool TAG>
__global__ void __launch_bounds__(kThreads, 4) k_locus_xchg(const __grid_constant__ gbrs_em_dev d) {
  __shared__ double red[32];
  __shared__ int s_fail;
  if (blockIdx.x == 0 && threadIdx.x == 0) d.ctrl[GBRS_CTRL_TILE_NEXT] = 0;
  if (!UNIT && d.ctrl[GBRS_CTRL_DONE]) return;  // every rank takes the same decision: the epochs stay in step
  const uint32_t e = (uint32_t) d.ctrl[GBRS_CTRL_XEPOCH] + 1u;  // read by every block before the last one bumps it
  const int par = d.ctrl[GBRS_CTRL_PARITY];
  const int me = d.xchg_rank;
  const int64_t slice = push_slice_len(d);
  const int h = threadIdx.x & 7;
  const unsigned long long tag = (e & 1u) ? kTagBit : 0ull;  // tag form: the sign bit every double of this exchange carries
  TagWait tw;
  // phase time stamps of block 0 (ns since the kernel started) for bench.py: part[kStampSlot + 0..5]
  const bool stamp = blockIdx.x == 0 && threadIdx.x == 0;
  const unsigned long long t_start = stamp ? globaltimer_ns() : 0ull;
  auto mark = [&](int i) { if (stamp) d.part[kStampSlot + i] = (double) (globaltimer_ns() - t_start); };
  // tag form: slot 3 = block 0's absolute start (low 40 bits of the ns clock), slots 5..7 = the LATEST block's end of phase
  // A / B / C on the same clock (the kernel lasts as long as its slowest block, not as long as block 0)
  auto mark_max = [&](int i) {
#ifndef GBRS_SIMT_EMULATION
    if (TAG && threadIdx.x == 0)
      atomicMax(reinterpret_cast<unsigned long long*>(d.part + kStampSlot + i), globaltimer_ns() & 0xFFFFFFFFFFull);
#endif
  };
  if (TAG && stamp) {
    d.part[kStampSlot + 3] = (double) (t_start & 0xFFFFFFFFFFull);
    d.part[kStampSlot + 5] = d.part[kStampSlot + 6] = d.part[kStampSlot + 7] = 0.0;
  }
  // ---- A: local numerator, pushed to the owners ----------------------------------------------------------------------
  {
    const double* __restrict__ th = d.theta + (size_t) par * d.T * GBRS_HPAD;
    const int slice32 = (int) slice;
    locus_walk(d, UNIT ? nullptr : th, nullptr, [&](int t, int hh, double W, bool valid, double th_o, double) {
      if (valid) {
        const int o = t * GBRS_HPAD + hh;
        const double a = UNIT ? ((hh < d.H) ? W : 0.0) : th_o * W;
        const int owner = o / slice32;
        double* const slot = push_recv(d, owner, me) + (o - owner * slice32);
        if (TAG) {
          if (a < 0.0) d.ctrl[GBRS_CTRL_ERROR] = 1;  // a negative theta: not an expression estimate (the sign bit is the tag)
          st_relaxed_sys_b64(slot, tag_bits(a, tag));
        } else {
          st_relaxed_sys_f64(slot, a);
        }
      }
    });
  }
  mark(0);  // numerator of block 0 done
  mark_max(5);
  if (!TAG) push_signal(d, 0, e, GBRS_CTRL_TICKET + 1);
  // ---- B: sum my slice over the ranks, broadcast the totals ---------------------------------------------------------
  if (!TAG && !push_wait(d, 0, e, &s_fail)) return;
  if (!TAG) mark(1);  // every rank's numerator has arrived
  if (TAG) {
    const int total_n = d.T * GBRS_HPAD;
    const int lo = (int) slice * me, hi = lo + (int) slice < total_n ? lo + (int) slice : total_n;  // (both even)
    const int stride = (int) (gridDim.x * blockDim.x);
    double* const mc_total = d.xchg_mc ? static_cast<double*>(d.xchg_mc) + (size_t) d.n_ranks * slice : nullptr;
    bool first = true;
    for (int i = lo + 2 * (int) (blockIdx.x * blockDim.x + threadIdx.x); i < hi; i += 2 * stride) {
      ulonglong2 v[8];
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < d.n_ranks) v[r] = ld_relaxed_sys_b64x2(push_recv(d, me, r) + (i - lo));
      double2 sum = make_double2(0.0, 0.0);
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < d.n_ranks) {
          while ((v[r].x & kTagBit) != tag || (v[r].y & kTagBit) != tag) {  // not there yet: poll this pair
            if (tw.give_up(d)) { v[r].x = v[r].y = tag; break; }
            v[r] = ld_relaxed_sys_b64x2(push_recv(d, me, r) + (i - lo));
          }
          sum.x += untag(v[r].x);  // rank order: the same bits whichever rank owns the slice
          sum.y += untag(v[r].y);
        }
      if (first) { mark(1); first = false; }  // first pair of block 0 complete
      const ulonglong2 out = make_ulonglong2(tag_bits(sum.x, tag), tag_bits(sum.y, tag));
      if (mc_total) {
        multimem_st_b64x2(mc_total + i, out);
      } else {
#pragma unroll
        for (int r = 0; r < 8; ++r)
          if (r < d.n_ranks) st_relaxed_sys_b64x2(push_total(d, r) + i, out);
      }
    }
  } else {
    const int total_n = d.T * GBRS_HPAD;
    const int lo = (int) slice * me, hi = lo + (int) slice < total_n ? lo + (int) slice : total_n;  // (both even)
    const int stride = (int) (gridDim.x * blockDim.x);
    // with an NVSwitch multicast mapping the totals leave this GPU once instead of once per peer
    double* const mc_total = d.xchg_mc ? static_cast<double*>(d.xchg_mc) + (size_t) d.n_ranks * slice : nullptr;
    for (int i = lo + 2 * (int) (blockIdx.x * blockDim.x + threadIdx.x); i < hi; i += 2 * stride) {
      double2 v[8];
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < d.n_ranks) v[r] = ld_relaxed_sys_f64x2(push_recv(d, me, r) + (i - lo));
      double2 sum = make_double2(0.0, 0.0);
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < d.n_ranks) {
          sum.x += v[r].x;
          sum.y += v[r].y;
        }
      if (mc_total) {
        multimem_st_f64x2(mc_total + i, sum);  // one store, replicated to every rank by the switch
      } else {
#pragma unroll
        for (int r = 0; r < 8; ++r)
          if (r < d.n_ranks) st_relaxed_sys_f64x2(push_total(d, r) + i, sum);
      }
    }
  }
  mark(2);  // slice of block 0 reduced and broadcast
  mark_max(6);
  if (!TAG) push_signal(d, 1, e, GBRS_CTRL_TICKET + 2);
  // ---- C: the update, from the totals every owner has stored here -------------------------------------------------------
  if (!TAG && !push_wait(d, 1, e, &s_fail)) return;
  if (!TAG) mark(3);  // every owner's totals have arrived (tag form: nothing to wait for, the elements are polled below)
  {
    const double* __restrict__ src = push_total(d, me);
    double* __restrict__ dst = d.theta + (size_t) (par ^ 1) * d.T * GBRS_HPAD;
    double* __restrict__ iso = d.iso + (size_t) (par ^ 1) * d.T;
    const int total = d.T * GBRS_HPAD;
    const int stride = (int) (gridDim.x * blockDim.x);
    const int rounds = (total + stride - 1) / stride;
    const int i0 = (int) (blockIdx.x * blockDim.x + threadIdx.x);
    double mine = 0.0;
    // The rounds of a thread are independent: the totals (and lengths) of a whole batch of rounds are requested together and,
    // in the tag form, polled together -- the thread waits once for the slowest of them instead of once per round, and the
    // update of a batch costs one memory round trip instead of one per round.
    constexpr int BATCH = 6;
    for (int r0 = 0; r0 < rounds; r0 += BATCH) {
      unsigned long long raw[BATCH];
      double len[BATCH];
#pragma unroll
      for (int k = 0; k < BATCH; ++k) {
        const int i = i0 + (r0 + k) * stride;
        const bool valid = r0 + k < rounds && i < total;
        raw[k] = tag;
        len[k] = 1.0;
        if (valid) {  // written by peers: never through a stale L1 line
          raw[k] = TAG ? ld_relaxed_sys_b64(src + i) : (unsigned long long) __double_as_longlong(__ldcg(src + i));
          len[k] = d.efflen[i];
        }
      }
      if (TAG) {
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
          const int i = i0 + (r0 + k) * stride;
          while ((raw[k] & kTagBit) != tag) {  // not there yet (only ever true for a valid element)
            if (tw.give_up(d)) { raw[k] = tag; break; }
            raw[k] = ld_relaxed_sys_b64(src + i);
          }
        }
      }
#pragma unroll
      for (int k = 0; k < BATCH; ++k) {
        if (r0 + k < rounds) {  // (uniform over the grid: the warp collectives below are safe)
          const int i = i0 + (r0 + k) * stride;
          const bool valid = i < total;
          double v = 0.0;
          if (valid) {
            const double a = TAG ? untag(raw[k]) : __longlong_as_double((long long) raw[k]);
            d.acc[i] = a;  // the summed numerator, where the reports read it
            v = fast_div(a, len[k]);
            dst[i] = v;
          }
          const double sum8 = group8_sum(v);
          if (valid && h == 0) {
            iso[i >> 3] = sum8;
            mine += sum8;
          }
          write_subset_rows(d, i >> 3, h, v, valid);
        }
      }
    }
    const double bs = block_sum(mine, red);
    if (threadIdx.x == 0) d.part[blockIdx.x] = bs;
  }
  mark(4);  // update of block 0 done
  mark_max(7);
  if (TAG) {  // bookkeeping only, nobody waits for it: the last block to leave advances the epoch for the next launch
    __syncthreads();
    if (threadIdx.x == 0) {
      const int ticket = atomicAdd(d.ctrl + GBRS_CTRL_TICKET + 1, 1);
      if (ticket == (int) gridDim.x - 1) {
        d.ctrl[GBRS_CTRL_TICKET + 1] = 0;
        d.ctrl[GBRS_CTRL_XEPOCH] = (int32_t) e;
      }
    }
  }
}

// Stop test of EMfactory.run (EMfactory.py:267-279) on the device.
//   INIT: record sum of the current isoform totals as "prev" (after prepare / set_theta).  Launched with one block.
//   else: err = sum_t | iso'[t] * 1e6 / S' - iso[t] * 1e6 / S |, log it, flip the ping-pong, decide.  Many blocks:
//         every block re-derives S' from the same partials in the same order (bit-identical), reduces its slice of
//         the error, and the last block to arrive (ticket counter) sums the block errors in index order and takes the
//         decision -- the result does not depend on which block that is.
constexpr int kHalfSlots = GBRS_PART_SLOTS / 2;
template <bool INIT>
__global__ void __launch_bounds__(kThreads) k_converge(const gbrs_em_dev d, int nparts) {
  __shared__ double red[32];
  __shared__ int s_last;
  if (!INIT && d.ctrl[GBRS_CTRL_DONE]) return;
  double v = 0.0;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) v += d.part[i];
  const double S_new = block_sum(v, red);
  if (INIT) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
      d.scal[GBRS_SCAL_SUM_PREV] = S_new;
      d.scal[GBRS_SCAL_SUM_CUR] = S_new;
      if (!isfinite(S_new)) d.ctrl[GBRS_CTRL_ERROR] = 1;
    }
    return;
  }
  const int par = d.ctrl[GBRS_CTRL_PARITY];
  const double* __restrict__ iso_old = d.iso + (size_t) par * d.T;
  const double* __restrict__ iso_new = d.iso + (size_t) (par ^ 1) * d.T;
  const double f_new = 1000000.0 / S_new;
  const double f_old = 1000000.0 / d.scal[GBRS_SCAL_SUM_PREV];
  double e = 0.0;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < d.T; t += gridDim.x * blockDim.x)
    e += fabs(iso_new[t] * f_new - iso_old[t] * f_old);
  const double eb = block_sum(e, red);
  if (threadIdx.x == 0) {
    d.part[kHalfSlots + blockIdx.x] = eb;
    __threadfence();
    const int ticket = atomicAdd(d.ctrl + GBRS_CTRL_TICKET, 1);
    s_last = (ticket == (int) gridDim.x - 1);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  double x = 0.0;
  for (int i = threadIdx.x; i < (int) gridDim.x; i += blockDim.x) x += __ldcg(d.part + kHalfSlots + i);
  const double err = block_sum(x, red);
  if (threadIdx.x == 0) {
    const int it = d.ctrl[GBRS_CTRL_ITERS];
    if (it < d.max_iters_cap) d.err_log[it] = err;
    d.scal[GBRS_SCAL_ERR] = err;
    d.scal[GBRS_SCAL_SUM_PREV] = S_new;
    d.scal[GBRS_SCAL_SUM_CUR] = S_new;
    d.ctrl[GBRS_CTRL_ITERS] = it + 1;
    d.ctrl[GBRS_CTRL_PARITY] = par ^ 1;
    d.ctrl[GBRS_CTRL_TICKET] = 0;
    const bool bad = !isfinite(err) || !isfinite(S_new);
    if (bad) d.ctrl[GBRS_CTRL_ERROR] = 1;
    const bool go_on = !bad && err > d.scal[GBRS_SCAL_TARGET] && (it + 1) < d.ctrl[GBRS_CTRL_MAX_ITERS];
    d.ctrl[GBRS_CTRL_DONE] = go_on ? 0 : 1;
  }
}

__global__ void k_flip_parity(const gbrs_em_dev d) {
  if (threadIdx.x == 0 && blockIdx.x == 0) d.ctrl[GBRS_CTRL_PARITY] ^= 1;
}

__global__ void k_run_begin(const gbrs_em_dev d, double tol, int max_iters) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    d.ctrl[GBRS_CTRL_ITERS] = 0;
    d.ctrl[GBRS_CTRL_MAX_ITERS] = max_iters;
    d.ctrl[GBRS_CTRL_ERROR] = 0;
    d.ctrl[GBRS_CTRL_TICKET] = 0;
    d.scal[GBRS_SCAL_ERR] = 1000000.0;
    d.scal[GBRS_SCAL_TARGET] = 1000000.0 * tol;
    // while err_sum > target_err and num_iters < max_iters   (EMfactory.py:267) with err_sum = 1e6 initially
    d.ctrl[GBRS_CTRL_DONE] = (1000000.0 > 1000000.0 * tol && 0 < max_iters) ? 0 : 1;
  }
}

__global__ void k_reset_ctrl(const gbrs_em_dev d) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    d.ctrl[GBRS_CTRL_ITERS] = 0;
    d.ctrl[GBRS_CTRL_DONE] = 0;
    d.ctrl[GBRS_CTRL_ERROR] = 0;
    d.ctrl[GBRS_CTRL_PARITY] = 0;
    d.ctrl[GBRS_CTRL_MAX_ITERS] = 0;
    d.ctrl[GBRS_CTRL_PREPARED] = 1;
    d.ctrl[GBRS_CTRL_TICKET] = 0;
    d.ctrl[GBRS_CTRL_TILE_NEXT] = 0;
  }
}

// pseudocount rule of EMfactory.prepare (EMfactory.py:105-111): every haplotype of a locus with any non-zero theta gets
// +pseudocount; afterwards theta is rescaled to its original sum.  Operates on the current theta in place.
__global__ void __launch_bounds__(kThreads) k_pseudocount_add(const gbrs_em_dev d, double pc) {
  double* th = d.theta + (size_t) d.ctrl[GBRS_CTRL_PARITY] * d.T * GBRS_HPAD;
  const int lane8 = threadIdx.x & 7;
  const int64_t total = (int64_t) d.T * GBRS_HPAD;
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  const int64_t rounds = (total + stride - 1) / stride;
  int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t r = 0; r < rounds; ++r, i += stride) {
    const double v = (i < total) ? th[i] : 0.0;
    const unsigned nzmask = __ballot_sync(0xFFFFFFFFu, v != 0.0);
    const unsigned grp = (nzmask >> ((threadIdx.x & 31) & ~7)) & 0xFFu;
    if (i < total && grp != 0u && lane8 < d.H) th[i] = v + pc;
  }
}

__global__ void __launch_bounds__(kThreads) k_scale_theta(const gbrs_em_dev d, const double* num, const double* den) {
  double* th = d.theta + (size_t) d.ctrl[GBRS_CTRL_PARITY] * d.T * GBRS_HPAD;
  const double f = *num / *den;
  const int64_t total = (int64_t) d.T * GBRS_HPAD;
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) th[i] *= f;
}

__global__ void k_copy_scalar(double* dst, const double* src) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *dst = *src;
}

// report_alignment_counts (AlignmentPropertyMatrix.py:389-459); one-off, scatter with fp64 atomics.
__global__ void __launch_bounds__(kThreads) k_alignment_counts(const gbrs_em_dev d, int gene_level, int n_real_genes,
                                                               double* aln, double* uniq, double* locus_uniq) {
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t n = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; n < d.n_classes; n += stride) {
    const uint32_t b = d.rowptr[n], e = d.rowptr[n + 1];
    const double c = d.count[n];
    if (!gene_level) {
      int nz = 0;
      for (uint32_t p = b; p < e; ++p) nz += __popc(d.pairs[p] >> 24);
      const bool u1 = nz == 1, l1 = (e - b) == 1;
      for (uint32_t p = b; p < e; ++p) {
        const uint32_t w = d.pairs[p], t = w & kLocusMask, m = w >> 24;
        for (int h = 0; h < 8; ++h)
          if ((m >> h) & 1u) {
            atomicAdd(aln + (size_t) t * GBRS_HPAD + h, c);
            if (u1) atomicAdd(uniq + (size_t) t * GBRS_HPAD + h, c);
          }
        if (l1) atomicAdd(locus_uniq + t, c);
      }
    } else {
      int nb = 0, nr = 0;
      for (uint32_t p = b; p < e;) {
        const int32_t g = d.gene_of[d.pairs[p] & kLocusMask];
        uint32_t um = 0;
        for (; p < e && d.gene_of[d.pairs[p] & kLocusMask] == g; ++p) um |= d.pairs[p] >> 24;
        if (g < n_real_genes) { nb += __popc(um); ++nr; }
      }
      for (uint32_t p = b; p < e;) {
        const int32_t g = d.gene_of[d.pairs[p] & kLocusMask];
        uint32_t um = 0;
        for (; p < e && d.gene_of[d.pairs[p] & kLocusMask] == g; ++p) um |= d.pairs[p] >> 24;
        if (g >= n_real_genes) continue;
        for (int h = 0; h < 8; ++h)
          if ((um >> h) & 1u) {
            atomicAdd(aln + (size_t) g * GBRS_HPAD + h, c);
            if (nb == 1) atomicAdd(uniq + (size_t) g * GBRS_HPAD + h, c);
          }
        if (nr == 1) atomicAdd(locus_uniq + g, c);
      }
    }
  }
}

// arrays of the two-pass (row pass + column pass) kernels: all models without a tile layout, models 1-3 always
int check_twopass(const gbrs_em_dev* d, const char* who) {
  if (!d->pairs || !d->count || !d->item_desc || !d->locus_desc || !d->weights || !d->wit) {
    gbrs_set_error(std::string(who) + ": the two-pass kernels need pairs / count / item_desc / locus_desc / weights / wit");
    return GBRS_E_ARG;
  }
  return GBRS_OK;
}

int check_dev(const gbrs_em_dev* d, const char* who) {
  if (!d) { gbrs_set_error(std::string(who) + ": null descriptor"); return GBRS_E_ARG; }
  if (d->T <= 0 || d->H < 1 || d->H > GBRS_HPAD || (d->entry_bytes != 4 && d->entry_bytes != 8)) {
    gbrs_set_error(std::string(who) + ": bad descriptor shape"); return GBRS_E_ARG;
  }
  // Needed by every model.  rowptr / runptr / ent_pair / ent_run are read only by models 1-3, the wide-class row pass
  // and the alignment counts (checked there): a caller that runs model 4 only need not make them resident.
  // item_off / item_order / locus_order / locus_item_ptr describe the layout for the host; no kernel reads them.
  if (!d->theta || !d->efflen || !d->acc || !d->iso || !d->subsets || !d->part || !d->err_log || !d->scal || !d->ctrl) {
    gbrs_set_error(std::string(who) + ": null device buffer in descriptor"); return GBRS_E_ARG;
  }
  if (d->tile_blob) {  // fused model-4 path: the tile arrays must be complete
    if (!d->tile_desc || !d->tile_locus_desc || !d->tile_partial || d->n_tiles < 0 || d->tile_max_loci < 0) {
      gbrs_set_error(std::string(who) + ": incomplete tile layout in descriptor"); return GBRS_E_ARG;
    }
  } else if (int rc = check_twopass(d, who)) {
    return rc;
  }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    gbrs_set_error(std::string(who) + ": no CUDA device (there is no CPU fallback)"); return GBRS_E_CUDA;
  }
  return GBRS_OK;
}

inline int locus_grid(const gbrs_em_dev* d) {  // k_locus_update: one thread per (locus, haplotype slot)
  int g = grid_for((int64_t) d->T * GBRS_HPAD, 8);
  return g > kHalfSlots ? kHalfSlots : g;
}
inline int acc_grid(const gbrs_em_dev* d) {  // k_locus_acc: one thread per (locus, haplotype slot), 40 registers
  int g = grid_for((int64_t) d->T * GBRS_HPAD, 1536 / kThreads);
  return g > kHalfSlots ? kHalfSlots : g;
}
inline int converge_grid(const gbrs_em_dev* d) {
  int g = (d->T + 1023) / 1024;
  return g < 1 ? 1 : (g > 128 ? 128 : g);
}

int check_exchange(const gbrs_em_dev* d) {
  if (d->n_ranks < 2 || d->n_ranks > 8 || d->xchg_rank < 0 || d->xchg_rank >= d->n_ranks) {
    gbrs_set_error("fused exchange: 2..8 ranks and a valid rank index are required");
    return GBRS_E_ARG;
  }
  for (int r = 0; r < d->n_ranks; ++r)
    if (!d->xchg_peer[r]) { gbrs_set_error("fused exchange: null peer buffer"); return GBRS_E_ARG; }
  return GBRS_OK;
}

// grid of the push-form update kernel: all blocks resident, one (locus, haplotype) per thread at most
template <bool UNIT>
int push_grid(const gbrs_em_dev* d) {
  int g = d->xchg_enabled == 3 ? resident_grid(k_locus_xchg<UNIT, true>, (int64_t) d->T * GBRS_HPAD)
                               : resident_grid(k_locus_xchg<UNIT, false>, (int64_t) d->T * GBRS_HPAD);
  return g > kHalfSlots ? kHalfSlots : g;
}

template <bool UNIT>
int launch_push(const gbrs_em_dev* d, cudaStream_t s) {
  if (int rc = check_exchange(d)) return rc;
  if (d->xchg_enabled == 3) k_locus_xchg<UNIT, true><<<push_grid<UNIT>(d), kThreads, 0, s>>>(*d);
  else k_locus_xchg<UNIT, false><<<push_grid<UNIT>(d), kThreads, 0, s>>>(*d);
  GBRS_LAUNCH_CHECK("k_locus_xchg");
  return GBRS_OK;
}

// Fused NVLink exchange (descriptor flag); otherwise the caller all-reduces `acc` between the two halves of an update.
int launch_exchange(const gbrs_em_dev* d, cudaStream_t s) {
  if (!d->xchg_enabled) return GBRS_OK;
  if (int rc = check_exchange(d)) return rc;
  const int64_t slice = ((int64_t) d->T * GBRS_HPAD / 2 + d->n_ranks - 1) / d->n_ranks;
  k_xchg_reduce<<<resident_grid(k_xchg_reduce, slice), kThreads, 0, s>>>(*d);
  GBRS_LAUNCH_CHECK("k_xchg_reduce");
  return GBRS_OK;
}

template <bool UNIT, int KLO, int KHI, bool ZA>
int launch_row_m4_range(const gbrs_em_dev* d, cudaStream_t s) {
  RowPlan plan;
  int64_t units = 0;
  // the subset-sum tables of the current theta were written by the locus kernel of the previous update (or by
  // prepare / set_theta)
  for (int i = 0; i <= KHI - KLO; ++i) {  // widest bucket of the range first
    const int k = KHI - i, cpu = 32 * unr_of(k);
    units += (d->bucket_class0[k] - d->bucket_class0[k - 1] + cpu - 1) / cpu;
    plan.unit_end[i] = units;
  }
  if (units > 0) {
    k_weights_m4<UNIT, KLO, KHI, ZA><<<resident_grid(k_weights_m4<UNIT, KLO, KHI, ZA>, units * 32), kThreads, 0, s>>>(*d, plan);
    GBRS_LAUNCH_CHECK("k_weights_m4");
  }
  return GBRS_OK;
}

template <bool UNIT, bool ZA = false>
int launch_row_m4(const gbrs_em_dev* d, cudaStream_t s) {
  // one launch for all widths: here the narrow classes set the register budget (four classes per thread), so a split by
  // width buys no occupancy and would cost a launch gap (models 2-3 do split: their wide classes need 64-98 registers)
  if (int rc = launch_row_m4_range<UNIT, 1, GBRS_KMAX, ZA>(d, s)) return rc;
  const int64_t n_long = d->n_classes - d->bucket_class0[GBRS_KMAX];
  if (n_long > 0) {
    if (!d->rowptr) { gbrs_set_error("row pass: classes wider than GBRS_KMAX need rowptr"); return GBRS_E_ARG; }
    k_weights_m4_long<UNIT, ZA><<<grid_for(n_long), kThreads, 0, s>>>(*d);
    GBRS_LAUNCH_CHECK("k_weights_m4_long");
  }
  return GBRS_OK;
}

template <int VEC>
int launch_column(const gbrs_em_dev* d, const void* ents, bool honour_done, cudaStream_t s) {
  if (!ents) { gbrs_set_error("column pass: entry array missing from descriptor"); return GBRS_E_ARG; }
  if (d->n_items == 0) return GBRS_OK;
  const int64_t threads = (d->n_long_items + ((d->n_items - d->n_long_items + 3) >> 2)) * 32;  // (an upper bound: tiny items share warps)
  if (d->entry_bytes == 4)
    k_column_reduce<uint32_t, VEC><<<resident_grid(k_column_reduce<uint32_t, VEC>, threads), kThreads, 0, s>>>(
        *d, static_cast<const uint32_t*>(ents), honour_done);
  else
    k_column_reduce<unsigned long long, VEC>
        <<<resident_grid(k_column_reduce<unsigned long long, VEC>, threads), kThreads, 0, s>>>(
            *d, static_cast<const unsigned long long*>(ents), honour_done);
  GBRS_LAUNCH_CHECK("k_column_reduce");
  return GBRS_OK;
}

// fused model-4 / prepare pass over the tile layout
template <bool UNIT>
int launch_tiles(const gbrs_em_dev* d, cudaStream_t s) {
  if (d->n_tiles <= 0) return GBRS_OK;
  const TileSmem L = tile_smem_layout(*d);
  const uint32_t smem_bytes = L.per_warp * (uint32_t) (kTileThreads / 32);
  if (smem_bytes > 227u * 1024u) { gbrs_set_error("tile kernel: tile caps exceed the shared memory of an SM"); return GBRS_E_LIMIT; }
  static uint32_t attr_set = 0;  // per instantiation
  static std::unordered_map<uint32_t, int> occ_cache;
  if (smem_bytes > attr_set) {
    GBRS_CUDA(cudaFuncSetAttribute(k_tile_em<UNIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem_bytes));
    attr_set = smem_bytes;
  }
  int occ;
  auto it = occ_cache.find(smem_bytes);
  if (it == occ_cache.end()) {
    occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_tile_em<UNIT>, kTileThreads, (size_t) smem_bytes) != cudaSuccess || occ < 1) occ = 1;
    occ_cache[smem_bytes] = occ;
  } else {
    occ = it->second;
  }
  const int64_t warps_per_block = kTileThreads / 32;
  int64_t grid = (int64_t) sm_count() * occ;
  if (grid * warps_per_block > d->n_tiles) grid = (d->n_tiles + warps_per_block - 1) / warps_per_block;
  k_tile_em<UNIT><<<(int) grid, kTileThreads, smem_bytes, s>>>(*d, L);
  GBRS_LAUNCH_CHECK("k_tile_em");
  return GBRS_OK;
}

// the locus kernel reads a locus' partial sums from consecutive slots: item sums of the column pass, or tile partials
inline gbrs_em_dev locus_view(const gbrs_em_dev* d, bool tiles) {
  gbrs_em_dev v = *d;
  if (tiles) {
    v.wit = d->tile_partial;
    v.locus_desc = d->tile_locus_desc;
    v.n_deep_loci = d->tile_n_deep_loci;
  }
  return v;
}

// Row pass (E-step weights) of `model` on the two-pass layout, for d->n_classes > 0: the launches of an EM update, shared by
// the update (launch_local_impl) and the posterior (gbrs_em_posterior).  Model 4 reads the subset tables, models 1-3 the
// gene totals too (k_gene_totals before this).
int launch_row_pass(const gbrs_em_dev* d, int model, cudaStream_t s) {
  switch (model) {
    case 4: {
      const int rc4 = d->zero_count_absent ? launch_row_m4<false, true>(d, s) : launch_row_m4<false>(d, s);
      if (rc4) return rc4;
      break;
    }
    case 3:
    case 2: {
      const int64_t n_fixed = d->bucket_class0[GBRS_KMAX], n_long = d->n_classes - n_fixed;
      if (n_fixed > 0) {  // wide classes first, then the narrow ones at their own (smaller) register budget
        int rcf = model == 3 ? launch_m23_fixed<3, 4, GBRS_KMAX>(d, s) : launch_m23_fixed<2, 4, GBRS_KMAX>(d, s);
        if (!rcf) rcf = model == 3 ? launch_m23_fixed<3, 1, 3>(d, s) : launch_m23_fixed<2, 1, 3>(d, s);
        if (rcf) return rcf;
      }
      if (n_long > 0) {
        if (model == 3) k_weights_m3<<<grid_for(n_long), kThreads, 0, s>>>(*d, n_fixed);
        else k_weights_m2<<<grid_for(n_long), kThreads, 0, s>>>(*d, n_fixed);
      }
      break;
    }
    default: {
      // narrow classes thread-per-class without row pointers, the rest through the generic CSR walk
      const int64_t n_narrow = d->bucket_class0[kM1Narrow], n_rest = d->n_classes - n_narrow;
      if (n_rest > 0) k_weights_m1<<<grid_for(n_rest), kThreads, 0, s>>>(*d, n_narrow);
      int rcn = launch_m1_narrow<3>(d, s);
      if (!rcn) rcn = launch_m1_narrow<2>(d, s);
      if (!rcn) rcn = launch_m1_narrow<1>(d, s);
      if (rcn) return rcn;
      break;
    }
  }
  GBRS_LAUNCH_CHECK("k_weights");
  return GBRS_OK;
}


// ---------------------------------------------------------------------------------------------------------------------
// Posterior P[n,t,h] of one E-step on an output pattern (gbrs_em_posterior).  The row pass of the model runs unmodified on
// a copy of the descriptor whose theta is theta_src, whose counts are ones and whose work tables are scratch; then, since
// count_n P[n,t,h] = theta[t][h] W[idx(n,t,h)] (k_locus_acc sums exactly these products), every entry of the output CSC
// is theta_src[t][h] times one weight.  Error codes in ctrl[GBRS_CTRL_ERROR] of the scratch copy: 1 = zero normaliser or
// non-finite value, 2 = the output pattern is not the packed one.
// ---------------------------------------------------------------------------------------------------------------------
constexpr uint32_t kNoClass = 0xFFFFFFFFu;

__global__ void __launch_bounds__(kThreads) k_post_init(int64_t N, uint32_t* class_pos, int64_t n_classes, double* ones) {
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  const int64_t n = N > n_classes ? N : n_classes;
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    if (i < N) class_pos[i] = kNoClass;
    if (i < n_classes) ones[i] = 1.0;
  }
}

// class_pos = inverse of the packer's class order (input class id -> packed class)
__global__ void __launch_bounds__(kThreads) k_post_class_pos(int64_t n_classes, const uint32_t* __restrict__ class_id, int64_t N,
                                                             uint32_t* __restrict__ class_pos, int32_t* ctrl) {
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t p = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; p < n_classes; p += stride) {
    const uint32_t c = __ldg(class_id + p);
    if ((int64_t) c < N) class_pos[c] = (uint32_t) p;
    else atomicMax(ctrl + GBRS_CTRL_ERROR, 2);
  }
}

// Models 1-3 guard their divisions, so a class whose entries all have theta 0 gets weights 0 instead of 0 / 0.  Every
// normaliser of such a class is 0 exactly when the sum of theta over its entries is (each is bounded below by one of its
// non-zero terms): that sum, from the subset tables of theta_src.
__global__ void __launch_bounds__(kThreads) k_post_dead_classes(const gbrs_em_dev d) {
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t n = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; n < d.n_classes; n += stride) {
    const uint32_t b = __ldg(d.rowptr + n), e = __ldg(d.rowptr + n + 1);
    double s = 0.0;
    for (uint32_t p = b; p < e; ++p) s += pair_sum(d.subsets, __ldg(d.pairs + p));
    if (!(s > 0.0)) atomicMax(d.ctrl + GBRS_CTRL_ERROR, 1);
  }
}

// One warp per locus column of haplotype h, lanes over its entries (consecutive: coalesced index loads and value stores).
// idx of the entry's weight: the packed class (model 4); otherwise its pair in the class' row, found by a walk over the
// row (pairs sorted by (gene, locus)) that counts the gene runs on the way (model 3: the run, model 1: run * 8 + h).
template <typename I, int MODEL>
__global__ void __launch_bounds__(kThreads) k_post_gather(const gbrs_em_dev d, int h, int64_t N, const uint32_t* __restrict__ class_pos,
                                                          const int64_t* __restrict__ indptr, const I* __restrict__ indices,
                                                          double* __restrict__ values) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = ((int64_t) gridDim.x * blockDim.x) >> 5;
  const double* __restrict__ th = d.theta;  // theta_src (parity 0 of the scratch control block)
  int err = 0;
  for (int64_t t = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < d.T; t += nwarps) {
    const int64_t b = __ldg(indptr + t), e = __ldg(indptr + t + 1);
    if (b == e) continue;
    const double x = __ldg(th + (size_t) t * GBRS_HPAD + h);
    for (int64_t i = b + lane; i < e; i += 32) {
      const int64_t n = (int64_t) __ldg(indices + i);
      const uint32_t p = (n >= 0 && n < N) ? __ldg(class_pos + n) : kNoClass;
      double v = 0.0;
      if (n < 0 || n >= N) {
        err = 2;
      } else if (p != kNoClass) {
        size_t idx = p;
        if (MODEL != 4) {
          const uint32_t rb = __ldg(d.rowptr + p), re = __ldg(d.rowptr + p + 1);
          uint32_t q = rb, run = MODEL == 2 ? 0u : __ldg(d.runptr + p), w = 0u;
          int32_t g_prev = 0;
          for (; q < re; ++q) {
            w = __ldg(d.pairs + q);
            const uint32_t tl = w & kLocusMask;
            if (MODEL != 2) {
              const int32_t g = __ldg(d.gene_of + tl);
              if (q > rb && g != g_prev) ++run;
              g_prev = g;
            }
            if ((int64_t) tl == t) break;
          }
          idx = MODEL == 2 ? (size_t) q : (MODEL == 3 ? (size_t) run : (size_t) run * GBRS_HPAD + h);
          if (q == re || !((w >> (24 + h)) & 1u)) {
            err = 2;
            idx = 0;
          }
        }
        v = x * d.weights[idx];
        if (!isfinite(v) && err == 0) err = 1;
      }
      values[i] = v;
    }
  }
  if (err) atomicMax(d.ctrl + GBRS_CTRL_ERROR, err);
}

template <typename I>
int launch_post_gather(const gbrs_em_dev* v, int model, int h, int64_t N, const uint32_t* class_pos, const int64_t* indptr,
                       const void* indices, double* values, cudaStream_t s) {
  const I* ix = static_cast<const I*>(indices);
  const int64_t threads = (int64_t) v->T * 32;
  switch (model) {
    case 4: k_post_gather<I, 4><<<resident_grid(k_post_gather<I, 4>, threads), kThreads, 0, s>>>(*v, h, N, class_pos, indptr, ix, values); break;
    case 3: k_post_gather<I, 3><<<resident_grid(k_post_gather<I, 3>, threads), kThreads, 0, s>>>(*v, h, N, class_pos, indptr, ix, values); break;
    case 2: k_post_gather<I, 2><<<resident_grid(k_post_gather<I, 2>, threads), kThreads, 0, s>>>(*v, h, N, class_pos, indptr, ix, values); break;
    default: k_post_gather<I, 1><<<resident_grid(k_post_gather<I, 1>, threads), kThreads, 0, s>>>(*v, h, N, class_pos, indptr, ix, values); break;
  }
  GBRS_LAUNCH_CHECK("k_post_gather");
  return GBRS_OK;
}

// scratch of gbrs_em_posterior: byte offsets (each 256-byte aligned)
struct PostScratch {
  int64_t ctrl, part, iso, subsets, gene_hap, gamma, count, weights, class_pos, total;
};
inline PostScratch post_scratch(const gbrs_em_dev* d, int model, int64_t N) {
  auto up = [](int64_t b) { return (b + 255) & ~int64_t(255); };
  const int64_t runs = d->n_runs, T = d->T;
  int64_t wlen = d->n_classes > d->n_pairs ? d->n_classes : d->n_pairs;
  if (runs > wlen) wlen = runs;
  if (model == 1 && 8 * runs > wlen) wlen = 8 * runs;
  wlen += 8;
  PostScratch L;
  int64_t o = 0;
  L.ctrl = o;      o += up(16 * sizeof(int32_t));
  L.part = o;      o += up(GBRS_PART_SLOTS * sizeof(double));
  L.iso = o;       o += up(T * sizeof(double));
  L.subsets = o;   o += up(T * 32 * sizeof(double));
  L.gene_hap = o;  o += up((int64_t) (d->n_gene_ids > 1 ? d->n_gene_ids : 1) * GBRS_HPAD * sizeof(double));
  L.gamma = o;     o += up(T * sizeof(double));
  L.count = o;     o += up((d->n_classes > 1 ? d->n_classes : 1) * sizeof(double));
  L.weights = o;   o += up(wlen * sizeof(double));
  L.class_pos = o; o += up((N > 1 ? N : 1) * sizeof(uint32_t));
  L.total = o;
  return L;
}

__global__ void __launch_bounds__(kThreads) k_copy_theta(const gbrs_em_dev d, int previous, double* dst) {
  const double* __restrict__ src = d.theta + (size_t) (d.ctrl[GBRS_CTRL_PARITY] ^ previous) * d.T * GBRS_HPAD;
  const int64_t total = (int64_t) d.T * GBRS_HPAD;
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) dst[i] = src[i];
}

// ---------------------------------------------------------------------------------------------------------------------
// Bootstrap resampler (gbrs_boot_guide / gbrs_boot_resample; the contract is in include/gbrs_em.h).  Draws come from
// Philox4x32-10 (Salmon et al., SC'11; the constants of Random123 and of curand), written out here so that the host SIMT
// shim compiles it as it is.  A draw u is read floor(u * M / 2^64), the high half of the product; its class is an upper bound on the
// int64 prefix of the counts.  A plain binary search over the whole prefix (40 MB at C2) is a chain of ~23 dependent
// gathers per draw; the guide table cuts it to the few classes between two guide entries: with G = 2^bits entries,
// entry g = class of read floor(g * M / G) = class of the draw g << (64 - bits), and a draw u lies between entries
// u >> (64 - bits) and the next one (both readings are monotone in u).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kBootGuideBitsMax = 24;

// high halves of the 32 x 32 and 64 x 64-bit products: the hardware intrinsics on the device, the same arithmetic in
// portable C++ where the kernels are compiled for the host (__CUDA_ARCH__ undefined)
__device__ __forceinline__ uint32_t mul32hi(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t) (((uint64_t) a * b) >> 32);
#endif
}

__device__ __forceinline__ uint64_t mul64hi(uint64_t a, uint64_t b) {
#ifdef __CUDA_ARCH__
  return __umul64hi(a, b);
#else
  return (uint64_t) (((unsigned __int128) a * b) >> 64);
#endif
}

__device__ __forceinline__ void philox4x32_10(uint32_t (&x)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = mul32hi(0xD2511F53u, x[0]), lo0 = 0xD2511F53u * x[0];
    const uint32_t hi1 = mul32hi(0xCD9E8D57u, x[2]), lo1 = 0xCD9E8D57u * x[2];
    const uint32_t y0 = hi1 ^ x[1] ^ k0, y2 = hi0 ^ x[3] ^ k1;
    x[0] = y0;
    x[1] = lo1;
    x[2] = y2;
    x[3] = lo0;
    k0 += 0x9E3779B9u;  // key schedule (the bump after the last round is never used)
    k1 += 0xBB67AE85u;
  }
}

// first class n in [lo, hi] with P[n] > k (the caller guarantees P[hi] > k)
__device__ __forceinline__ int64_t boot_upper_bound(const int64_t* __restrict__ P, int64_t lo, int64_t hi, int64_t k) {
  while (lo < hi) {
    const int64_t mid = lo + ((hi - lo) >> 1);
    if (__ldg(P + mid) > k) hi = mid;
    else lo = mid + 1;
  }
  return lo;
}

__global__ void __launch_bounds__(kThreads) k_boot_guide(const int64_t* __restrict__ P, int64_t N, uint64_t M, int bits,
                                                         uint32_t* __restrict__ guide) {
  const int64_t G = int64_t(1) << bits, stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t g = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; g <= G; g += stride) {
    int64_t c = N - 1;  // entry G: past every read
    if (g < G) {
      const uint64_t u = bits ? (uint64_t) g << (64 - bits) : 0ull;
      c = boot_upper_bound(P, 0, N - 1, (int64_t) mul64hi(u, M));
    }
    guide[g] = (uint32_t) c;
  }
}

// one thread per draw pair (grid-stride): Philox, the two reads, their classes, one integer atomic per draw
__global__ void __launch_bounds__(kThreads) k_boot_sample(const int64_t* __restrict__ P, uint64_t M, int bits,
                                                          const uint32_t* __restrict__ guide, uint64_t seed, uint32_t rep,
                                                          unsigned long long* __restrict__ hist) {
  const uint64_t n_pairs = (M + 1) >> 1, stride = (uint64_t) gridDim.x * blockDim.x;
  const uint32_t k0 = (uint32_t) seed, k1 = (uint32_t) (seed >> 32);
  for (uint64_t j = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; j < n_pairs; j += stride) {
    uint32_t x[4] = {(uint32_t) j, (uint32_t) (j >> 32), rep, 0u};
    philox4x32_10(x, k0, k1);
    const uint64_t u[2] = {(uint64_t) x[0] | ((uint64_t) x[1] << 32), (uint64_t) x[2] | ((uint64_t) x[3] << 32)};
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      if (2 * j + q >= M) break;  // odd M: the second draw of the last pair is unused
      const int64_t k = (int64_t) mul64hi(u[q], M);
      const uint64_t g = bits ? u[q] >> (64 - bits) : 0ull;
      const int64_t n = boot_upper_bound(P, __ldg(guide + g), __ldg(guide + g + 1), k);
      atomicAdd(hist + n, 1ull);
    }
  }
}

// replicate counts in packed class order
__global__ void __launch_bounds__(kThreads) k_boot_scatter(const unsigned long long* __restrict__ hist,
                                                           const uint32_t* __restrict__ class_id, int64_t n_classes,
                                                           double* __restrict__ count) {
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t p = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; p < n_classes; p += stride)
    count[p] = (double) hist[__ldg(class_id + p)];
}

inline int boot_bits(int64_t N) {
  int b = 0;
  while (b < kBootGuideBitsMax && (int64_t(1) << b) < N) ++b;
  return b;
}

// scratch of the resampler: histogram uint64 [N] | guide uint32 [G + 1] (each 256-byte aligned)
struct BootScratch {
  int64_t hist, guide, total;
};
inline BootScratch boot_scratch(int64_t N) {
  auto up = [](int64_t b) { return (b + 255) & ~int64_t(255); };
  BootScratch L;
  L.hist = 0;
  L.guide = up(N * (int64_t) sizeof(unsigned long long));
  L.total = L.guide + up(((int64_t(1) << boot_bits(N)) + 1) * (int64_t) sizeof(uint32_t));
  return L;
}

int check_boot(const int64_t* prefix, int64_t N, int64_t M, void* scratch, int64_t scratch_bytes, const char* who) {
  if (!prefix || !scratch || N < 1 || N >= (int64_t(1) << 32) || M < 1 || M > (int64_t(1) << 53)) {
    gbrs_set_error(std::string(who) + ": bad argument (1 <= N < 2^32 classes and 1 <= M <= 2^53 reads)");
    return GBRS_E_ARG;
  }
  if (scratch_bytes < boot_scratch(N).total) { gbrs_set_error(std::string(who) + ": scratch too small"); return GBRS_E_ARG; }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { gbrs_set_error(std::string(who) + ": no CUDA device (there is no CPU fallback)"); return GBRS_E_CUDA; }
  return GBRS_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Bootstrap summaries (gbrs_boot_derive / gbrs_boot_summarize; the contract is in include/gbrs_em.h and DESIGN.md 7.3).
// Derive turns the replicates' [B][T][8] theta or numerator into the [B][E] values of one (level, quantity), element
// e = h * L + l (h = H: the total column).  Summarize reduces each column of a [B][E] matrix: mean and sd in replicate
// order, then a bitonic sort in shared memory (NaN last) for the quantiles, interpolated as numpy's method="linear".
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kBootSumThreads = 512;               // k_bsum_tpm: one block per replicate row
constexpr int kBootSummarySmem = 232448;           // dynamic shared memory of one summarize block (227 KB)
constexpr int kBootSummaryMaxTile = 64;            // columns per summarize block

__device__ __forceinline__ double boot_nan() { return __longlong_as_double(0x7FF8000000000000LL); }

// one thread per (replicate, locus): the level's values x[h] (isoform: the locus line; gene: the sum over the gene's
// loci in gene_loci order), then by `what`: 0 raw x[h] (TPM before scaling), 1 x[h] and the total column, 2 shares
__global__ void __launch_bounds__(kThreads) k_bsum_level(const double* __restrict__ src, int64_t B, int32_t T, int32_t H,
                                                         int32_t L, const uint32_t* __restrict__ gene_ptr,
                                                         const uint32_t* __restrict__ gene_loci, int what,
                                                         double* __restrict__ out) {
  const int64_t total = B * L, stride = (int64_t) gridDim.x * blockDim.x;
  const int64_t E = (int64_t) L * (what == 2 ? H : H + 1);
  for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int64_t b = i / L, l = i - b * L;
    const double* rep = src + (size_t) b * T * GBRS_HPAD;
    double x[GBRS_HPAD];
    if (!gene_ptr) {
      load8(rep + (size_t) l * GBRS_HPAD, x);
    } else {
#pragma unroll
      for (int h = 0; h < GBRS_HPAD; ++h) x[h] = 0.0;
      for (uint32_t p = __ldg(gene_ptr + l), e = __ldg(gene_ptr + l + 1); p < e; ++p) {
        double v[GBRS_HPAD];
        load8(rep + (size_t) __ldg(gene_loci + p) * GBRS_HPAD, v);
#pragma unroll
        for (int h = 0; h < GBRS_HPAD; ++h) x[h] += v[h];
      }
    }
    double* row = out + (size_t) b * E;
    double sum = 0.0;
#pragma unroll
    for (int h = 0; h < GBRS_HPAD; ++h)
      if (h < H) sum += x[h];
#pragma unroll
    for (int h = 0; h < GBRS_HPAD; ++h)
      if (h < H) row[(int64_t) h * L + l] = what != 2 ? x[h] : (sum != 0.0 ? x[h] / sum : boot_nan());
    if (what == 1) row[(int64_t) H * L + l] = sum;
  }
}

// TPM: per replicate row (one block each), the sum S of its H * L raw values in a fixed order (thread-strided partial
// sums, then a tree over the block), then value = x * (1e6 / S) and the total column
__global__ void __launch_bounds__(kBootSumThreads) k_bsum_tpm(int64_t B, int32_t H, int32_t L, double* __restrict__ out) {
  __shared__ double red[kBootSumThreads];
  const int64_t n = (int64_t) H * L, E = (int64_t) (H + 1) * L;
  for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
    double* row = out + (size_t) b * E;
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += row[i];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int w = kBootSumThreads / 2; w > 0; w >>= 1) {
      if ((int) threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
      __syncthreads();
    }
    const double f = 1000000.0 / red[0];
    for (int64_t l = threadIdx.x; l < L; l += blockDim.x) {
      double t = 0.0;
      for (int h = 0; h < H; ++h) {
        const double v = __dmul_rn(row[(int64_t) h * L + l], f);
        row[(int64_t) h * L + l] = v;
        t += v;
      }
      row[(int64_t) H * L + l] = t;
    }
    __syncthreads();  // red[0] is rewritten by the next row
  }
}

struct BootQuantiles {
  double q[GBRS_BOOT_MAX_QUANTILES];
};

// compensated sum (Neumaier) in the order of the adds: the error of a column of 16k replicates stays at a few ulp
struct BootSum {
  double s = 0.0, c = 0.0;
  __device__ __forceinline__ void add(double x) {
    const double t = __dadd_rn(s, x);
    c = __dadd_rn(c, fabs(s) >= fabs(x) ? __dadd_rn(__dadd_rn(s, -t), x) : __dadd_rn(__dadd_rn(x, -t), s));
    s = t;
  }
  __device__ __forceinline__ double value() const { return __dadd_rn(s, c); }
};

// NaN sorts after every number
__device__ __forceinline__ bool boot_after(double a, double b) { return a > b || (a != a && b == b); }

// numpy.quantile(method="linear") of the n sorted numbers s[0..n): virtual index (n - 1) q, _lerp with its t >= 0.5
// branch (numpy/lib/_function_base_impl.py), every operation rounded on its own (no FMA)
__device__ __forceinline__ double boot_quantile(const double* s, int n, double q) {
  const double v = __dmul_rn((double) (n - 1), q);
  if (v >= (double) (n - 1)) return s[n - 1];
  const double lo = floor(v);
  const int i = (int) lo;
  const double a = s[i], b = s[i + 1], t = __dadd_rn(v, -lo);
  const double diff = __dadd_rn(b, -a);
  return t >= 0.5 ? __dadd_rn(b, -__dmul_rn(diff, __dadd_rn(1.0, -t))) : __dadd_rn(a, __dmul_rn(diff, t));
}

// one block per tile of K columns (grid-stride over tiles): the tile is loaded transposed into shared memory (column k
// at k * ld, ld = P + 1 with P the next power of two >= B, NaN padding), reads coalesced along E for each replicate;
// thread k then takes mean, sd and n of column k in replicate order; a bitonic sort of all K columns follows, and the
// quantiles are read off the sorted columns
__global__ void __launch_bounds__(kThreads) k_boot_summarize(const double* __restrict__ values, int64_t B, int64_t E, int P,
                                                             int K, const __grid_constant__ BootQuantiles Q, int nq, double* __restrict__ mean,
                                                             double* __restrict__ sd, double* __restrict__ qout,
                                                             int32_t* __restrict__ nout) {
#ifdef GBRS_SIMT_EMULATION
  static double s[kBootSummarySmem / sizeof(double)];
#else
  extern __shared__ double s[];
#endif
  const int ld = P + 1, half = P >> 1;
  int half_bits = 0;
  while ((1 << half_bits) < half) ++half_bits;
  const int64_t n_tiles = (E + K - 1) / K;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t e0 = tile * K;
    const int64_t cells = (int64_t) K * P;
    for (int64_t i = threadIdx.x; i < cells; i += blockDim.x) {
      const int64_t b = i / K;
      const int k = (int) (i - b * K);
      s[k * ld + b] = (b < B && e0 + k < E) ? values[(size_t) b * E + e0 + k] : boot_nan();
    }
    __syncthreads();
    if ((int) threadIdx.x < K && e0 + threadIdx.x < E) {
      const double* c = s + threadIdx.x * ld;
      BootSum sum;
      int n = 0;
      for (int64_t b = 0; b < B; ++b)
        if (c[b] == c[b]) { sum.add(c[b]); ++n; }
      const double m = n > 0 ? sum.value() / n : boot_nan();
      BootSum ss;
      for (int64_t b = 0; b < B; ++b)
        if (c[b] == c[b]) { const double dv = __dadd_rn(c[b], -m); ss.add(__dmul_rn(dv, dv)); }
      const int64_t e = e0 + threadIdx.x;
      mean[e] = m;
      sd[e] = n > 1 ? sqrt(ss.value() / (n - 1)) : boot_nan();
      if (nout) nout[e] = n;
    }
    __syncthreads();
    for (int size = 2; size <= P; size <<= 1)
      for (int st = size >> 1; st > 0; st >>= 1) {
        for (int64_t i = threadIdx.x; i < (int64_t) K * half; i += blockDim.x) {
          const int k = (int) (i >> half_bits), j = (int) (i & (half - 1));
          const int lo = 2 * st * (j / st) + (j % st), hi = lo + st;
          double* c = s + k * ld;
          const double a = c[lo], b = c[hi];
          if ((lo & size) == 0 ? boot_after(a, b) : boot_after(b, a)) { c[lo] = b; c[hi] = a; }
        }
        __syncthreads();
      }
    for (int64_t i = threadIdx.x; i < (int64_t) K * nq; i += blockDim.x) {
      const int k = (int) (i % K), j = (int) (i / K);
      const int64_t e = e0 + k;
      if (e >= E) continue;
      const double* c = s + k * ld;
      int n = 0;  // the defined values are the sorted prefix
      for (int step = P; step > 0; step >>= 1)
        if (n + step <= P && c[n + step - 1] == c[n + step - 1]) n += step;
      qout[(size_t) j * E + e] = n > 0 ? boot_quantile(c, n, Q.q[j]) : boot_nan();
    }
    __syncthreads();  // the next tile overwrites the columns
  }
}

inline int boot_pow2(int64_t B) {
  int P = 2;
  while (P < B) P <<= 1;
  return P;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------------------------
extern "C" int gbrs_em_prepare_local(const gbrs_em_dev* d, void* stream) {
  if (int rc = check_dev(d, "gbrs_em_prepare_local")) return rc;
  NvtxRange nvtx_prep("gbrs:prepare");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  k_reset_ctrl<<<1, 32, 0, s>>>(*d);
  GBRS_LAUNCH_CHECK("k_reset_ctrl");
  const bool tiles = d->tile_blob != nullptr;
  if (tiles) {
    if (int rc = launch_tiles<true>(d, s)) return rc;
  } else {
    if (int rc = launch_row_m4<true>(d, s)) return rc;
    if (int rc = launch_column<1>(d, d->ent_cls, false, s)) return rc;
  }
  const gbrs_em_dev lv = locus_view(d, tiles);
  if (d->n_ranks > 1 && d->xchg_enabled >= 2) return launch_push<true>(&lv, s);  // numerator + exchange + theta0 in one launch
  k_locus_acc<true, false><<<acc_grid(d), kThreads, 0, s>>>(lv, false);
  GBRS_LAUNCH_CHECK("k_locus_acc<unit>");
  return GBRS_OK;
}

extern "C" int gbrs_em_prepare_finish(const gbrs_em_dev* d, double pseudocount, void* stream) {
  if (int rc = check_dev(d, "gbrs_em_prepare_finish")) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int lg = locus_grid(d);
  if (d->n_ranks > 1 && d->xchg_enabled >= 2) {
    lg = push_grid<true>(d);  // gbrs_em_prepare_local has done exchange and update already; its blocks wrote the partials
  } else {
    if (int rc = launch_exchange(d, s)) return rc;
    // theta[1] = acc / efflen ; then make it the current estimate
    k_locus_update<true><<<lg, kThreads, 0, s>>>(*d);
    GBRS_LAUNCH_CHECK("k_locus_update");
  }
  k_flip_parity<<<1, 32, 0, s>>>(*d);
  GBRS_LAUNCH_CHECK("k_flip_parity");
  k_converge<true><<<1, kThreads, 0, s>>>(*d, lg);
  GBRS_LAUNCH_CHECK("k_converge<init>");
  if (pseudocount > 0.0) {
    // scal[4] keeps the original sum
    k_copy_scalar<<<1, 32, 0, s>>>(d->scal + 4, d->scal + GBRS_SCAL_SUM_CUR);
    k_pseudocount_add<<<lg, kThreads, 0, s>>>(*d, pseudocount);
    GBRS_LAUNCH_CHECK("k_pseudocount_add");
    k_locus_update<false><<<lg, kThreads, 0, s>>>(*d);
    k_converge<true><<<1, kThreads, 0, s>>>(*d, lg);
    k_scale_theta<<<lg, kThreads, 0, s>>>(*d, d->scal + 4, d->scal + GBRS_SCAL_SUM_CUR);
    GBRS_LAUNCH_CHECK("k_scale_theta");
    k_locus_update<false><<<lg, kThreads, 0, s>>>(*d);
    k_converge<true><<<1, kThreads, 0, s>>>(*d, lg);
    GBRS_LAUNCH_CHECK("pseudocount chain");
  }
  k_subset_tables<<<resident_grid(k_subset_tables, (int64_t) d->T * 32), kThreads, 0, s>>>(*d);
  GBRS_LAUNCH_CHECK("k_subset_tables");
  return GBRS_OK;
}

extern "C" int gbrs_em_set_theta(const gbrs_em_dev* d, const double* theta_dev, void* stream) {
  if (int rc = check_dev(d, "gbrs_em_set_theta")) return rc;
  if (!theta_dev) { gbrs_set_error("gbrs_em_set_theta: null theta"); return GBRS_E_ARG; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  k_reset_ctrl<<<1, 32, 0, s>>>(*d);
  GBRS_LAUNCH_CHECK("k_reset_ctrl");
  GBRS_CUDA(cudaMemcpyAsync(d->theta, theta_dev, sizeof(double) * (size_t) d->T * GBRS_HPAD, cudaMemcpyDeviceToDevice, s));
  const int lg = locus_grid(d);
  k_locus_update<false><<<lg, kThreads, 0, s>>>(*d);
  GBRS_LAUNCH_CHECK("k_locus_update<refresh>");
  k_converge<true><<<1, kThreads, 0, s>>>(*d, lg);
  GBRS_LAUNCH_CHECK("k_converge<init>");
  k_subset_tables<<<resident_grid(k_subset_tables, (int64_t) d->T * 32), kThreads, 0, s>>>(*d);
  GBRS_LAUNCH_CHECK("k_subset_tables");
  return GBRS_OK;
}

extern "C" int gbrs_em_read_ctrl(const gbrs_em_dev* d, void* stream, int32_t* ctrl_host, double* scal_host) {
  if (int rc = check_dev(d, "gbrs_em_read_ctrl")) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (ctrl_host) GBRS_CUDA(cudaMemcpyAsync(ctrl_host, d->ctrl, sizeof(int32_t) * 16, cudaMemcpyDeviceToHost, s));
  if (scal_host) GBRS_CUDA(cudaMemcpyAsync(scal_host, d->scal, sizeof(double) * 8, cudaMemcpyDeviceToHost, s));
  GBRS_CUDA(cudaStreamSynchronize(s));
  return GBRS_OK;
}

extern "C" int gbrs_em_current_theta(const gbrs_em_dev* d, void* stream, double** theta_dev) {
  if (!theta_dev) { gbrs_set_error("gbrs_em_current_theta: null out pointer"); return GBRS_E_ARG; }
  int32_t ctrl[16];
  if (int rc = gbrs_em_read_ctrl(d, stream, ctrl, nullptr)) return rc;
  *theta_dev = d->theta + (size_t) ctrl[GBRS_CTRL_PARITY] * d->T * GBRS_HPAD;
  return GBRS_OK;
}

extern "C" int gbrs_em_run_begin(const gbrs_em_dev* d, double tol, int max_iters, void* stream) {
  if (int rc = check_dev(d, "gbrs_em_run_begin")) return rc;
  if (max_iters < 0 || max_iters > d->max_iters_cap) {
    gbrs_set_error("gbrs_em_run_begin: max_iters exceeds the err_log capacity of the descriptor"); return GBRS_E_ARG;
  }
  k_run_begin<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(*d, tol, max_iters);
  GBRS_LAUNCH_CHECK("k_run_begin");
  return GBRS_OK;
}

struct gbrs_prof {
  int capacity = 0, used = 0;
  std::vector<cudaEvent_t> ev;  // 4 per recorded update: before row pass, after row pass, after column pass, after acc
};

extern "C" int gbrs_prof_create(int capacity, gbrs_prof_t* out) {
  if (!out || capacity < 1) { gbrs_set_error("gbrs_prof_create: bad argument"); return GBRS_E_ARG; }
  auto* p = new gbrs_prof();
  p->capacity = capacity;
  p->ev.resize((size_t) capacity * 4);
  for (auto& e : p->ev) {
    cudaError_t rc = cudaEventCreate(&e);
    if (rc != cudaSuccess) { gbrs_set_error(std::string("cudaEventCreate: ") + cudaGetErrorString(rc)); delete p; return GBRS_E_CUDA; }
  }
  *out = p;
  return GBRS_OK;
}

extern "C" int gbrs_prof_read(gbrs_prof_t p, double* ms_row, double* ms_col, double* ms_acc, int32_t* n) {
  if (!p) { gbrs_set_error("gbrs_prof_read: null"); return GBRS_E_ARG; }
  double r = 0, c = 0, a = 0;
  for (int i = 0; i < p->used; ++i) {
    float x = 0;
    GBRS_CUDA(cudaEventSynchronize(p->ev[4 * i + 3]));
    GBRS_CUDA(cudaEventElapsedTime(&x, p->ev[4 * i + 0], p->ev[4 * i + 1])); r += x;
    GBRS_CUDA(cudaEventElapsedTime(&x, p->ev[4 * i + 1], p->ev[4 * i + 2])); c += x;
    GBRS_CUDA(cudaEventElapsedTime(&x, p->ev[4 * i + 2], p->ev[4 * i + 3])); a += x;
  }
  if (ms_row) *ms_row = r;
  if (ms_col) *ms_col = c;
  if (ms_acc) *ms_acc = a;
  if (n) *n = p->used;
  p->used = 0;
  return GBRS_OK;
}

extern "C" int gbrs_prof_free(gbrs_prof_t p) {
  if (p) {
    for (auto& e : p->ev) cudaEventDestroy(e);
    delete p;
  }
  return GBRS_OK;
}

static int launch_local_impl(const gbrs_em_dev* d, int model, void* stream, gbrs_prof* prof, bool estep_only = false);

extern "C" int gbrs_em_launch_local(const gbrs_em_dev* d, int model, void* stream) {
  return launch_local_impl(d, model, stream, nullptr);
}

// E-step alone (EMfactory.update_probability_at_read_level, EMfactory.py:146-212): the numerator sum_n c[n] P[n,t,h] of
// this rank's shard goes to `acc` and NOTHING else changes -- no theta', no isoform totals, no subset tables, no exchange
// flags -- so it may be called any number of times between updates, exactly like the reference's method.
extern "C" int gbrs_em_launch_estep(const gbrs_em_dev* d, int model, void* stream) {
  if (!d) { gbrs_set_error("gbrs_em_launch_estep: null descriptor"); return GBRS_E_ARG; }
  gbrs_em_dev plain = *d;
  plain.xchg_enabled = 0;  // the caller sums `acc` over ranks (if any) itself
  return launch_local_impl(&plain, model, stream, nullptr, true);
}

extern "C" int gbrs_em_launch_local_profiled(const gbrs_em_dev* d, int model, void* stream, gbrs_prof_t prof) {
  if (!prof || prof->used >= prof->capacity) { gbrs_set_error("gbrs_em_launch_local_profiled: profile buffer full"); return GBRS_E_ARG; }
  return launch_local_impl(d, model, stream, prof);
}

static int launch_local_impl(const gbrs_em_dev* d, int model, void* stream, gbrs_prof* prof, bool estep_only) {
  if (int rc = check_dev(d, "gbrs_em_launch_local")) return rc;
  if (model < 1 || model > 4) {
    gbrs_set_error("The read normalization model should be 1, 2, 3, or 4."); return GBRS_E_ARG;  // EMfactory.py:209-212
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool honour_done = (d->n_ranks <= 1 || d->xchg_enabled >= 2) && !estep_only;
  const bool tiles = model == 4 && d->tile_blob != nullptr;
  int rc = GBRS_OK;
  if (!tiles && d->tile_blob)
    if (int rc2 = check_twopass(d, "gbrs_em_launch_local")) return rc2;
  if (model != 4) {
    if (!d->gene_of || !d->gene_ptr || !d->gene_loci || !d->gene_hap || !d->gamma || !d->runptr) {
      gbrs_set_error("Group information matrix is missing.");  // AlignmentPropertyMatrix.py:345-346
      return GBRS_E_ARG;
    }
    if (!d->rowptr || !d->ent_pair || !d->ent_run) {
      gbrs_set_error("models 1-3 need rowptr / ent_pair / ent_run in the descriptor");
      return GBRS_E_ARG;
    }
    k_gene_totals<<<grid_for((int64_t) d->n_gene_ids * 8), kThreads, 0, s>>>(*d);
    GBRS_LAUNCH_CHECK("k_gene_totals");
  }
  const int cg = grid_for(d->n_classes);
  cudaEvent_t* ev = prof ? &prof->ev[(size_t) prof->used * 4] : nullptr;
  if (ev) GBRS_CUDA(cudaEventRecord(ev[0], s));
  {
  NvtxRange nvtx_row(tiles ? "gbrs:tile_pass" : "gbrs:row_pass");
  if (tiles) {
    if (int rct = launch_tiles<false>(d, s)) return rct;
  } else if (d->n_classes > 0) {
    if (int rcr = launch_row_pass(d, model, s)) return rcr;
  }
  }
  if (ev) GBRS_CUDA(cudaEventRecord(ev[1], s));
  {
  NvtxRange nvtx_col("gbrs:column_pass");
  if (!tiles) switch (model) {
    case 4: rc = launch_column<1>(d, d->ent_cls, honour_done, s); break;
    case 3: rc = launch_column<1>(d, d->ent_run, honour_done, s); break;
    case 2: rc = launch_column<1>(d, d->ent_pair, honour_done, s); break;
    default: rc = launch_column<8>(d, d->ent_run, honour_done, s); break;
  }
  }
  if (rc) return rc;
  if (ev) GBRS_CUDA(cudaEventRecord(ev[2], s));
  NvtxRange nvtx_locus(d->n_ranks > 1 && d->xchg_enabled >= 2 ? "gbrs:locus_exchange_update" : "gbrs:locus_numerator");
  const gbrs_em_dev lv = locus_view(d, tiles);
  if (d->n_ranks > 1 && d->xchg_enabled >= 2 && !estep_only) {
    if (int rcp = launch_push<false>(&lv, s)) return rcp;
  } else {
    if (d->n_ranks <= 1 && !estep_only) k_locus_acc<false, true><<<acc_grid(d), kThreads, 0, s>>>(lv, true);
    else k_locus_acc<false, false><<<acc_grid(d), kThreads, 0, s>>>(lv, false);
    GBRS_LAUNCH_CHECK("k_locus_acc");
  }
  if (ev) {
    GBRS_CUDA(cudaEventRecord(ev[3], s));
    ++prof->used;
  }
  return GBRS_OK;
}

extern "C" int gbrs_em_launch_update(const gbrs_em_dev* d, void* stream) {
  if (int rc = check_dev(d, "gbrs_em_launch_update")) return rc;
  NvtxRange nvtx_upd("gbrs:update_and_stop_test");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int nparts = acc_grid(d);  // single rank: k_locus_acc already produced theta', iso' and the partial sums
  if (d->n_ranks > 1 && d->xchg_enabled >= 2) {
    nparts = push_grid<false>(d);  // k_locus_xchg (queued by gbrs_em_launch_local) has updated theta already
  } else if (d->n_ranks > 1) {
    nparts = locus_grid(d);
    static const bool two_launches = std::getenv("GBRS_XCHG_SPLIT") != nullptr;  // A/B knob: reduce as its own kernel
    if (d->xchg_enabled && !two_launches) {
      if (int rc = check_exchange(d)) return rc;
      // all blocks resident at once (see k_locus_update<true, true>)
      const int cap = resident_grid(k_locus_update<true, true>, (int64_t) d->T * GBRS_HPAD);
      if (nparts > cap) nparts = cap;
      k_locus_update<true, true><<<nparts, kThreads, 0, s>>>(*d);
    } else {
      if (int rc = launch_exchange(d, s)) return rc;
      k_locus_update<true><<<nparts, kThreads, 0, s>>>(*d);
    }
    GBRS_LAUNCH_CHECK("k_locus_update");
  }
  k_converge<false><<<converge_grid(d), kThreads, 0, s>>>(*d, nparts);
  GBRS_LAUNCH_CHECK("k_converge");
  return GBRS_OK;
}

namespace {
struct GraphEntry { uint64_t key; cudaGraphExec_t exec; uint64_t stamp; };
std::vector<GraphEntry> g_graph_cache;
std::mutex g_graph_mutex;
uint64_t g_graph_stamp = 0;

uint64_t graph_key(const gbrs_em_dev* d, int model, int poll_every) {  // FNV-1a over the descriptor bytes
  uint64_t h = 1469598103934665603ull;
  const unsigned char* p = reinterpret_cast<const unsigned char*>(d);
  for (size_t i = 0; i < sizeof(gbrs_em_dev); ++i) h = (h ^ p[i]) * 1099511628211ull;
  int dev = 0;
  cudaGetDevice(&dev);
  const uint64_t extra[3] = {(uint64_t) model, (uint64_t) poll_every, (uint64_t) dev};
  p = reinterpret_cast<const unsigned char*>(extra);
  for (size_t i = 0; i < sizeof(extra); ++i) h = (h ^ p[i]) * 1099511628211ull;
  return h;
}
}  // namespace

extern "C" int gbrs_em_run(const gbrs_em_dev* d, int model, double tol, int max_iters, int poll_every, void* stream,
                           int32_t* iters_out, double* errs_host) {
  return gbrs_em_run_cb(d, model, tol, max_iters, poll_every, stream, iters_out, errs_host, nullptr, nullptr);
}

extern "C" int gbrs_em_run_cb(const gbrs_em_dev* d, int model, double tol, int max_iters, int poll_every, void* stream,
                              int32_t* iters_out, double* errs_host, gbrs_poll_cb on_poll, void* user) {
  if (int rc = check_dev(d, "gbrs_em_run")) return rc;
  if (d->n_ranks > 1) {
    gbrs_set_error("gbrs_em_run: row-sharded runs interleave the exchange step; drive launch_local / launch_update");
    return GBRS_E_ARG;
  }
  if (poll_every < 1) poll_every = 4;
  // The loop body (poll_every updates = 4 * poll_every kernels) is captured once into a CUDA graph and replayed until
  // the device-side stop flag is seen; the kernels read the ping-pong parity / stop flag from device memory, so one
  // graph serves every update.  Capture needs a non-legacy stream: work submitted to the legacy default stream is
  // moved onto a private stream (after draining the caller's).
  static const bool use_graph = std::getenv("GBRS_NO_GRAPH") == nullptr;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaStream_t own = nullptr;
  if (use_graph && (s == nullptr || s == cudaStreamLegacy)) {
    GBRS_CUDA(cudaStreamSynchronize(s));
    GBRS_CUDA(cudaStreamCreateWithFlags(&own, cudaStreamNonBlocking));
    s = own;
  }
  int rc = gbrs_em_run_begin(d, tol, max_iters, s);
  int32_t ctrl[16];
  std::memset(ctrl, 0, sizeof(ctrl));
  if (!rc) rc = gbrs_em_read_ctrl(d, s, ctrl, nullptr);
  // The instantiated graph is kept across calls (capture + instantiation cost about as much as ten updates): it bakes
  // the descriptor in by value, so it is keyed by the descriptor's bytes, the model and the poll interval.
  cudaGraphExec_t exec = nullptr;
  if (!rc && !ctrl[GBRS_CTRL_DONE] && use_graph) {
    const uint64_t key = graph_key(d, model, poll_every);
    std::lock_guard<std::mutex> lock(g_graph_mutex);
    for (auto& e : g_graph_cache)
      if (e.key == key) { exec = e.exec; e.stamp = ++g_graph_stamp; break; }
    if (!exec) {
      cudaGraph_t graph = nullptr;
      if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
        for (int i = 0; i < poll_every && !rc; ++i) {
          rc = gbrs_em_launch_local(d, model, s);
          if (!rc) rc = gbrs_em_launch_update(d, s);
        }
        const cudaError_t ce = cudaStreamEndCapture(s, &graph);
        if (rc || ce != cudaSuccess || cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) {
          exec = nullptr;
          cudaGetLastError();
          if (!rc) rc = GBRS_OK;  // fall back to plain launches below
        }
        if (graph) cudaGraphDestroy(graph);
      } else {
        cudaGetLastError();
      }
      if (exec) {
        if (g_graph_cache.size() >= 8) {  // drop the least recently used
          size_t lru = 0;
          for (size_t i = 1; i < g_graph_cache.size(); ++i)
            if (g_graph_cache[i].stamp < g_graph_cache[lru].stamp) lru = i;
          cudaGraphExecDestroy(g_graph_cache[lru].exec);
          g_graph_cache.erase(g_graph_cache.begin() + lru);
        }
        g_graph_cache.push_back({key, exec, ++g_graph_stamp});
      }
    }
  }
  int reported = 0;
  std::vector<double> poll_buf;
  while (!rc && !ctrl[GBRS_CTRL_DONE]) {
    if (exec) {
      if (cudaGraphLaunch(exec, s) != cudaSuccess) { gbrs_set_error("cudaGraphLaunch failed"); rc = GBRS_E_CUDA; break; }
    } else {
      for (int i = 0; i < poll_every && !rc; ++i) {
        rc = gbrs_em_launch_local(d, model, s);
        if (!rc) rc = gbrs_em_launch_update(d, s);
      }
    }
    if (!rc) rc = gbrs_em_read_ctrl(d, s, ctrl, nullptr);
    if (!rc && on_poll && ctrl[GBRS_CTRL_ITERS] > reported) {
      // progress rows as they happen (the reference prints one line per iteration, EMfactory.py:280-287)
      const int n_new = ctrl[GBRS_CTRL_ITERS] - reported;
      poll_buf.resize((size_t) n_new);
      if (cudaMemcpyAsync(poll_buf.data(), d->err_log + reported, sizeof(double) * (size_t) n_new, cudaMemcpyDeviceToHost, s) !=
              cudaSuccess ||
          cudaStreamSynchronize(s) != cudaSuccess) {
        gbrs_set_error("copying the error log failed");
        rc = GBRS_E_CUDA;
        break;
      }
      on_poll(reported, n_new, poll_buf.data(), user);
      reported = ctrl[GBRS_CTRL_ITERS];
    }
  }
  if (!rc && errs_host && ctrl[GBRS_CTRL_ITERS] > 0) {
    if (cudaMemcpyAsync(errs_host, d->err_log, sizeof(double) * (size_t) ctrl[GBRS_CTRL_ITERS], cudaMemcpyDeviceToHost, s) !=
            cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess) {
      gbrs_set_error("copying the error log failed");
      rc = GBRS_E_CUDA;
    }
  }
  if (own) {
    cudaStreamSynchronize(own);
    cudaStreamDestroy(own);
  }
  if (rc) return rc;
  if (iters_out) *iters_out = ctrl[GBRS_CTRL_ITERS];
  if (ctrl[GBRS_CTRL_ERROR]) {
    gbrs_set_error("non-finite value in the EM update (zero normaliser or overflow)");
    return GBRS_E_NUMERIC;
  }
  return GBRS_OK;
}

extern "C" int gbrs_em_alignment_counts(const gbrs_em_dev* d, int gene_level, int32_t n_real_genes, double* aln_dev,
                                        double* uniq_dev, double* locus_uniq_dev, void* stream) {
  if (int rc = check_dev(d, "gbrs_em_alignment_counts")) return rc;
  if (!aln_dev || !uniq_dev || !locus_uniq_dev) { gbrs_set_error("gbrs_em_alignment_counts: null output"); return GBRS_E_ARG; }
  if (gene_level && !d->gene_of) { gbrs_set_error("No group information is available for bundling."); return GBRS_E_ARG; }
  if (!d->rowptr) { gbrs_set_error("gbrs_em_alignment_counts: rowptr missing from descriptor"); return GBRS_E_ARG; }
  if (d->n_classes == 0) return GBRS_OK;
  k_alignment_counts<<<grid_for(d->n_classes), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      *d, gene_level, n_real_genes, aln_dev, uniq_dev, locus_uniq_dev);
  GBRS_LAUNCH_CHECK("k_alignment_counts");
  return GBRS_OK;
}

extern "C" int gbrs_em_posterior_scratch_bytes(const gbrs_em_dev* d, int model, int64_t N, int64_t* bytes) {
  if (!d || !bytes || model < 1 || model > 4 || N < 0) { gbrs_set_error("gbrs_em_posterior_scratch_bytes: bad argument"); return GBRS_E_ARG; }
  *bytes = post_scratch(d, model, N).total;
  return GBRS_OK;
}

extern "C" int gbrs_em_posterior(const gbrs_em_dev* d, int model, const double* theta_src, const uint32_t* class_id, int64_t N,
                                 const int64_t* const* indptr, const void* const* indices, int32_t index_bytes,
                                 double* const* values, void* scratch, int64_t scratch_bytes, void* stream) {
  const char* who = "gbrs_em_posterior";
  if (!d) { gbrs_set_error("gbrs_em_posterior: null descriptor"); return GBRS_E_ARG; }
  if (model < 1 || model > 4) { gbrs_set_error("The read normalization model should be 1, 2, 3, or 4."); return GBRS_E_ARG; }
  if (d->T <= 0 || d->H < 1 || d->H > GBRS_HPAD || N < 0 || N >= (int64_t(1) << 32) || (index_bytes != 4 && index_bytes != 8) ||
      !theta_src || !indptr || !indices || !values || !scratch) {
    gbrs_set_error("gbrs_em_posterior: bad argument"); return GBRS_E_ARG;
  }
  for (int h = 0; h < d->H; ++h)
    if (!indptr[h] || !indices[h] || !values[h]) { gbrs_set_error("gbrs_em_posterior: null output pattern array"); return GBRS_E_ARG; }
  if (d->n_classes > 0 && (!d->pairs || !class_id)) { gbrs_set_error("gbrs_em_posterior: pairs / class_id missing"); return GBRS_E_ARG; }
  if (model != 4 && (!d->gene_of || !d->gene_ptr || !d->gene_loci || !d->rowptr || !d->runptr)) {
    gbrs_set_error("gbrs_em_posterior: models 1-3 need rowptr / runptr and the gene tables"); return GBRS_E_ARG;
  }
  const PostScratch L = post_scratch(d, model, N);
  if (scratch_bytes < L.total) { gbrs_set_error("gbrs_em_posterior: scratch too small"); return GBRS_E_ARG; }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { gbrs_set_error(std::string(who) + ": no CUDA device (there is no CPU fallback)"); return GBRS_E_CUDA; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  char* base = static_cast<char*>(scratch);
  uint32_t* class_pos = reinterpret_cast<uint32_t*>(base + L.class_pos);
  // the row pass' view: theta_src at parity 0 of a zeroed control block, unit counts, own tables -- one rank, no tiles
  gbrs_em_dev v = *d;
  v.theta = const_cast<double*>(theta_src);
  v.ctrl = reinterpret_cast<int32_t*>(base + L.ctrl);
  v.part = reinterpret_cast<double*>(base + L.part);
  v.iso = reinterpret_cast<double*>(base + L.iso);
  v.subsets = reinterpret_cast<double*>(base + L.subsets);
  v.gene_hap = reinterpret_cast<double*>(base + L.gene_hap);
  v.gamma = reinterpret_cast<double*>(base + L.gamma);
  double* ones = reinterpret_cast<double*>(base + L.count);
  v.count = ones;
  v.weights = reinterpret_cast<double*>(base + L.weights);
  v.acc = v.wit = v.err_log = v.scal = nullptr;  // the EM's buffers: nothing here writes them
  v.xchg_enabled = 0;
  v.n_ranks = 1;
  v.xchg_mc = nullptr;
  v.tile_blob = nullptr;
  v.tile_desc = v.tile_locus_desc = nullptr;
  v.tile_partial = nullptr;
  GBRS_CUDA(cudaMemsetAsync(v.ctrl, 0, 16 * sizeof(int32_t), s));
  const int64_t n_init = N > d->n_classes ? N : d->n_classes;
  if (n_init > 0) {
    k_post_init<<<grid_for(n_init), kThreads, 0, s>>>(N, class_pos, d->n_classes, ones);
    GBRS_LAUNCH_CHECK("k_post_init");
  }
  if (d->n_classes > 0) {
    k_post_class_pos<<<grid_for(d->n_classes), kThreads, 0, s>>>(d->n_classes, class_id, N, class_pos, v.ctrl);
    GBRS_LAUNCH_CHECK("k_post_class_pos");
  }
  k_subset_tables<<<resident_grid(k_subset_tables, (int64_t) d->T * 32), kThreads, 0, s>>>(v);
  GBRS_LAUNCH_CHECK("k_subset_tables");
  if (model == 2) {  // isoform totals of theta_src (into iso[0]), summed as the EM sums them
    k_locus_update<false><<<locus_grid(&v), kThreads, 0, s>>>(v);
    GBRS_LAUNCH_CHECK("k_locus_update<refresh>");
  }
  if (model != 4) {
    k_gene_totals<<<grid_for((int64_t) d->n_gene_ids * 8), kThreads, 0, s>>>(v);
    GBRS_LAUNCH_CHECK("k_gene_totals");
  }
  if (d->n_classes > 0) {
    if (int rc = launch_row_pass(&v, model, s)) return rc;
    if (model != 4) {
      k_post_dead_classes<<<grid_for(d->n_classes), kThreads, 0, s>>>(v);
      GBRS_LAUNCH_CHECK("k_post_dead_classes");
    }
  }
  for (int h = 0; h < d->H; ++h) {
    const int rc = index_bytes == 4 ? launch_post_gather<uint32_t>(&v, model, h, N, class_pos, indptr[h], indices[h], values[h], s)
                                    : launch_post_gather<unsigned long long>(&v, model, h, N, class_pos, indptr[h], indices[h], values[h], s);
    if (rc) return rc;
  }
  int32_t ctrl[16];
  GBRS_CUDA(cudaMemcpyAsync(ctrl, v.ctrl, sizeof(ctrl), cudaMemcpyDeviceToHost, s));
  GBRS_CUDA(cudaStreamSynchronize(s));
  if (ctrl[GBRS_CTRL_ERROR] == 2) {
    gbrs_set_error("gbrs_em_posterior: the output pattern holds an entry the packed incidence does not");
    return GBRS_E_ARG;
  }
  if (ctrl[GBRS_CTRL_ERROR]) {
    gbrs_set_error("non-finite posterior probability (a class with a zero normaliser)");
    return GBRS_E_NUMERIC;
  }
  return GBRS_OK;
}

extern "C" int gbrs_em_copy_theta(const gbrs_em_dev* d, int previous, double* dst, void* stream) {
  if (int rc = check_dev(d, "gbrs_em_copy_theta")) return rc;
  if (!dst || (previous != 0 && previous != 1)) { gbrs_set_error("gbrs_em_copy_theta: bad argument"); return GBRS_E_ARG; }
  k_copy_theta<<<grid_for((int64_t) d->T * GBRS_HPAD), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(*d, previous, dst);
  GBRS_LAUNCH_CHECK("k_copy_theta");
  return GBRS_OK;
}

extern "C" int gbrs_boot_scratch_bytes(int64_t N, int64_t* bytes) {
  if (!bytes || N < 1) { gbrs_set_error("gbrs_boot_scratch_bytes: bad argument"); return GBRS_E_ARG; }
  *bytes = boot_scratch(N).total;
  return GBRS_OK;
}

extern "C" int gbrs_boot_guide(const int64_t* prefix, int64_t N, int64_t M, void* scratch, int64_t scratch_bytes, void* stream) {
  if (int rc = check_boot(prefix, N, M, scratch, scratch_bytes, "gbrs_boot_guide")) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int bits = boot_bits(N);
  uint32_t* guide = reinterpret_cast<uint32_t*>(static_cast<char*>(scratch) + boot_scratch(N).guide);
  k_boot_guide<<<grid_for((int64_t(1) << bits) + 1), kThreads, 0, s>>>(prefix, N, (uint64_t) M, bits, guide);
  GBRS_LAUNCH_CHECK("k_boot_guide");
  return GBRS_OK;
}

extern "C" int gbrs_boot_resample(const int64_t* prefix, int64_t N, int64_t M, uint64_t seed, uint32_t replicate,
                                  const uint32_t* class_id, int64_t n_classes, void* scratch, int64_t scratch_bytes,
                                  double* count_out, void* stream) {
  if (int rc = check_boot(prefix, N, M, scratch, scratch_bytes, "gbrs_boot_resample")) return rc;
  if (n_classes < 0 || n_classes > N || (n_classes > 0 && (!class_id || !count_out))) {
    gbrs_set_error("gbrs_boot_resample: bad packed class arguments"); return GBRS_E_ARG;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const BootScratch L = boot_scratch(N);
  char* base = static_cast<char*>(scratch);
  unsigned long long* hist = reinterpret_cast<unsigned long long*>(base + L.hist);
  const uint32_t* guide = reinterpret_cast<const uint32_t*>(base + L.guide);
  GBRS_CUDA(cudaMemsetAsync(hist, 0, sizeof(unsigned long long) * (size_t) N, s));
  const int64_t n_pairs = (M + 1) >> 1;
  k_boot_sample<<<resident_grid(k_boot_sample, n_pairs), kThreads, 0, s>>>(prefix, (uint64_t) M, boot_bits(N), guide, seed,
                                                                            replicate, hist);
  GBRS_LAUNCH_CHECK("k_boot_sample");
  if (n_classes > 0) {
    k_boot_scatter<<<grid_for(n_classes), kThreads, 0, s>>>(hist, class_id, n_classes, count_out);
    GBRS_LAUNCH_CHECK("k_boot_scatter");
  }
  return GBRS_OK;
}

extern "C" int gbrs_boot_derive(const double* src, int64_t B, int32_t T, int32_t H, int32_t quantity, const uint32_t* gene_ptr,
                                const uint32_t* gene_loci, int32_t n_genes, double* values, void* stream) {
  if (!src || !values || B < 1 || T < 1 || H < 1 || H > GBRS_HPAD || quantity < GBRS_BOOT_TPM ||
      quantity > GBRS_BOOT_SHARE || (gene_ptr != nullptr) != (gene_loci != nullptr) || (gene_ptr && n_genes < 1)) {
    gbrs_set_error("gbrs_boot_derive: bad argument");
    return GBRS_E_ARG;
  }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { gbrs_set_error("gbrs_boot_derive: no CUDA device (there is no CPU fallback)"); return GBRS_E_CUDA; }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int32_t L = gene_ptr ? n_genes : T;
  const int what = quantity == GBRS_BOOT_TPM ? 0 : quantity == GBRS_BOOT_COUNTS ? 1 : 2;
  k_bsum_level<<<grid_for(B * L), kThreads, 0, s>>>(src, B, T, H, L, gene_ptr, gene_loci, what, values);
  GBRS_LAUNCH_CHECK("k_bsum_level");
  if (quantity == GBRS_BOOT_TPM) {
    k_bsum_tpm<<<(int) (B < 65535 ? B : 65535), kBootSumThreads, 0, s>>>(B, H, L, values);
    GBRS_LAUNCH_CHECK("k_bsum_tpm");
  }
  return GBRS_OK;
}

extern "C" int gbrs_boot_summarize(const double* values, int64_t B, int64_t E, const double* q, int32_t nq, double* mean,
                                   double* sd, double* qout, int32_t* n, void* stream) {
  if (!values || B < 1 || E < 0 || nq < 0 || nq > GBRS_BOOT_MAX_QUANTILES || (nq > 0 && (!q || !qout)) || !mean || !sd) {
    gbrs_set_error("gbrs_boot_summarize: bad argument");
    return GBRS_E_ARG;
  }
  if (B > GBRS_BOOT_SUMMARY_MAX_B) {
    gbrs_set_error("gbrs_boot_summarize: at most " + std::to_string(GBRS_BOOT_SUMMARY_MAX_B) + " replicates");
    return GBRS_E_LIMIT;
  }
  BootQuantiles Q{};
  for (int j = 0; j < nq; ++j) {
    if (!(q[j] >= 0.0 && q[j] <= 1.0)) { gbrs_set_error("gbrs_boot_summarize: quantiles must be in [0, 1]"); return GBRS_E_ARG; }
    Q.q[j] = q[j];
  }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { gbrs_set_error("gbrs_boot_summarize: no CUDA device (there is no CPU fallback)"); return GBRS_E_CUDA; }
  if (E == 0) return GBRS_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int P = boot_pow2(B);
  const int64_t col_bytes = (int64_t) (P + 1) * (int64_t) sizeof(double);
  int64_t K = kBootSummarySmem / col_bytes;
  if (K > kBootSummaryMaxTile) K = kBootSummaryMaxTile;
  if (K > E) K = E;
  const int smem_bytes = (int) (K * col_bytes);
  GBRS_CUDA(cudaFuncSetAttribute(k_boot_summarize, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  const int64_t n_tiles = (E + K - 1) / K;
  const int grid = (int) (n_tiles < (int64_t) sm_count() * 8 ? n_tiles : (int64_t) sm_count() * 8);
  k_boot_summarize<<<grid, kThreads, smem_bytes, s>>>(values, B, E, P, (int) K, Q, nq, mean, sd, qout, n);
  GBRS_LAUNCH_CHECK("k_boot_summarize");
  return GBRS_OK;
}
