// Internals shared by the host-side packers (pack.cpp: class-major + locus-major arrays; tile_pack.cpp: the per-tile
// blobs of the fused model-4 kernel).  Not part of the C ABI.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <memory>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "gbrs_em.h"

#ifdef _OPENMP
#include <omp.h>
#endif

void gbrs_set_error(const std::string& s);  // em_kernels.cu

// Large work arrays: allocation without the value-initialising pass of std::vector (a single thread touching hundreds
// of megabytes page by page cost more than any packing stage); whatever needs a defined start value is filled by all
// threads (par_fill), which also spreads the first touch of the pages.
template <typename T>
struct noinit_alloc : std::allocator<T> {
  template <typename U> struct rebind { using other = noinit_alloc<U>; };
  noinit_alloc() = default;
  template <typename U> noinit_alloc(const noinit_alloc<U>&) {}
  template <typename U, typename... A> void construct(U* p, A&&... a) {
    if constexpr (sizeof...(A) == 0) ::new (static_cast<void*>(p)) U;  // default-init: no write
    else ::new (static_cast<void*>(p)) U(std::forward<A>(a)...);
  }
};
template <typename T> using bigvec = std::vector<T, noinit_alloc<T>>;

template <typename V, typename T>
void par_fill(V& v, size_t n, T value) {
  v.resize(n);
  auto* p = v.data();
#pragma omp parallel for schedule(static)
  for (int64_t i = 0; i < (int64_t) n; ++i) p[i] = value;
}

struct gbrs_pack {
  gbrs_pack_info info{};
  int32_t T = 0, H = 0;
  bigvec<uint32_t> rowptr, pairs, runptr;
  bigvec<uint32_t> class_id;  // [n_classes] input class id of every packed class
  std::vector<uint32_t> item_off, item_order, item_desc, locus_item_ptr, locus_order, locus_desc, gene_ptr, gene_loci;
  std::vector<int32_t> gene_of;
  bigvec<double> count;
  bigvec<uint8_t> ent_cls, ent_pair, ent_run;  // entry words, 4 or 8 bytes each
};


// Host threads for the packer.  The caller's OpenMP setting is NOT inherited: torchrun exports OMP_NUM_THREADS=1 to every
// rank, which made each rank pack on one core (1.7 s instead of 0.2 s at 5 M classes).  GBRS_PACK_THREADS overrides;
// otherwise the machine's hardware threads are divided among the ranks of this node (LOCAL_WORLD_SIZE).
inline int pack_threads() {
  if (const char* e = std::getenv("GBRS_PACK_THREADS")) {
    const int n = std::atoi(e);
    if (n > 0) return n;
  }
  int hw = (int) std::thread::hardware_concurrency();
#ifdef _OPENMP
  if (hw <= 0) hw = omp_get_num_procs();
#endif
  if (hw <= 0) hw = 1;
  int ranks = 1;
  if (const char* e = std::getenv("LOCAL_WORLD_SIZE")) ranks = std::max(1, std::atoi(e));
  return std::max(1, hw / ranks);
}

struct OmpThreadsGuard {  // sets the team size for the parallel regions of one call, restores the caller's setting
  int saved = 1;
  explicit OmpThreadsGuard(int n) {
#ifdef _OPENMP
    saved = omp_get_max_threads();
    omp_set_num_threads(n);
#endif
  }
  ~OmpThreadsGuard() {
#ifdef _OPENMP
    omp_set_num_threads(saved);
#endif
  }
};

