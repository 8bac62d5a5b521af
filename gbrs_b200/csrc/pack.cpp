// Host-side packer: H x CSC(N x T) incidence  ->  class-major + locus-major packed rows (see include/gbrs_em.h).
//
// What it replaces in the reference: the reference keeps the incidence as a python list of H scipy CSC matrices
// (src/gbrs/emase/Sparse3DMatrix.py:26-66) and walks all H of them several times per EM iteration
// (reset :220-228, multiply :314-377, APM.sum / normalize_reads src/gbrs/emase/AlignmentPropertyMatrix.py:275-370).
// Here the same information is re-laid once, on the host, into the two orders the GPU passes stream through:
//
//   class-major  rowptr / pairs[]   one 32-bit word per (class, locus): locus | hapmask << 24, classes re-ordered by
//                                   their smallest locus so that neighbouring classes touch neighbouring theta lines
//   locus-major  ent_*[] / item_off one word per (locus, class): index | hapmask << top byte, cut into work items
//
// The `-G` genotype restriction (src/gbrs/gbrs/emase_utils.py:247-273: multiply by gtmask + eliminate_zeros) is an AND of
// every pair's mask with a per-locus byte; pairs and classes that become empty are dropped.
#include <algorithm>
#include <climits>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <memory>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "gbrs_em.h"

#ifdef _OPENMP
#include <omp.h>
#endif

void gbrs_set_error(const std::string& s);  // capi.cu

#include "pack_internal.h"

namespace {

inline int64_t index_at(const void* base, int bytes, int64_t i) {
  return bytes == 4 ? (int64_t) static_cast<const int32_t*>(base)[i] : static_cast<const int64_t*>(base)[i];
}

inline void put_entry(bigvec<uint8_t>& v, int bytes, int64_t pos, uint64_t idx, uint32_t mask) {
  if (bytes == 4) {
    reinterpret_cast<uint32_t*>(v.data())[pos] = (uint32_t) idx | (mask << 24);
  } else {
    reinterpret_cast<uint64_t*>(v.data())[pos] = idx | ((uint64_t) mask << 56);
  }
}

}  // namespace

extern "C" int gbrs_pack_create(const gbrs_pack_input* in, gbrs_pack_t* out) {
  if (!in || !out) { gbrs_set_error("gbrs_pack_create: null argument"); return GBRS_E_ARG; }
  const int T = in->T, H = in->H;
  const int64_t N = in->N;
  if (T <= 0 || N < 0 || H <= 0 || !in->indptr || !in->indices || (in->index_bytes != 4 && in->index_bytes != 8) ||
      in->shard_count < 1 || in->shard_rank < 0 || in->shard_rank >= in->shard_count) {
    gbrs_set_error("gbrs_pack_create: bad shape / shard / index width");
    return GBRS_E_ARG;
  }
  if (H > GBRS_HPAD) { gbrs_set_error("gbrs_pack_create: more than 8 haplotypes is not supported by the mask layout"); return GBRS_E_LIMIT; }
  if (T >= (1 << 24)) { gbrs_set_error("gbrs_pack_create: T must be < 2^24"); return GBRS_E_LIMIT; }
  if (N >= (int64_t(1) << 32)) { gbrs_set_error("gbrs_pack_create: N must be < 2^32"); return GBRS_E_LIMIT; }
  for (int h = 0; h < H; ++h) {
    if (!in->indptr[h] || (!in->indices[h] && in->indptr[h][T] > 0) || in->indptr[h][0] != 0) {
      gbrs_set_error("gbrs_pack_create: bad CSC arrays"); return GBRS_E_ARG;
    }
    for (int t = 0; t < T; ++t)
      if (in->indptr[h][t + 1] < in->indptr[h][t]) { gbrs_set_error("gbrs_pack_create: indptr not monotone"); return GBRS_E_ARG; }
  }
  const int item_len = in->item_len > 0 ? (in->item_len + 7) / 8 * 8 : 64;
  const OmpThreadsGuard omp_guard(pack_threads());

  const bool timing = std::getenv("GBRS_PACK_TIMING") != nullptr;
  double t_last = omp_get_wtime();
  auto lap = [&](const char* what) {
    if (timing) { const double t = omp_get_wtime(); std::fprintf(stderr, "[pack] %-28s %8.1f ms\n", what, (t - t_last) * 1e3); t_last = t; }
  };
  try {
    // ---- 1. merge the H columns of every locus into (class, mask) pairs, locus-major, all classes -----------------
    std::vector<int64_t> ub(T + 1, 0);  // upper bound offsets
    for (int t = 0; t < T; ++t) {
      int64_t s = 0;
      for (int h = 0; h < H; ++h) s += in->indptr[h][t + 1] - in->indptr[h][t];
      ub[t + 1] = ub[t] + s;
    }
    bigvec<uint64_t> tmp((size_t) ub[T]);  // class << 8 | mask; every locus writes (and later reads) only its own prefix
    std::vector<int64_t> lcount(T, 0);
    int bad = 0;
#pragma omp parallel for schedule(dynamic, 64)
    for (int t = 0; t < T; ++t) {
      const uint32_t lm = in->locus_hapmask ? in->locus_hapmask[t] : 0xFFu;
      uint64_t* dst = tmp.data() + ub[t];
      // Fast path: every column is sorted by class id (what scipy / the EMASE writer produce) -> H-way merge, OR-ing
      // the haplotype bits of equal classes.  Any disorder, explicit zero or bad index falls back to gather + sort.
      int64_t m = 0;
      bool merged = !(in->values);
      if (merged) {
        int64_t pos[GBRS_HPAD], end[GBRS_HPAD];
        int nh = 0, hs[GBRS_HPAD];
        for (int h = 0; h < H; ++h)
          if ((lm >> h) & 1u) { pos[nh] = in->indptr[h][t]; end[nh] = in->indptr[h][t + 1]; hs[nh] = h; ++nh; }
        int64_t last = -1;
        while (merged) {
          int64_t best = INT64_MAX;
          for (int i = 0; i < nh; ++i)
            if (pos[i] < end[i]) {
              const int64_t c = index_at(in->indices[hs[i]], in->index_bytes, pos[i]);
              if (c < best) best = c;
            }
          if (best == INT64_MAX) break;
          if (best <= last || best < 0 || best >= N) { merged = false; break; }  // unsorted / duplicate / bad: redo slowly
          uint64_t mask = 0;
          for (int i = 0; i < nh; ++i)
            if (pos[i] < end[i] && index_at(in->indices[hs[i]], in->index_bytes, pos[i]) == best) {
              mask |= (uint64_t) 1 << hs[i];
              ++pos[i];
            }
          dst[m++] = ((uint64_t) best << 8) | mask;
          last = best;
        }
      }
      if (!merged) {
        int64_t n = 0;
        for (int h = 0; h < H; ++h) {
          if (!((lm >> h) & 1u)) continue;
          const int64_t b = in->indptr[h][t], e = in->indptr[h][t + 1];
          for (int64_t i = b; i < e; ++i) {
            if (in->values && in->values[h] && in->values[h][i] == 0.0) continue;
            const int64_t c = index_at(in->indices[h], in->index_bytes, i);
            if (c < 0 || c >= N) { bad = 1; continue; }
            dst[n++] = ((uint64_t) c << 8) | (uint64_t) h;
          }
        }
        std::sort(dst, dst + n);
        m = 0;
        for (int64_t i = 0; i < n;) {
          const uint64_t c = dst[i] >> 8;
          uint64_t mask = 0;
          while (i < n && (dst[i] >> 8) == c) { mask |= (uint64_t) 1 << (dst[i] & 0xFF); ++i; }
          dst[m++] = (c << 8) | mask;
        }
      }
      lcount[t] = m;
    }
    if (bad) { gbrs_set_error("gbrs_pack_create: class index out of range"); return GBRS_E_ARG; }

    lap("1 merge columns");
    // ---- 2. per-class pair / nnz counts, shard boundaries balanced by nnz -----------------------------------------
    // Every thread owns a contiguous range of class ids and walks ALL merged entries (a sequential scan of the
    // locus-major list), keeping only the entries of its own classes: no atomics, and the loci come by in ascending
    // order, so the first locus seen for a class is its smallest one.
    bigvec<uint32_t> npair, minloc, secloc, nz;
    par_fill(npair, (size_t) N, 0u);
    par_fill(minloc, (size_t) N, 0xFFFFFFFFu);
    par_fill(secloc, (size_t) N, 0u);  // second-smallest locus (> 0 when there is one)
    par_fill(nz, (size_t) N, 0u);
    {
      int nt = 1;
#ifdef _OPENMP
      nt = omp_get_max_threads();
#endif
#pragma omp parallel for schedule(static, 1) num_threads(nt)
      for (int k = 0; k < nt; ++k) {
        const uint64_t c_lo = (uint64_t) (N * k / nt), c_hi = (uint64_t) (N * (k + 1) / nt);
        if (c_lo >= c_hi) continue;
        for (int t = 0; t < T; ++t) {
          const uint64_t* src = tmp.data() + ub[t];
          const int64_t m = lcount[t];
          for (int64_t i = 0; i < m; ++i) {
            const uint64_t c = src[i] >> 8;
            if (c < c_lo || c >= c_hi) continue;
            ++npair[c];
            nz[c] += (uint32_t) __builtin_popcountll(src[i] & 0xFF);
            if (minloc[c] == 0xFFFFFFFFu) minloc[c] = (uint32_t) t;
            else if (secloc[c] == 0u) secloc[c] = (uint32_t) t;
          }
        }
      }
    }
    int64_t nnz_total = 0, nclass_total = 0;
#pragma omp parallel for reduction(+ : nnz_total, nclass_total)
    for (int64_t c = 0; c < N; ++c) { nnz_total += nz[c]; nclass_total += npair[c] > 0; }
    // class c goes to shard floor(cum_before(c) * R / total)
    const int R = in->shard_count, rank = in->shard_rank;
    int64_t lo = 0, hi = N;
    if (R > 1) {
      int64_t cum = 0;
      lo = N; hi = N;
      bool lo_set = false;
      for (int64_t c = 0; c < N; ++c) {
        const int r = nnz_total > 0 ? (int) std::min<int64_t>(R - 1, (__int128) cum * R / nnz_total) : 0;
        if (!lo_set && r >= rank) { lo = c; lo_set = true; }
        if (r > rank) { hi = c; break; }
        cum += nz[c];
      }
      if (!lo_set) lo = N;
      if (hi < lo) hi = lo;
    }

    lap("2 class counts + shard");
    // ---- 3. order the shard's non-empty classes by (pairs capped at KMAX+1, smallest locus, second-smallest locus): stable
    // counting sorts ----
    // Equal-width classes are contiguous so the row pass needs no row pointers for them; within a width the classes are
    // ordered by smallest locus so that neighbouring classes touch neighbouring theta lines.
    const int NB = GBRS_KMAX + 1;  // buckets: widths 1..KMAX, then "long"
    auto bucket_of = [&](uint32_t np) { return (int) std::min<uint32_t>(np, GBRS_KMAX + 1) - 1; };
    std::vector<int64_t> bucket((size_t) NB * T + 1, 0);
    int64_t n_classes = 0, n_pairs = 0, nnz = 0;
    int64_t bclass[GBRS_KMAX + 2] = {0}, bpair[GBRS_KMAX + 2] = {0};
    for (int64_t c = lo; c < hi; ++c)
      if (npair[c]) {
        const int b = bucket_of(npair[c]);
        ++bucket[(size_t) b * T + minloc[c] + 1];
        ++bclass[b + 1];
        bpair[b + 1] += npair[c];
        ++n_classes; n_pairs += npair[c]; nnz += nz[c];
      }
    if (n_pairs >= (int64_t(1) << 32)) { gbrs_set_error("gbrs_pack_create: more than 2^32 pairs in one shard"); return GBRS_E_LIMIT; }
    for (size_t i = 0; i < (size_t) NB * T; ++i) bucket[i + 1] += bucket[i];
    for (int b = 0; b < NB; ++b) { bclass[b + 1] += bclass[b]; bpair[b + 1] += bpair[b]; }
    bigvec<uint32_t> new_id;
    par_fill(new_id, (size_t) N, 0xFFFFFFFFu);
    {
      // minor key: the second-smallest locus (stable counting sort first, then the (width, smallest locus) one walks the
      // classes in that order).  Classes sharing their two smallest loci end up next to each other: a warp of the row pass
      // reads fewer distinct table rows, and the entries of a locus gather runs of consecutive weights in the column pass.
      std::vector<int64_t> sec_start((size_t) T + 2, 0);
      for (int64_t c = lo; c < hi; ++c)
        if (npair[c]) ++sec_start[(size_t) secloc[c] + 1];
      for (int t = 0; t <= T; ++t) sec_start[(size_t) t + 1] += sec_start[(size_t) t];
      bigvec<uint32_t> by_sec((size_t) n_classes);
      for (int64_t c = lo; c < hi; ++c)
        if (npair[c]) by_sec[(size_t) sec_start[secloc[c]]++] = (uint32_t) c;
      for (int64_t i = 0; i < n_classes; ++i) {
        const uint32_t c = by_sec[(size_t) i];
        new_id[c] = (uint32_t) bucket[(size_t) bucket_of(npair[c]) * T + minloc[c]]++;
      }
    }

    lap("3 class order");
    auto* P = new gbrs_pack();
    P->T = T;
    P->H = H;
    par_fill(P->rowptr, (size_t) n_classes + 1, 0u);
    par_fill(P->count, (size_t) n_classes, 1.0);
    P->class_id.resize((size_t) n_classes);  // every slot is written below (new_id is a bijection onto [0, n_classes))
#pragma omp parallel for schedule(static)
    for (int64_t c = lo; c < hi; ++c)
      if (npair[c]) {
        P->rowptr[new_id[c] + 1] = npair[c];
        P->class_id[new_id[c]] = (uint32_t) c;
        if (in->count) P->count[new_id[c]] = in->count[c];
      }
    for (int64_t n = 0; n < n_classes; ++n) P->rowptr[n + 1] += P->rowptr[n];

    lap("3b rowptr/count");
    // ---- 4. class-major fill (loci ascending within a class), then order pairs by (gene, locus) and cut runs -----
    P->pairs.resize((size_t) n_pairs);  // every slot is claimed exactly once below
    {
      // all threads scatter; the slot inside a class is claimed atomically, the (gene, locus) sort below makes the
      // final order independent of the claiming order
      bigvec<uint32_t> cur(P->rowptr.begin(), P->rowptr.end() - 1);
#pragma omp parallel for schedule(dynamic, 256)
      for (int t = 0; t < T; ++t) {
        const uint64_t* src = tmp.data() + ub[t];
        for (int64_t i = 0; i < lcount[t]; ++i) {
          const uint32_t nid = new_id[src[i] >> 8];
          if (nid == 0xFFFFFFFFu) continue;
          const uint32_t slot = __atomic_fetch_add(&cur[nid], 1u, __ATOMIC_RELAXED);
          P->pairs[slot] = (uint32_t) t | ((uint32_t)(src[i] & 0xFF) << 24);
        }
      }
    }
    P->gene_of.resize(T);
    for (int t = 0; t < T; ++t) {
      P->gene_of[t] = in->gene_of ? in->gene_of[t] : t;
      if (P->gene_of[t] < 0) { delete P; gbrs_set_error("gbrs_pack_create: negative gene id"); return GBRS_E_ARG; }
    }
    const int32_t n_gene_ids = 1 + *std::max_element(P->gene_of.begin(), P->gene_of.end());
    P->runptr.resize((size_t) n_classes + 1);  // [0] set here, [n + 1] by the loop below
    P->runptr[0] = 0;
    bigvec<uint32_t> run_in_class((size_t) n_pairs);  // run number of a pair inside its class (written for every pair)
    int max_k = 0;
#pragma omp parallel for schedule(static) reduction(max : max_k)
    for (int64_t n = 0; n < n_classes; ++n) {
      uint32_t* b = P->pairs.data() + P->rowptr[n];
      const int k = (int) (P->rowptr[n + 1] - P->rowptr[n]);
      max_k = std::max(max_k, k);
      const int32_t* go = P->gene_of.data();
      // insertion sort by (gene, locus); k is small
      for (int i = 1; i < k; ++i) {
        const uint32_t w = b[i];
        const int64_t key = ((int64_t) go[w & 0xFFFFFF] << 24) | (w & 0xFFFFFF);
        int j = i - 1;
        while (j >= 0 && (((int64_t) go[b[j] & 0xFFFFFF] << 24) | (b[j] & 0xFFFFFF)) > key) { b[j + 1] = b[j]; --j; }
        b[j + 1] = w;
      }
      uint32_t runs = k > 0 ? 1 : 0;
      uint32_t* ric = run_in_class.data() + P->rowptr[n];
      if (k > 0) ric[0] = 0;
      for (int i = 1; i < k; ++i) {
        runs += go[b[i] & 0xFFFFFF] != go[b[i - 1] & 0xFFFFFF];
        ric[i] = runs - 1;
      }
      P->runptr[n + 1] = runs;
    }
    for (int64_t n = 0; n < n_classes; ++n) P->runptr[n + 1] += P->runptr[n];
    const int64_t n_runs = P->runptr[n_classes];

    lap("4 class-major fill + runs");
    // ---- 5. locus-major entries of this shard.  Within a locus: first the entries whose mask is partial, then the
    // entries hitting all H haplotypes ("full"), each part in ascending new class id.  Full entries need no per-haplotype
    // masking in the column pass (one add instead of eight masked ones) and are the commonest kind.
    // Every part is padded to a multiple of 4 entries with dummy words (empty mask, index = one past the last real
    // index, whose weight slot is kept at zero), so that items start 16-byte aligned and the column pass can fetch four
    // entries per load.
    // 32-bit entry words hold a 24-bit index; larger shards (> 16.7 M classes / pairs / runs) switch to 64-bit words.
    // GBRS_FORCE_ENTRY64 forces the wide words on small inputs so that tests can exercise that path.
    const bool force64 = std::getenv("GBRS_FORCE_ENTRY64") != nullptr;
    const int entry_bytes = (!force64 && std::max({n_classes, n_pairs, n_runs}) + 1 < (int64_t(1) << 24)) ? 4 : 8;
    const uint32_t full_mask = (1u << H) - 1u;
    auto pad4 = [](int64_t x) { return (x + 3) / 4 * 4; };
    std::vector<int64_t> lcnt(T, 0), lpart(T, 0);
#pragma omp parallel for schedule(dynamic, 256)
    for (int t = 0; t < T; ++t) {  // entries of this shard per locus, and how many of them have a partial mask
      const uint64_t* src = tmp.data() + ub[t];
      int64_t c_all = 0, c_part = 0;
      for (int64_t i = 0; i < lcount[t]; ++i)
        if (new_id[src[i] >> 8] != 0xFFFFFFFFu) { ++c_all; c_part += (src[i] & 0xFF) != full_mask; }
      lcnt[t] = c_all;
      lpart[t] = c_part;
    }
    // only deep loci are split into a partial and a full part; a shallow locus stays one (mixed) part, otherwise the
    // many tiny loci would double their item count for nothing
    std::vector<uint8_t> split(T, 0);
    std::vector<int64_t> lptr(T + 1, 0), ppart(T, 0), pfull(T, 0);  // padded start of the locus, padded part lengths
    for (int t = 0; t < T; ++t) {
      split[t] = lcnt[t] > 8 * (int64_t) item_len;
      if (!split[t]) lpart[t] = lcnt[t];
      ppart[t] = pad4(lpart[t]);
      pfull[t] = pad4(lcnt[t] - lpart[t]);
      lptr[t + 1] = lptr[t] + ppart[t] + pfull[t];
    }
    const int64_t n_entries = lptr[T];
    if (n_entries >= (int64_t(1) << 32)) { delete P; gbrs_set_error("gbrs_pack_create: more than 2^32 entries in one shard"); return GBRS_E_LIMIT; }
    P->ent_cls.resize((size_t) n_entries * entry_bytes);
    P->ent_pair.resize((size_t) n_entries * entry_bytes);
    P->ent_run.resize((size_t) n_entries * entry_bytes);
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n_entries; ++i) {
      put_entry(P->ent_cls, entry_bytes, i, (uint64_t) n_classes, 0);
      put_entry(P->ent_pair, entry_bytes, i, (uint64_t) n_pairs, 0);
      put_entry(P->ent_run, entry_bytes, i, (uint64_t) n_runs, 0);
    }
    {
      // Every locus is filled by one thread from its merged column (step 1): the surviving (class, mask) entries are
      // ordered by NEW class id (within a split locus: partial masks first), and the pair word of each entry is looked
      // up in its class row (a handful of words), which gives its pair index and run.  The writes of a locus are
      // sequential; loci are handed out dynamically, the few very deep ones first would not matter at this grain.
#pragma omp parallel
      {
        std::vector<uint64_t> keys;
#pragma omp for schedule(dynamic, 64)
        for (int t = 0; t < T; ++t) {
          if (lcnt[t] == 0) continue;
          const uint64_t* src = tmp.data() + ub[t];
          keys.clear();
          for (int64_t i = 0; i < lcount[t]; ++i) {
            const uint32_t nid = new_id[src[i] >> 8];
            if (nid == 0xFFFFFFFFu) continue;
            const uint64_t m = src[i] & 0xFF;
            const uint64_t part = (split[t] && m == full_mask) ? 1 : 0;  // full-mask entries of a deep locus go last
            keys.push_back((part << 40) | ((uint64_t) nid << 8) | m);
          }
          std::sort(keys.begin(), keys.end());
          int64_t pos_part = lptr[t], pos_full = lptr[t] + ppart[t];
          for (const uint64_t k : keys) {
            const uint32_t n = (uint32_t) ((k >> 8) & 0xFFFFFFFFu), m = (uint32_t) (k & 0xFF);
            uint32_t p = P->rowptr[n];
            while ((P->pairs[p] & 0xFFFFFF) != (uint32_t) t) ++p;  // the class does hit this locus
            const int64_t pos = (k >> 40) ? pos_full++ : pos_part++;
            put_entry(P->ent_cls, entry_bytes, pos, (uint64_t) n, m);
            put_entry(P->ent_pair, entry_bytes, pos, (uint64_t) p, m);
            put_entry(P->ent_run, entry_bytes, pos, (uint64_t) P->runptr[n] + run_in_class[p], m);
          }
        }
      }
    }
    bigvec<uint64_t>().swap(tmp);

    lap("5 locus-major entries");
    // ---- 6. column-pass work items ------------------------------------------------------------------------------
    // Each part (partial / full) of a locus is cut separately.  A part with up to 8 * item_len entries becomes short
    // items (<= item_len entries, one aligned 8-lane group each); a deeper part becomes long items (<= 32 * item_len
    // entries, a whole warp each), so that the per-locus combine in k_locus_acc, which walks a locus' items serially,
    // stays short even for the deepest loci.
    const char* lf_env = std::getenv("GBRS_LONG_FACTOR");  // tuning knob: long item = factor * item_len entries
    const int64_t long_factor = lf_env ? std::max(8, std::atoi(lf_env)) : 32;
    const int64_t long_len = long_factor * (int64_t) item_len;
    auto item_len_of = [&](int64_t len) -> int64_t {
      if (len <= 8 * (int64_t) item_len) return item_len;
      const int64_t n = (len + long_len - 1) / long_len;
      return ((len + n - 1) / n + 31) / 32 * 32;
    };
    auto items_of = [&](int64_t len) -> int64_t { return len ? (len + item_len_of(len) - 1) / item_len_of(len) : 0; };
    P->locus_item_ptr.assign((size_t) T + 1, 0);
    for (int t = 0; t < T; ++t) {
      P->locus_item_ptr[t + 1] = P->locus_item_ptr[t] + (uint32_t) (items_of(ppart[t]) + items_of(pfull[t]));
    }
    const int64_t n_items = P->locus_item_ptr[T];
    if (n_items >= (int64_t(1) << 31)) { delete P; gbrs_set_error("gbrs_pack_create: too many work items"); return GBRS_E_LIMIT; }
    P->item_off.assign((size_t) n_items + 1, 0);
    std::vector<uint8_t> item_full((size_t) n_items, 0);
    for (int t = 0; t < T; ++t) {
      uint32_t it = P->locus_item_ptr[t];
      const int64_t np = ppart[t], nf = pfull[t];
      const int64_t ilp = item_len_of(np), ilf = item_len_of(nf);
      for (int64_t o = 0; o < np; o += ilp) P->item_off[it++] = (uint32_t) (lptr[t] + o);
      for (int64_t o = 0; o < nf; o += ilf) { item_full[it] = 1; P->item_off[it++] = (uint32_t) (lptr[t] + np + o); }
    }
    P->item_off[n_items] = (uint32_t) n_entries;
    P->info.n_entries = n_entries;
    // Visiting order: long items first, then short ones; inside each, partial before full (a warp works on items of
    // one kind), longest first (the deep loci must not form the tail).  Bit 31 of an item_order word marks a full item.
    {
      std::vector<uint32_t> idx((size_t) n_items);
      std::iota(idx.begin(), idx.end(), 0u);
      auto len_of = [&](uint32_t i) { return (int64_t) P->item_off[i + 1] - (int64_t) P->item_off[i]; };
      std::stable_sort(idx.begin(), idx.end(), [&](uint32_t x, uint32_t y) {
        const int64_t lx = len_of(x), ly = len_of(y);
        const int kx = (lx > item_len ? 0 : 2) + item_full[x], ky = (ly > item_len ? 0 : 2) + item_full[y];
        if (kx != ky) return kx < ky;
        return lx > ly;
      });
      P->item_order.assign((size_t) n_items, 0);
      // + a two-descriptor trailer: where the short items change kind / size class in the visiting order (the column pass
      // gives an item of one quad one lane, of two quads two lanes, anything longer eight)
      P->item_desc.assign((size_t) (n_items + 2) * 4, 0);
      int64_t sp_all = 0, sp_gt8 = 0, sp_gt4 = 0, sf_gt8 = 0, sf_gt4 = 0;
      for (int64_t i = 0; i < n_items; ++i) {
        const int64_t len_i = len_of(idx[i]);
        if (len_i <= item_len) {
          const bool f = item_full[idx[i]];
          sp_all += !f;
          (f ? sf_gt8 : sp_gt8) += len_i > 8;
          (f ? sf_gt4 : sp_gt4) += len_i > 4;
        }
      }
      for (int64_t i = 0; i < n_items; ++i) {
        P->item_order[i] = idx[i] | (item_full[idx[i]] ? 0x80000000u : 0u);
        P->info.n_long_items += len_of(idx[i]) > item_len;
        // one 16-byte descriptor per visiting slot: begin, end, item id, flags (bit 0 = full)
        P->item_desc[4 * i + 0] = P->item_off[idx[i]];
        P->item_desc[4 * i + 1] = P->item_off[idx[i] + 1];
        P->item_desc[4 * i + 2] = idx[i];
        P->item_desc[4 * i + 3] = item_full[idx[i]];
      }
      const int64_t nl = P->info.n_long_items, f0 = nl + sp_all;
      uint32_t* tr = P->item_desc.data() + 4 * (size_t) n_items;
      tr[0] = (uint32_t) (nl + sp_gt8);
      tr[1] = (uint32_t) (nl + sp_gt4);
      tr[2] = (uint32_t) f0;
      tr[3] = (uint32_t) (f0 + sf_gt8);
      tr[4] = (uint32_t) (f0 + sf_gt4);
    }
    // (3) loci in descending item count: the per-locus combine starts with the deepest loci.  locus_desc carries, per
    // visiting slot, everything the combine needs in one 16-byte load: locus, first item, one-past-last item.
    {
      P->locus_order.resize((size_t) T);
      std::iota(P->locus_order.begin(), P->locus_order.end(), 0u);
      std::stable_sort(P->locus_order.begin(), P->locus_order.end(), [&](uint32_t x, uint32_t y) {
        return P->locus_item_ptr[x + 1] - P->locus_item_ptr[x] > P->locus_item_ptr[y + 1] - P->locus_item_ptr[y];
      });
      P->locus_desc.assign((size_t) T * 4, 0);
      for (int i = 0; i < T; ++i) {
        const uint32_t t = P->locus_order[i];
        P->locus_desc[4 * (size_t) i + 0] = t;
        P->locus_desc[4 * (size_t) i + 1] = P->locus_item_ptr[t];
        P->locus_desc[4 * (size_t) i + 2] = P->locus_item_ptr[t + 1];
        P->info.n_deep_loci += P->locus_item_ptr[t + 1] - P->locus_item_ptr[t] > GBRS_DEEP_LOCUS_ITEMS;
      }
    }

    // ---- 6b. lane-interleaved entry order inside every work item ----------------------------------------------------
    // The column pass gives every lane four consecutive entry words per 128-bit load (lane j of a LANES-wide group holds
    // words 4j .. 4j+3 of a block of 4 * LANES words) and then gathers the weight of its i-th word in round i.  With the
    // entries in plain ascending class order, the lanes of one gather round would be four entries apart and touch up
    // to LANES different 128-byte lines of the weight vector; the gather rate is bound by lines per load instruction
    // (L1 wavefronts), not by bytes.  So the ascending sequence is dealt round-robin instead: word 4j + i of a block
    // holds its (i * nq + j)-th smallest entry (nq = quads in the block), which makes every gather round read LANES
    // *consecutive* entries -- neighbouring classes, mostly the same one or two lines.
    const int64_t nit = n_items;
#pragma omp parallel
    {
      std::vector<uint64_t> buf(128);
#pragma omp for schedule(dynamic, 256)
      for (int64_t it = 0; it < nit; ++it) {
        const int64_t b = P->item_off[it], e = P->item_off[it + 1];
        const int64_t B = (e - b > item_len) ? 128 : 32;  // long items: a warp; short items: an 8-lane group
        for (int64_t k = b; k < e; k += B) {
          const int64_t m = std::min<int64_t>(B, e - k), nq = m / 4;
          for (bigvec<uint8_t>* arr : {&P->ent_cls, &P->ent_pair, &P->ent_run}) {
            if (entry_bytes == 4) {
              uint32_t* w = reinterpret_cast<uint32_t*>(arr->data()) + k;
              for (int64_t r = 0; r < m; ++r) buf[r] = w[r];
              for (int64_t r = 0; r < m; ++r) w[4 * (r % nq) + r / nq] = (uint32_t) buf[r];
            } else {
              uint64_t* w = reinterpret_cast<uint64_t*>(arr->data()) + k;
              for (int64_t r = 0; r < m; ++r) buf[r] = w[r];
              for (int64_t r = 0; r < m; ++r) w[4 * (r % nq) + r / nq] = buf[r];
            }
          }
        }
      }
    }

    lap("6 items + orders");
    // ---- 7. gene -> loci CSR ------------------------------------------------------------------------------------
    P->gene_ptr.assign((size_t) n_gene_ids + 1, 0);
    for (int t = 0; t < T; ++t) ++P->gene_ptr[P->gene_of[t] + 1];
    for (int g = 0; g < n_gene_ids; ++g) P->gene_ptr[g + 1] += P->gene_ptr[g];
    P->gene_loci.assign((size_t) T, 0);
    {
      std::vector<uint32_t> cur(P->gene_ptr.begin(), P->gene_ptr.end() - 1);
      for (int t = 0; t < T; ++t) P->gene_loci[cur[P->gene_of[t]]++] = (uint32_t) t;
    }

    lap("7 gene csr");
    P->info.n_classes = n_classes;
    P->info.n_pairs = n_pairs;
    P->info.n_runs = n_runs;
    P->info.n_items = n_items;
    P->info.nnz = nnz;
    P->info.nnz_total = nnz_total;
    P->info.n_classes_total = nclass_total;
    P->info.entry_bytes = entry_bytes;
    P->info.n_gene_ids = n_gene_ids;
    P->info.max_pairs_per_class = max_k;
    for (int b = 0; b < GBRS_KMAX + 2; ++b) { P->info.bucket_class0[b] = bclass[b]; P->info.bucket_pair0[b] = bpair[b]; }
    *out = P;
    return GBRS_OK;
  } catch (const std::bad_alloc&) {
    gbrs_set_error("gbrs_pack_create: out of host memory");
    return GBRS_E_NOMEM;
  }
}

extern "C" int gbrs_pack_get_info(gbrs_pack_t p, gbrs_pack_info* info) {
  if (!p || !info) { gbrs_set_error("gbrs_pack_get_info: null argument"); return GBRS_E_ARG; }
  *info = p->info;
  return GBRS_OK;
}

extern "C" int gbrs_pack_get_array(gbrs_pack_t p, const char* name, const void** ptr, int64_t* bytes) {
  if (!p || !name || !ptr || !bytes) { gbrs_set_error("gbrs_pack_get_array: null argument"); return GBRS_E_ARG; }
  const std::string s(name);
#define GBRS_ARR(nm, vec)                                                      \
  if (s == nm) {                                                               \
    *ptr = (vec).data();                                                       \
    *bytes = (int64_t) ((vec).size() * sizeof((vec)[0]));                      \
    return GBRS_OK;                                                            \
  }
  GBRS_ARR("rowptr", p->rowptr)
  GBRS_ARR("pairs", p->pairs)
  GBRS_ARR("count", p->count)
  GBRS_ARR("runptr", p->runptr)
  GBRS_ARR("class_id", p->class_id)
  GBRS_ARR("ent_cls", p->ent_cls)
  GBRS_ARR("ent_pair", p->ent_pair)
  GBRS_ARR("ent_run", p->ent_run)
  GBRS_ARR("item_off", p->item_off)
  GBRS_ARR("item_order", p->item_order)
  GBRS_ARR("item_desc", p->item_desc)
  GBRS_ARR("locus_order", p->locus_order)
  GBRS_ARR("locus_desc", p->locus_desc)
  GBRS_ARR("locus_item_ptr", p->locus_item_ptr)
  GBRS_ARR("gene_ptr", p->gene_ptr)
  GBRS_ARR("gene_loci", p->gene_loci)
  GBRS_ARR("gene_of", p->gene_of)
#undef GBRS_ARR
  gbrs_set_error("gbrs_pack_get_array: unknown array name '" + s + "'");
  return GBRS_E_ARG;
}

extern "C" int gbrs_pack_free(gbrs_pack_t p) {
  delete p;
  return GBRS_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Read rows for `gbrs compress` (src/gbrs/gbrs/emase_utils.py:52-71): H x CSC(reads x loci)  ->  one row of
// (locus | hapmask << 24) words per read, ascending locus inside a read.  The reference converts every matrix to CSR
// and walks the reads in python; this is the packer's merge (step 1 above) followed by a transposition: every thread
// owns a contiguous range of reads, scans the merged locus-major list in ascending locus order and appends to its own
// reads, so the rows come out sorted without atomics.  Stored zeros are not alignments.
// ---------------------------------------------------------------------------------------------------------------------
struct gbrs_rows {
  bigvec<int64_t> rowptr;
  bigvec<uint32_t> words;
};

extern "C" int gbrs_rows_create(const gbrs_pack_input* in, gbrs_rows_t* out) {
  if (!in || !out) { gbrs_set_error("gbrs_rows_create: null argument"); return GBRS_E_ARG; }
  const int T = in->T, H = in->H;
  const int64_t N = in->N;
  if (T <= 0 || N < 0 || H <= 0 || !in->indptr || !in->indices || (in->index_bytes != 4 && in->index_bytes != 8)) {
    gbrs_set_error("gbrs_rows_create: bad shape / index width"); return GBRS_E_ARG;
  }
  if (H > GBRS_HPAD) { gbrs_set_error("gbrs_rows_create: more than 8 haplotypes is not supported by the mask layout"); return GBRS_E_LIMIT; }
  if (T >= (1 << 24)) { gbrs_set_error("gbrs_rows_create: T must be < 2^24"); return GBRS_E_LIMIT; }
  const OmpThreadsGuard omp_guard(pack_threads());
  try {
    // per locus: (read << 8 | mask), reads ascending (gather + sort: the columns of a read-level file are small)
    std::vector<int64_t> ub(T + 1, 0);
    for (int t = 0; t < T; ++t) {
      int64_t s = 0;
      for (int h = 0; h < H; ++h) {
        if (!in->indptr[h] || in->indptr[h][t + 1] < in->indptr[h][t]) { gbrs_set_error("gbrs_rows_create: bad CSC arrays"); return GBRS_E_ARG; }
        s += in->indptr[h][t + 1] - in->indptr[h][t];
      }
      ub[t + 1] = ub[t] + s;
    }
    bigvec<uint64_t> tmp((size_t) ub[T]);
    std::vector<int64_t> lcount(T, 0);
    int bad = 0;
#pragma omp parallel for schedule(dynamic, 64)
    for (int t = 0; t < T; ++t) {
      uint64_t* dst = tmp.data() + ub[t];
      int64_t n = 0;
      for (int h = 0; h < H; ++h) {
        const int64_t b = in->indptr[h][t], e = in->indptr[h][t + 1];
        for (int64_t i = b; i < e; ++i) {
          if (in->values && in->values[h] && in->values[h][i] == 0.0) continue;
          const int64_t r = index_at(in->indices[h], in->index_bytes, i);
          if (r < 0 || r >= N) { bad = 1; continue; }
          dst[n++] = ((uint64_t) r << 8) | (uint64_t) h;
        }
      }
      std::sort(dst, dst + n);
      int64_t m = 0;
      for (int64_t i = 0; i < n;) {
        const uint64_t r = dst[i] >> 8;
        uint64_t mask = 0;
        while (i < n && (dst[i] >> 8) == r) { mask |= (uint64_t) 1 << (dst[i] & 0xFF); ++i; }
        dst[m++] = (r << 8) | mask;
      }
      lcount[t] = m;
    }
    if (bad) { gbrs_set_error("gbrs_rows_create: read index out of range"); return GBRS_E_ARG; }
    auto* R = new gbrs_rows();
    par_fill(R->rowptr, (size_t) N + 1, (int64_t) 0);
    int nt = 1;
#ifdef _OPENMP
    nt = omp_get_max_threads();
#endif
    // pairs per read (read-range ownership), prefix sum, then the fill with the same ownership
#pragma omp parallel for schedule(static, 1) num_threads(nt)
    for (int k = 0; k < nt; ++k) {
      const uint64_t r_lo = (uint64_t) (N * k / nt), r_hi = (uint64_t) (N * (k + 1) / nt);
      if (r_lo >= r_hi) continue;
      for (int t = 0; t < T; ++t) {
        const uint64_t* src = tmp.data() + ub[t];
        for (int64_t i = 0; i < lcount[t]; ++i) {
          const uint64_t r = src[i] >> 8;
          if (r >= r_lo && r < r_hi) ++R->rowptr[r + 1];
        }
      }
    }
    for (int64_t r = 0; r < N; ++r) R->rowptr[r + 1] += R->rowptr[r];
    R->words.resize((size_t) R->rowptr[N]);
    bigvec<int64_t> cur(R->rowptr.begin(), R->rowptr.end() - 1);
#pragma omp parallel for schedule(static, 1) num_threads(nt)
    for (int k = 0; k < nt; ++k) {
      const uint64_t r_lo = (uint64_t) (N * k / nt), r_hi = (uint64_t) (N * (k + 1) / nt);
      if (r_lo >= r_hi) continue;
      for (int t = 0; t < T; ++t) {
        const uint64_t* src = tmp.data() + ub[t];
        for (int64_t i = 0; i < lcount[t]; ++i) {
          const uint64_t r = src[i] >> 8;
          if (r >= r_lo && r < r_hi) R->words[cur[r]++] = (uint32_t) t | ((uint32_t) (src[i] & 0xFF) << 24);
        }
      }
    }
    *out = R;
    return GBRS_OK;
  } catch (const std::bad_alloc&) {
    gbrs_set_error("gbrs_rows_create: out of host memory");
    return GBRS_E_NOMEM;
  }
}

extern "C" int gbrs_rows_get(gbrs_rows_t r, const int64_t** rowptr, const uint32_t** words, int64_t* n_words) {
  if (!r || !rowptr || !words || !n_words) { gbrs_set_error("gbrs_rows_get: null argument"); return GBRS_E_ARG; }
  *rowptr = r->rowptr.data();
  *words = r->words.data();
  *n_words = (int64_t) r->words.size();
  return GBRS_OK;
}

extern "C" int gbrs_rows_free(gbrs_rows_t r) {
  delete r;
  return GBRS_OK;
}
