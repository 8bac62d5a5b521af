/*
 * gbrs_em.h -- C ABI of the B200-native multiway EM quantifier (the loop behind `gbrs quantify -M 1..4`).
 *
 * The reference (churchill-lab/gbrs) is pure Python and has no FFI boundary for this path; its boundary is the
 * Python class `EMfactory` (src/gbrs/emase/EMfactory.py:15-392) working on an `AlignmentPropertyMatrix`
 * (src/gbrs/emase/AlignmentPropertyMatrix.py:25-111).  This header is the boundary a maintainer would bind from that
 * class with ctypes (see INTEGRATION.md): each entry point names the reference method(s) whose inner loop it replaces.
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in signatures (streams are passed as `void*` = cudaStream_t).
 *   - every function returns 0 on success, a negative GBRS_E_* code on failure; `gbrs_last_error()` gives the text.
 *   - the library owns NO device memory.  All device buffers are allocated by the caller (PyTorch tensors used as
 *     raw buffers) and handed over in `gbrs_em_dev`; host-side packing results live in a `gbrs_pack_t` until freed.
 *   - all launches are asynchronous on the given stream; only gbrs_em_run() / gbrs_em_read_ctrl() synchronise.
 *   - there is no CPU fallback: every compute entry point fails with GBRS_E_CUDA if no sm_100 device is usable.
 *
 * Device layout (DESIGN.md section 3): theta / effective lengths / numerators are stored locus-major with the haplotype
 * index minor and padded to 8 ( [T][8] doubles = one 64-byte line per locus ).  An alignment class is a row of
 * (locus, 8-bit haplotype mask) pair words; the incidence matrix is stored twice, class-major (row pass, E-step
 * normaliser) and locus-major (column pass, M-step reduction), so that both passes are gathers and no atomics are needed.
 */
#ifndef GBRS_EM_H
#define GBRS_EM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GBRS_EM_ABI_VERSION 8
#define GBRS_HPAD 8 /* haplotype slots per locus line */
#define GBRS_KMAX 8 /* classes with up to this many (class, locus) pairs take the fixed-width row pass */
#define GBRS_DEEP_LOCUS_ITEMS 8 /* a locus with more partial sums (column-pass items / tile slots) than this is summed by a
                                  whole warp in the locus kernel instead of eight lanes */

enum {
  GBRS_OK = 0,
  GBRS_E_ARG = -1,      /* bad argument (shape, model, null pointer) */
  GBRS_E_LIMIT = -2,    /* input exceeds a packing limit (H > 8, T >= 2^24, pairs >= 2^32) */
  GBRS_E_CUDA = -3,     /* CUDA runtime error / no usable device */
  GBRS_E_NUMERIC = -4,  /* non-finite value in the EM (reference: FloatingPointError under np.seterr(all='raise'),
                           src/gbrs/emase/EMfactory.py:256-257) */
  GBRS_E_NOMEM = -5,
  GBRS_E_STATE = -6     /* call order violated (e.g. run before prepare) */
};

const char* gbrs_last_error(void);
int gbrs_abi_version(void);

/* ------------------------------------------------------------------------------------------------------------------
 * Host-side packing: H x CSC(N x T) incidence  ->  class-major + locus-major packed rows.
 * Replaces the storage walked by Sparse3DMatrix (src/gbrs/emase/Sparse3DMatrix.py:26-66, reset :220-228,
 * multiply :314-377) and the `-G` masking of quantify (src/gbrs/gbrs/emase_utils.py:240-273).
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct gbrs_pack* gbrs_pack_t;

typedef struct {
  int32_t T;                   /* loci */
  int32_t H;                   /* haplotypes, 1..8 */
  int64_t N;                   /* alignment classes (rows of every CSC matrix) */
  const int64_t* const* indptr;  /* H pointers, each [T+1]: column pointers of haplotype h */
  const void* const* indices;    /* H pointers, each [indptr[h][T]]: class ids of the stored entries */
  int32_t index_bytes;         /* 4 (int32) or 8 (int64) for `indices` */
  const double* const* values; /* optional H pointers to the stored values; entries whose value is 0 are dropped
                                  (explicit zeros behave like `eliminate_zeros`); NULL = pure incidence */
  const double* count;         /* [N] class counts or NULL (= all ones, AlignmentPropertyMatrix.py:291-293) */
  const uint8_t* locus_hapmask;/* [T] or NULL: bit h set = haplotype h of this locus survives the -G genotype
                                  restriction (gtmask of emase_utils.py:247-269, one byte per locus) */
  const int32_t* gene_of;      /* [T] gene id per locus (ungrouped loci carry unique ids) or NULL (each locus alone) */
  int32_t shard_rank;          /* this rank's index ... */
  int32_t shard_count;         /* ... of this many row shards (classes split in contiguous ranges balanced by nnz) */
  int32_t item_len;            /* max entries per column-pass work item; 0 = default */
} gbrs_pack_input;

typedef struct {
  int64_t n_classes;   /* non-empty classes in this shard (after masking) */
  int64_t n_pairs;     /* (class, locus) pair words in this shard */
  int64_t n_runs;      /* (class, gene) runs in this shard */
  int64_t n_items;     /* column-pass work items */
  int64_t n_entries;   /* locus-major entry words incl. padding (every item starts at a multiple of 4 entries) */
  int64_t n_long_items;/* of which long (deep loci, up to 32 * item_len entries, processed by a whole warp) */
  int64_t nnz;         /* incidence entries in this shard (popcount over pair masks) */
  int64_t nnz_total;   /* incidence entries over all shards */
  int64_t n_classes_total;
  int32_t entry_bytes; /* 4 or 8: width of the locus-major entry words */
  int32_t n_gene_ids;  /* 1 + max gene id */
  int32_t max_pairs_per_class;
  int32_t n_deep_loci;  /* loci with more than GBRS_DEEP_LOCUS_ITEMS work items (they come first in locus_desc) */
  /* Classes are ordered by (min(pairs, GBRS_KMAX + 1), smallest locus, second-smallest locus, input class id).  bucket_class0[k-1] / bucket_pair0[k-1] is the
   * first class / first pair word of the classes with exactly k pairs (k = 1..GBRS_KMAX); index GBRS_KMAX starts the
   * "long" classes (more than GBRS_KMAX pairs), index GBRS_KMAX+1 is the end (= n_classes / n_pairs). */
  int64_t bucket_class0[GBRS_KMAX + 2];
  int64_t bucket_pair0[GBRS_KMAX + 2];
} gbrs_pack_info;

int gbrs_pack_create(const gbrs_pack_input* in, gbrs_pack_t* out);
int gbrs_pack_get_info(gbrs_pack_t p, gbrs_pack_info* info);
/* Borrowed host pointers to the packed arrays (valid until gbrs_pack_free).  `name` is one of:
 *   "rowptr"  uint32 [n_classes+1]   "pairs"   uint32 [n_pairs]  (locus | mask<<24, sorted by (gene, locus) in a class;
 *                                     class n < bucket_class0[GBRS_KMAX] with k pairs starts at bucket_pair0[k-1] + (n - bucket_class0[k-1]) * k)
 *   "count"   double [n_classes]     "runptr"  uint32 [n_classes+1]
 *   "class_id" uint32 [n_classes]    input class id of every packed class (the inverse of the class order)
 *   "ent_cls" / "ent_pair" / "ent_run"  entry words [n_entries], locus-major (index | mask << (8*entry_bytes-8));
 *                                     padding words carry an empty mask and index n_classes / n_pairs / n_runs
 *   "item_off" uint32 [n_items+1]    "locus_item_ptr" uint32 [T+1]   "item_order" uint32 [n_items]
 *   "item_desc" uint32 [n_items + 2][4] (two trailer descriptors, see gbrs_em_dev)  "locus_order" uint32 [T]   "locus_desc" uint32 [T][4]
 *   "gene_ptr" uint32 [n_gene_ids+1] "gene_loci" uint32 [T]     "gene_of" int32 [T]
 */
int gbrs_pack_get_array(gbrs_pack_t p, const char* name, const void** ptr, int64_t* bytes);
int gbrs_pack_free(gbrs_pack_t p);

/* Device-side packer: the same inputs (HOST arrays, pinned or not) and the same outputs as gbrs_pack_create -- array for
 * array, bit for bit -- built on the GPU; the packed arrays stay in device memory (nothing returns to the host but the
 * info record).  All device memory, results and temporaries alike, comes from the caller's allocator: `alloc(bytes, tag,
 * user)` returns device memory (256-byte aligned) or NULL; tags starting with "tmp:" may be released as soon as the call
 * returns, the others are the arrays named in gbrs_device_pack.  The call synchronises the stream.  GBRS_E_LIMIT for
 * inputs it does not take (stored values, N >= 2^31, more than 2^32 stored entries): use gbrs_pack_create.
 * No CPU fallback inside: without a CUDA device it fails with GBRS_E_CUDA. */
typedef void* (*gbrs_alloc_fn)(int64_t bytes, const char* tag, void* user);
typedef struct {
  const uint32_t* rowptr;      /* [n_classes + 1] */
  const uint32_t* pairs;       /* [n_pairs] */
  const double* count;         /* [n_classes] */
  const uint32_t* runptr;      /* [n_classes + 1] */
  const uint32_t* class_id;    /* [n_classes] */
  const void* ent_cls;         /* [n_entries] entry words (entry_bytes each) */
  const void* ent_pair;
  const void* ent_run;
  const uint32_t* item_desc;   /* [n_items + 2][4] */
  const uint32_t* locus_desc;  /* [T][4] */
  const int32_t* gene_of;      /* [T] */
  const uint32_t* gene_ptr;    /* [n_gene_ids + 1] */
  const uint32_t* gene_loci;   /* [T] */
} gbrs_device_pack;
int gbrs_pack_device(const gbrs_pack_input* in, gbrs_alloc_fn alloc, void* user, void* stream, gbrs_pack_info* info_out,
                     gbrs_device_pack* out);

/* ------------------------------------------------------------------------------------------------------------------
 * Tile layout of the fused model-4 update (DESIGN.md section 4): the classes of a shard, ordered by their smallest
 * locus, are cut into TILES (contiguous class ranges that touch at most `max_loci` distinct loci).  Everything a tile
 * needs is one contiguous blob, staged into shared memory with two bulk copies:
 *   part A  header, the tile's locus list + output slots, class counts, pair words as 16-bit (local locus | mask),
 *           laid out in "planes" (plane p = the p-th pair of every class that has one; classes sorted by descending
 *           width, so plane p holds classes 0 .. nplane[p]-1; every plane is padded to a multiple of 4 words with
 *           zero words = local locus 0 with an empty mask)
 *   part B  the tile's own locus-major copy for the M-step: work item words (sorted by key), a visiting order of the
 *           items (uint16, longest first), and 16-bit local class ids grouped by (local locus, nibble bucket) and cut
 *           into items of at most `item_len` ids
 * The kernel computes the class weights (E-step) into shared memory and reduces them per (locus, haplotype) without
 * leaving the SM -- no weight vector, no second full-size copy and no atomics; every tile writes one 64-byte partial
 * per locus it touches into its own slot, and the locus kernel sums a locus' slots in a fixed order (bit-reproducible).
 * Replaces, for model 4 / prepare: normalize_reads(READ) + sum(READ), AlignmentPropertyMatrix.py:288-298, 335-342.
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct gbrs_tiles* gbrs_tiles_t;

typedef struct {   /* 0 = default */
  int32_t max_classes;  /* classes per tile                  (default 128, at most 2047)            */
  int32_t max_loci;     /* distinct loci per tile            (default 16, at most 128)              */
  int32_t max_pairs;    /* pair words per tile               (default and at most 65535)            */
  int32_t max_entries;  /* M-step entries per tile           (default and at most 65535)            */
  int32_t max_items;    /* M-step work items per tile        (default 192)                          */
  int32_t item_len;     /* entries per work item             (default 16, at most 16)               */
} gbrs_tiles_params;

typedef struct {
  int64_t n_tiles;
  int64_t n_slots;       /* 64-byte partial-sum slots = sum over tiles of their locus count */
  int64_t blob_bytes;
  int64_t n_entries, n_items, n_pairs, n_classes;
  /* actual maxima over the tiles: the kernel sizes its shared memory from these */
  int32_t max_classes, max_loci, max_items, max_part_a_bytes, max_part_b_bytes, max_planes;
  int32_t max_slots_per_locus;
  int32_t item_len;
  int32_t n_deep_loci;  /* loci with more than GBRS_DEEP_LOCUS_ITEMS slots (first in locus_desc) */
  int32_t reserved;
} gbrs_tiles_info;

/* Builds the tile layout from a packed shard.  GBRS_E_LIMIT if a class touches more than `max_loci` loci (the caller
 * then stays on the two-pass kernels). */
int gbrs_tiles_create(gbrs_pack_t p, const gbrs_tiles_params* params, gbrs_tiles_t* out);
int gbrs_tiles_get_info(gbrs_tiles_t t, gbrs_tiles_info* info);
/* Borrowed host pointers (valid until gbrs_tiles_free):
 *   "blob"        bytes  [blob_bytes]      the tile blobs, each starting at a multiple of 128 bytes
 *   "tile_desc"   uint32 [n_tiles][16]     per VISITING slot (costliest tile first), see GBRS_TD_WORDS
 *   "locus_desc"  uint32 [T][4]            per visiting slot (most slots first): locus, first slot, one-past-last slot, 0 */
int gbrs_tiles_get_array(gbrs_tiles_t t, const char* name, const void** ptr, int64_t* bytes);
int gbrs_tiles_free(gbrs_tiles_t t);

/* A tile's blob = part A followed by part B (part B starts `a_bytes` after the tile's start); all sections start at
 * multiples of 16 bytes in the order listed, so their offsets follow from the counts in the tile descriptor.
 * Part A: header (GBRS_TH_WORDS uint32) | loci uint32 [n_loci] | slots uint32 [n_loci] | nplane uint16 [n_planes] |
 *         count double [n_classes] | pair planes uint16 (plane p: nplane[p] words, padded to a multiple of 4)
 * Part B: the tile's locus-major copy for the M-step.  A work item is a run of at most `item_len` entries (local class
 *         ids) of ONE key, key = local locus * 32 + bucket; bucket 0 = the pair hits all H haplotypes, 1..15 = value of
 *         the low mask nibble, 17..31 = 16 + value of the high mask nibble (a partial mask contributes one entry per
 *         non-zero nibble).  Items are numbered in key order and VISITED longest first, 32 at a time: a SLICE is 32
 *         consecutively visited items whose entries are stored transposed (sliced-ELL): entry i of the slice's lane l at
 *         word i * 32 + l, padded with the local class id n_classes (whose weight slot is zero) up to the slice's
 *         padded length (1, 2, 3, 4, 6, 8, 12 or 16).
 *         slice words uint32 [n_slices]: first word of the slice << 5 | padded length
 *         pos uint16 [n_items]: number (key order) of the item visited at that position
 *         run_key uint16 [n_runs], run_first uint16 [n_runs + 1]: items run_first[r] .. run_first[r+1]-1 (key order) make
 *         up key run_key[r]; keys without entries have no run
 *         entries uint16 [sell_words] */
enum { GBRS_TH_CLASSES = 0, GBRS_TH_LOCI = 1, GBRS_TH_PLANES = 2, GBRS_TH_RUNS = 3, GBRS_TH_ITEMS = 4, GBRS_TH_SLICES = 5,
       GBRS_TH_A_BYTES = 6, GBRS_TH_FULL = 7 /* the mask value meaning "all haplotypes" */, GBRS_TH_PAIRS = 8,
       GBRS_TH_ENTRIES = 9, GBRS_TH_B_BYTES = 10, GBRS_TH_SELL_WORDS = 11, GBRS_TH_WORDS = 12 };
/* Tile descriptor, GBRS_TD_WORDS uint32 per visiting slot (costliest tile first; the kernel reads only this, never the
 * header):  0 blob offset / 16 | 1 n_classes + (n_loci << 16) | 2 n_planes + (n_runs << 16) | 3 n_items + (n_slices << 16) |
 *   4 a_bytes | 5 full mask | 6 tile id | 7 bytes of the tile's blob | 8-11 byte offsets of slots, nplane, count, pair
 *   planes in part A | 12-15 byte offsets of pos, run_key, run_first, entries in part B */
enum { GBRS_TD_WORDS = 16 };

/* ------------------------------------------------------------------------------------------------------------------
 * Device descriptor: every pointer is a device pointer into a caller-owned buffer.
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t T, H;
  int32_t n_gene_ids;
  int32_t entry_bytes;
  int64_t n_classes, n_pairs, n_runs, n_items;
  int64_t n_entries;    /* locus-major entry words incl. padding */
  int64_t n_long_items; /* the first n_long_items entries of item_order are long items (one warp each) */
  int32_t n_ranks;     /* row shards taking part (1 = no exchange step) */
  int32_t max_iters_cap; /* capacity of err_log */
  int64_t bucket_class0[GBRS_KMAX + 2]; /* see gbrs_pack_info */
  int64_t bucket_pair0[GBRS_KMAX + 2];
  /* Fused cross-rank exchange over NVLink peer memory (optional, 2..8 ranks).  xchg_peer[r] is rank r's symmetric
   * exchange buffer as mapped into THIS process, zeroed once before first use.  xchg_enabled:
   *   0  the caller sums `acc` over ranks between gbrs_em_launch_local and gbrs_em_launch_update (e.g. ncclAllReduce)
   *   1  pull form: acc_local | acc_total | flags, (2 * 64 * T + 128) bytes; the owner of a slice loads it from every peer
   *   2  push form (default): recv[R][slice] | total | flags, (8 * (R * slice + 8 * T) + 128) bytes with
   *      slice = ((8 * T + R - 1) / R + 1) & ~1; every rank stores its values into the owners' recv rows while computing
   *      them, and the whole update is one launch (gbrs_em_launch_update then only runs the stop test)
   *   3  tag form: the push form (same buffer, same single launch) without flags -- every transported double carries
   *      the parity of its exchange number in its sign bit (the numerator is non-negative) and is polled by the thread
   *      that needs it; no tickets, fences or handshakes.  Negative theta is reported as GBRS_E_NUMERIC */
  int32_t xchg_enabled;
  int32_t xchg_rank;
  void* xchg_peer[8];
  void* xchg_mc;       /* optional: NVSwitch multicast mapping of the same symmetric buffers (NVLS); with it the
                          cross-rank sum is one multimem.ld_reduce + one multimem.st per element instead of peer
                          loads from / stores to every rank.  NULL = peer loads and stores */
  /* packed incidence (read-only) */
  const uint32_t* rowptr;
  const uint32_t* pairs;
  const double* count;
  const uint32_t* runptr;
  const void* ent_cls;
  const void* ent_pair;
  const void* ent_run;
  const uint32_t* item_off;
  const uint32_t* item_order;   /* [n_items] item ids in visiting order, bit 31 = full-mask item */
  const uint32_t* item_desc;    /* [n_items + 2][4] per visiting slot: first entry, one-past-last entry, item id, flags; then
                                   a trailer of two descriptors with the visiting-order positions where the SHORT items change
                                   kind / size class: {first short partial item of <= 8 words, of <= 4 words, first short full
                                   item, first short full item of <= 8 words}, {first short full item of <= 4 words, 0, 0, 0}
                                   (the column pass gives an item of one quad one lane, of two quads two, else eight) */
  const uint32_t* locus_order;  /* [T] loci in descending item count */
  const uint32_t* locus_desc;   /* [T][4] per visiting slot of locus_order: locus, first item, one-past-last item, 0 */
  const uint32_t* locus_item_ptr;
  const int32_t* gene_of;
  const uint32_t* gene_ptr;
  const uint32_t* gene_loci;
  /* tile layout of the fused model-4 update (all NULL / 0: the two-pass kernels are used) */
  const uint8_t* tile_blob;
  const uint32_t* tile_desc;       /* [n_tiles][GBRS_TD_WORDS] */
  const uint32_t* tile_locus_desc; /* [T][4] */
  double* tile_partial;            /* [n_slots][8] per-(tile, locus) partial sums */
  int64_t n_tiles, n_tile_slots;
  int32_t n_deep_loci;     /* two-pass layout: loci with more than GBRS_DEEP_LOCUS_ITEMS items */
  int32_t xchg_timeout_ms; /* wall-clock limit of a wait for peer flags; 0 = 20 s.  On a timeout the error flag (3) and the
                              stop flag are set and every block of the kernel leaves */
  int32_t tile_max_classes, tile_max_loci, tile_max_items, tile_max_a_bytes, tile_max_b_bytes, tile_n_deep_loci;
  /* state */
  double* theta;    /* [2][T][8] ping-pong allelic expression */
  double* efflen;   /* [T][8] effective lengths (1.0 where unused / no length file) */
  double* acc;      /* [T][8] M-step numerator: local after gbrs_em_launch_local, global after the exchange */
  double* iso;      /* [2][T] isoform totals sum_h theta */
  double* weights;  /* [max(n_classes, n_pairs, 8*n_runs) + 8] per-class / per-pair / per-run weights; the slot(s) after
                       the last real index are read by padding entries and must stay zero */
  double* subsets;  /* [T][32] subset sums of theta per locus: [0,16) over haplotype slots 0-3, [16,32) over slots 4-7 */
  double* wit;      /* [n_items][8] column-pass partials */
  double* part;     /* [GBRS_PART_SLOTS] block partial sums */
  double* gene_hap; /* [n_gene_ids][8] per-gene per-haplotype totals (models 1-3) */
  double* gamma;    /* [T] gene total broadcast to loci (models 1-3) */
  double* err_log;  /* [max_iters_cap] err_sum per iteration */
  double* scal;     /* [8] device scalars */
  int32_t* ctrl;    /* [16] control block, see GBRS_CTRL_* */
  /* Row-pass variant (last, so that the kernels' parameter offsets of the fields above stay as they were).
     1: a class of count 0 is absent -- the model-4 row pass gives it weight 0 without dividing, so a class whose entries
     all have theta 0 contributes nothing instead of 0 / 0 (models 1-3 guard their divisions already).  This is the EM on
     the matrix with the count-0 classes removed, as a bootstrap replicate needs it (gbrs_boot_resample).  A class with a
     positive count and a zero normaliser still raises GBRS_E_NUMERIC.  0 (default): the ordinary row pass. */
  int32_t zero_count_absent;
  int32_t reserved;  /* 0 */
} gbrs_em_dev;

#define GBRS_PART_SLOTS 4096 /* [0, 2048): block partial sums of the isoform totals; [2048, 4096): of the error */
enum { GBRS_CTRL_ITERS = 0, GBRS_CTRL_DONE = 1, GBRS_CTRL_ERROR = 2, GBRS_CTRL_PARITY = 3, GBRS_CTRL_MAX_ITERS = 4,
       GBRS_CTRL_PREPARED = 5, GBRS_CTRL_TICKET = 8 /* 8, 9, 10: block tickets */, GBRS_CTRL_XEPOCH = 12,
       GBRS_CTRL_TILE_NEXT = 13 /* work counter of the tile kernel, zeroed by the locus kernel */ };
enum { GBRS_SCAL_ERR = 0, GBRS_SCAL_SUM_PREV = 1, GBRS_SCAL_TARGET = 2, GBRS_SCAL_SUM_CUR = 3 };

/* theta0 from the incidence alone.  EMfactory.prepare numeric part (EMfactory.py:95-111) / EMfactory.reset (:113-138).
 * Split in two so that a row-sharded run can sum `acc` across ranks in between:
 *   gbrs_em_prepare_local:   acc[t][h] = sum_n count[n] / nnz[n]           (normalize_reads(READ) + sum(READ))
 *   gbrs_em_prepare_finish:  theta0 = acc / efflen, pseudocount rule (:105-111), isoform totals, control reset */
int gbrs_em_prepare_local(const gbrs_em_dev* d, void* stream);
int gbrs_em_prepare_finish(const gbrs_em_dev* d, double pseudocount, void* stream);

/* Load a caller-supplied theta (device [T][8]) as the current estimate and reset the loop control. */
int gbrs_em_set_theta(const gbrs_em_dev* d, const double* theta_dev, void* stream);
/* Device pointer of the current theta ([T][8]) after all work queued on `stream` so far (synchronises the stream). */
int gbrs_em_current_theta(const gbrs_em_dev* d, void* stream, double** theta_dev);

/* Arm the loop: EMfactory.run prologue (EMfactory.py:262-266): err_sum = 1e6, target = 1e6 * tol, iteration cap. */
int gbrs_em_run_begin(const gbrs_em_dev* d, double tol, int max_iters, void* stream);

/* One EM update, first half, on this rank's shard: E-step normalisers for `model` (update_probability_at_read_level,
 * EMfactory.py:146-212, with normalize_reads AlignmentPropertyMatrix.py:305-370 and multiply Sparse3DMatrix.py:314-377)
 * and the count-weighted column reduce (APM.sum(READ), AlignmentPropertyMatrix.py:288-298) into `acc`. */
int gbrs_em_launch_local(const gbrs_em_dev* d, int model, void* stream);
/* The E-step alone, EMfactory.update_probability_at_read_level (EMfactory.py:146-212): same passes as
 * gbrs_em_launch_local, but ONLY `acc` (this rank's numerator) is written -- theta, the isoform totals, the subset tables
 * and the exchange flags stay as they are, so the call can be repeated or followed by a full update. */
int gbrs_em_launch_estep(const gbrs_em_dev* d, int model, void* stream);
/* Second half (after `acc` holds the sum over all shards): theta' = acc / efflen (EMfactory.py:228-232), TPM-scaled
 * isoform-total L1 change and the stop test (EMfactory.py:267-279), entirely on the device. */
int gbrs_em_launch_update(const gbrs_em_dev* d, void* stream);

/* Posterior read-origin probabilities P[n,t,h] of one E-step (EMfactory.update_probability_at_read_level,
 * EMfactory.py:146-212: what the reference leaves in `probability`), written on a caller-supplied pattern.  For every
 * model  count_n * P[n,t,h] = theta[t][h] * W[idx(n,t,h)]  with W the weight vector of the row pass (idx = class for
 * model 4, (class, gene) run for model 3, pair for model 2, run * 8 + h for model 1), so the call runs the row pass of
 * `model` on `theta_src` ([T][8], device) with unit counts into `scratch` and gathers theta_src[t][h] * W[idx] onto the
 * output pattern: per haplotype h < H a CSC over (N input classes) x T, `indptr[h]` int64 [T+1] and `indices[h]`
 * (`index_bytes` 4 or 8) device arrays, sorted indices.  Every entry must be a stored entry of the packed pattern (the
 * incidence the descriptor was packed from, minus the -G restriction) or belong to a class outside this shard, which
 * gets 0.  `class_id` is the packer's array of that name (device).  Nothing the EM owns is written: theta, acc, weights,
 * subset / gene tables, iso, ctrl / scal / err_log and the exchange buffers stay as they are.  `scratch` (device, 256-byte
 * aligned) holds at least gbrs_em_posterior_scratch_bytes(d, model, N) bytes.  Synchronises the stream; GBRS_E_NUMERIC
 * if a class has a zero normaliser or a value is not finite (the reference raises FloatingPointError). */
int gbrs_em_posterior_scratch_bytes(const gbrs_em_dev* d, int model, int64_t N, int64_t* bytes);
int gbrs_em_posterior(const gbrs_em_dev* d, int model, const double* theta_src, const uint32_t* class_id, int64_t N,
                      const int64_t* const* indptr, const void* const* indices, int32_t index_bytes,
                      double* const* values, void* scratch, int64_t scratch_bytes, void* stream);
/* ------------------------------------------------------------------------------------------------------------------
 * Bootstrap replicates (DESIGN.md section 7.2): resample the M = sum(count) reads with replacement on the device and
 * write the replicate's class counts, so that the EM can be rerun on them.  The reference has no counterpart.
 * Replicate `replicate` of `seed` is fixed by (seed, replicate, count) alone:
 *   draw pair j (j = 0 .. ceil(M/2)-1) = Philox4x32-10 with counter (j & 0xffffffff, j >> 32, replicate, 0) and key
 *     (seed & 0xffffffff, seed >> 32) -> words x0..x3; draw 2j = x0 | x1 << 32, draw 2j+1 = x2 | x3 << 32 (unused if M is
 *     odd and 2j+1 = M);
 *   draw u is read k = floor(u * M / 2^64), which lands in the first input class n with prefix[n] > k;
 *   the replicate's count of input class n is the number of draws landing in it (integers summing to M).
 * `prefix` (device, int64 [N]) is the inclusive prefix sum of the input counts in input class order; 1 <= M =
 * prefix[N-1] <= 2^53, N < 2^32.  gbrs_boot_guide builds, in `scratch`, a guide table (entry g: the class of read
 * floor(g * M / G), G = the smallest power of two >= N, at most 2^24) so that each search starts within a few classes;
 * it is built once per (prefix, N, M) and read by every gbrs_boot_resample call on that scratch.  gbrs_boot_resample
 * then counts the draws of one replicate (integer atomics: exact and independent of order) and writes
 * count_out[p] = count of input class class_id[p] for the packed classes p < n_classes (`class_id`: the packer's array of
 * that name), ready to be the `count` of a descriptor.  `scratch` (device, 256-byte aligned) holds at least
 * gbrs_boot_scratch_bytes(N) bytes.  Both calls are asynchronous on `stream`. */
int gbrs_boot_scratch_bytes(int64_t N, int64_t* bytes);
int gbrs_boot_guide(const int64_t* prefix, int64_t N, int64_t M, void* scratch, int64_t scratch_bytes, void* stream);
int gbrs_boot_resample(const int64_t* prefix, int64_t N, int64_t M, uint64_t seed, uint32_t replicate,
                       const uint32_t* class_id, int64_t n_classes, void* scratch, int64_t scratch_bytes, double* count_out,
                       void* stream);

/* Bootstrap summaries (DESIGN.md section 7.3): the spread of B replicates, reduced on the device.
 * gbrs_boot_derive writes the [B][E] values of one (level, quantity) from `src` ([B][T][8], device: per replicate the
 * theta of the EM for GBRS_BOOT_TPM / GBRS_BOOT_SHARE, the numerator `acc` for GBRS_BOOT_COUNTS).  The level is the
 * isoforms (gene_ptr = gene_loci = NULL, L = T) or the genes g < n_genes = L of the packer's gene-major CSR `gene_ptr` /
 * `gene_loci` (loci of gene ids >= n_genes, the ungrouped ones, take no part).  With x[h][l] the level's value of
 * replicate b (a gene: summed over its loci in gene_loci order), element e = h * L + l of row b is
 *   GBRS_BOOT_COUNTS  x[h][l] for h < H, and at h = H the total sum_h x[h][l] (in h order)           E = (H + 1) L
 *   GBRS_BOOT_TPM     x[h][l] * (1e6 / S), S the sum of the row's H * L values in a fixed tree order; total as above
 *   GBRS_BOOT_SHARE   x[h][l] / sum_h' x[h'][l], NaN where that sum is 0                                E = H L
 * Asynchronous on `stream`. */
#define GBRS_BOOT_TPM 0
#define GBRS_BOOT_COUNTS 1
#define GBRS_BOOT_SHARE 2
int gbrs_boot_derive(const double* src, int64_t B, int32_t T, int32_t H, int32_t quantity, const uint32_t* gene_ptr,
                     const uint32_t* gene_loci, int32_t n_genes, double* values, void* stream);
/* gbrs_boot_summarize reduces every column e of `values` ([B][E] doubles, device) over its n non-NaN entries:
 *   mean[e] = sum / n, the sum compensated (Neumaier) and taken in row order;
 *   sd[e] = sqrt(sum (x - mean)^2 / (n - 1)) (ddof 1, a second pass around that mean, its sum compensated the same way),
 *     NaN if n < 2;
 *   qout[j * E + e] = numpy.nanquantile(column, q[j], method="linear"), bit for bit (virtual index (n - 1) q, numpy's
 *     _lerp with its t >= 0.5 branch, each operation rounded on its own);
 *   n[e] = n (int32; `n` may be NULL).  Every statistic is NaN where n = 0.
 * `q` is a host array of nq <= GBRS_BOOT_MAX_QUANTILES values in [0, 1]; the outputs are device arrays.  B <=
 * GBRS_BOOT_SUMMARY_MAX_B (a column is sorted in shared memory), GBRS_E_LIMIT above.  Needs no scratch; asynchronous on
 * `stream`; the same call gives the same bits. */
#define GBRS_BOOT_MAX_QUANTILES 16
#define GBRS_BOOT_SUMMARY_MAX_B 16384
int gbrs_boot_summarize(const double* values, int64_t B, int64_t E, const double* q, int32_t nq, double* mean, double* sd,
                        double* qout, int32_t* n, void* stream);

/* Device-to-device copy of the current theta (previous = 0) or of the other half of the ping-pong (previous = 1: after
 * an update, the theta that entered it) into dst [T][8]; the parity is read on the device, nothing synchronises. */
int gbrs_em_copy_theta(const gbrs_em_dev* d, int previous, double* dst, void* stream);

/* Per-kernel device timing of the first half (CUDA events on `stream` around the row pass, the column pass and the
 * numerator kernel), used by bench.py for the roofline figure.  gbrs_prof_read synchronises, returns the summed
 * milliseconds of the `n` recorded updates and resets the buffer. */
typedef struct gbrs_prof* gbrs_prof_t;
int gbrs_prof_create(int capacity, gbrs_prof_t* out);
int gbrs_em_launch_local_profiled(const gbrs_em_dev* d, int model, void* stream, gbrs_prof_t prof);
int gbrs_prof_read(gbrs_prof_t p, double* ms_row, double* ms_col, double* ms_acc, int32_t* n);
int gbrs_prof_free(gbrs_prof_t p);

/* Whole loop for a single rank (n_ranks == 1): EMfactory.run (EMfactory.py:234-287).  Iterations are queued
 * `poll_every` at a time; the stop decision is taken on the device and read back at each poll.  Returns the number of
 * iterations performed and copies their err_sum values into errs_host[0..iters) (may be NULL). */
int gbrs_em_run(const gbrs_em_dev* d, int model, double tol, int max_iters, int poll_every, void* stream,
                int32_t* iters_out, double* errs_host);

/* Same, reporting progress: after every poll `on_poll(first_iter, n_new, errs_new, user)` is called with the err_sum values
 * of the iterations finished since the previous poll (the reference prints its table row by row, EMfactory.py:280-287). */
typedef void (*gbrs_poll_cb)(int32_t first_iter, int32_t n_new, const double* errs_new, void* user);
int gbrs_em_run_cb(const gbrs_em_dev* d, int model, double tol, int max_iters, int poll_every, void* stream,
                   int32_t* iters_out, double* errs_host, gbrs_poll_cb on_poll, void* user);

/* Read the control block (synchronises the stream): ctrl_host[16], scal_host[8]. */
int gbrs_em_read_ctrl(const gbrs_em_dev* d, void* stream, int32_t* ctrl_host, double* scal_host);

/* report_alignment_counts columns (AlignmentPropertyMatrix.py:389-459) on the packed (unmasked) incidence:
 *   aln[t][8], uniq[t][8] (classes with exactly one alignment), locus_uniq[t] (classes hitting exactly one locus).
 * If gene_level != 0 the loci are first bundled into genes (_bundle_inline, :155-188) using gene_of / `n_real_genes`
 * (gene ids >= n_real_genes are ungrouped loci and vanish); outputs are then indexed by gene id. */
int gbrs_em_alignment_counts(const gbrs_em_dev* d, int gene_level, int32_t n_real_genes, double* aln_dev,
                             double* uniq_dev, double* locus_uniq_dev, void* stream);

/* Report tables (EMfactory.report_read_counts / report_depths, EMfactory.py:289-380; APM.report_alignment_counts,
 * AlignmentPropertyMatrix.py:442-459): rows `name<TAB>v0<TAB>v1...[<TAB>note]`, every value formatted exactly like
 * python's str(numpy.float64).  `data` is [n_cols][n_rows] (the reference's `cntdata`), `order` an optional row
 * permutation, `header` is written verbatim first (unless NULL).  Host only; rows are formatted by all host threads. */
int gbrs_write_table(const char* path, const char* header, const char* const* names, int64_t n_rows, const double* data,
                     int32_t n_cols, const char* const* notes, const int64_t* order, int32_t append);
/* Length table of EMfactory.prepare (EMfactory.py:60-89): `locus_hap<TAB>length` lines (`locus<TAB>length` when
 * n_haps == 1) -> out[locus * n_haps + hap] = max(length - read_length + 1, 1), zero where the file has no line.  Host
 * only.  Stops at the first line it does not take as well-formed and returns its 1-based number in *bad_line (0 = the
 * whole file was parsed); the caller then falls back to the reference's line loop, which raises the reference's error. */
int gbrs_parse_lengths(const char* path, const char* const* lnames, int64_t n_loci, const char* const* hnames,
                       int32_t n_haps, double read_length, double* out, int64_t* bad_line);
/* python repr of one double into `out` (NUL-terminated); returns the length or GBRS_E_ARG if `cap` is too small. */
int gbrs_format_double(double x, char* out, int32_t cap);

/* Host side of `gbrs compress` (src/gbrs/gbrs/emase_utils.py:52-71): H x CSC(reads x loci) -> one row of pair words
 * (locus | hapmask << 24, ascending locus) per read, CSR form.  Uses T, H, N, indptr, indices, index_bytes and values of
 * the gbrs_pack_input struct -- stored zeros are dropped; the other fields are ignored.  rowptr [N+1] (int64) and words stay valid
 * until gbrs_rows_free. */
typedef struct gbrs_rows* gbrs_rows_t;
int gbrs_rows_create(const gbrs_pack_input* in, gbrs_rows_t* out);
int gbrs_rows_get(gbrs_rows_t r, const int64_t** rowptr, const uint32_t** words, int64_t* n_words);
int gbrs_rows_free(gbrs_rows_t r);

/* ------------------------------------------------------------------------------------------------------------------
 * `gbrs compress`: equivalence classes of reads (src/gbrs/gbrs/emase_utils.py:46-72).  A read is a row of pair words
 * (locus | hapmask << 24, ascending locus) in CSR form; reads with identical rows form one class, classes are numbered
 * in order of first appearance (the reference's dict insertion order) and carry the sum of their reads' counts.
 *   rowptr_dev [n_reads+1], pairs_dev [rowptr[n_reads]], count_dev [n_reads] or NULL (= all ones, :58-59)   inputs
 *   class_of_read_dev [n_reads], first_read_dev [n_reads] (first n_classes valid: the read a class was first seen
 *   at), class_count_dev [n_reads] (first n_classes valid)                                                  outputs
 * `workspace_dev` must hold gbrs_ec_workspace_bytes(n_reads) bytes.  Grouping is by a seeded 64-bit hash followed by an
 * exact comparison; if two different rows collide, *collisions_out is non-zero, the outputs are undefined and the
 * caller repeats the call with another seed.  Synchronises the stream.  No CPU fallback. */
int gbrs_ec_workspace_bytes(int64_t n_reads, int64_t* bytes);
int gbrs_ec_build(int64_t n_reads, const uint32_t* rowptr_dev, const uint32_t* pairs_dev, const double* count_dev,
                  uint64_t seed, uint32_t* class_of_read_dev, uint32_t* first_read_dev, double* class_count_dev,
                  void* workspace_dev, int64_t workspace_bytes, void* stream, int64_t* n_classes_out,
                  int64_t* collisions_out);

/* ------------------------------------------------------------------------------------------------------------------
 * `gbrs reconstruct`: diplotype HMM along the genes of every chromosome (src/gbrs/gbrs/gbrs_utils.py:382-609).
 * S = H (H + 1) / 2 diplotypes in itertools.combinations_with_replacement order (:452-454).  All tables are gene-major
 * ([gene][S]): the chains of one call -- chromosomes of one sample, or of all samples of a cohort -- are laid one after
 * the other along the gene axis and described by `gbrs_hmm_chain` records.  No CPU fallback.
 * ---------------------------------------------------------------------------------------------------------------- */
/* Emission log-probabilities (gbrs_utils.py:462-488; get_genotype_probability :80-100, unit_vector :63-67):
 *   expr_dev       [n_genes][H]  gene-level TPM per haplotype
 *   avec_dev       [n_avec][H][H] alignment-specificity matrices; avec_index_dev [n_genes] = row of the gene's matrix
 *                  or -1 (no entry: naive vectors eye + 1e-4 and sigma 0.45, :472-483)
 *   init_dev       [S] null-model log-probabilities (:462-469), used for genes whose TPM sum is below expr_threshold
 *   eprob_dev      [n_genes][S]  out */
int gbrs_hmm_emission(int64_t n_genes, int32_t H, const double* expr_dev, const double* avec_dev,
                      const int32_t* avec_index_dev, const double* init_dev, double expr_threshold, double sigma,
                      double* eprob_dev, void* stream);

typedef struct {
  int64_t gene0;    /* first gene row of the chain in eprob / alpha / scaler / gamma / delta / backptr */
  int64_t tprob0;   /* index of the chain's first S x S matrix in tprob_dev (chains of different samples may share) */
  int32_t n_genes;  /* >= 1 */
  int32_t n_steps;  /* matrices the transition file holds for this chromosome: n_genes - 1, or >= n_genes (legacy
                       files; the back-trace then also uses matrix n_genes - 1, gbrs_utils.py:585-590) */
  int64_t state0;   /* first slot of the chain in states_dev; it fills min(n_genes, n_steps) + 1 slots */
} gbrs_hmm_chain;

/* Scaled forward pass (:498-523), backward pass (:527-548), posterior (:552-558), Viterbi scores (:565-575) and the
 * back-trace (:578-594) of every chain; two thread blocks per chain (forward / backward / posterior on exp(tprob),
 * Viterbi on tprob).
 *   tprob_dev     [n_matrices][S][S] log transition matrices as stored in the file (tprob[i][k][j]: towards state k of
 *                 gene i+1 from state j of gene i)
 *   tprob_lin_dev [n_matrices][S][S] work space: receives exp(tprob), computed once per call
 *   alpha_dev   [genes][S], scaler_dev [genes]   out: normalised forward log-probabilities and -log normaliser
 *   gamma_dev   [genes][S]   out: posterior (the reference's genoprobs, transposed)
 *   delta_dev   [genes][S]   out: Viterbi scores;  backptr_dev [genes][S] bytes: work space
 *   states_dev  out: per chain the states of genes 0 .. m-1 (m = min(n_genes, n_steps): the genes that get a genotype
 *               call) followed by the arg-max state of the last gene -- the reference's `viterbi_states` list */
int gbrs_hmm_run(int32_t n_chains, const gbrs_hmm_chain* chains_dev, int32_t H, const double* init_dev,
                 const double* eprob_dev, const double* tprob_dev, int64_t n_matrices, double* tprob_lin_dev,
                 double* alpha_dev, double* scaler_dev, double* gamma_dev, double* delta_dev, uint8_t* backptr_dev,
                 int32_t* states_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GBRS_EM_H */
