// dtb_internal.h -- declarations shared by the engine's translation units.
// Host-side launch wrappers live next to their kernels; dtb_api.cu plans a
// call and strings them together on one stream.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include "../../include/dtb200.h"

namespace dtb {

constexpr int MAX_KEYS = 8;
constexpr int MAX_PASSES = 16;

// Thread-local error slot + launch counter (dtb_api.cu)
void set_error(const std::string& msg);
void count_launch(int n = 1);
// Optional CUDA-event timing of a kernel family (option "profile"); no-ops otherwise.
void prof_begin(const char* name, cudaStream_t s);
void prof_end(cudaStream_t s);

#define DTB_CUDA_CHECK(expr)                                                     \
  do {                                                                           \
    cudaError_t _e = (expr);                                                     \
    if (_e != cudaSuccess) {                                                     \
      ::dtb::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));      \
      return DTB_ECUDA;                                                          \
    }                                                                            \
  } while (0)

#define DTB_TRY(expr)                                                            \
  do { int _rc = (expr); if (_rc != DTB_OK) return _rc; } while (0)

// ---------------------------------------------------------------------------
// Column statistics (replaces NumericStats<T>::compute_minmax, stats.cc:601-634)
// ---------------------------------------------------------------------------
// For integer stypes lo/hi are the signed min/max of the non-NA values; for
// float stypes they are the min/max of the order-preserving unsigned image
// (sort.cc:809-845 ASC transform).  bits_or / bits_and are OR / AND of that
// same image over the non-NA rows: bits that never vary need not be sorted.
struct ColStats {
  unsigned long long lo;       // int: (uint64)(int64 min); float: min image
  unsigned long long hi;
  unsigned long long bits_or;
  unsigned long long bits_and;
  unsigned long long nacount;
  unsigned long long nvalid;
};

int launch_col_stats(const void* data, int stype, int64_t n, ColStats* d_stats,
                     cudaStream_t s);
// The same statistics AND, from the same read of the column, the histogram of the low 8 bits of u (the
// sign-extended integer / float image) of every 4096-row tile: tile_hist u16[ntiles][256], NA rows apart in
// tile_na u16[ntiles].  Once edge / inc are known, the first radix pass folds it into its digit counts
// (PassIO::raw_hist) instead of reading the column a second time.
size_t stats_hist_bytes(int64_t n);          // bytes of tile_hist (tile_na follows, stats_na_bytes)
size_t stats_na_bytes(int64_t n);
int launch_col_stats_hist(const void* data, int stype, int64_t n, ColStats* d_stats, unsigned short* tile_hist,
                          unsigned short* tile_na, cudaStream_t s);

// ---------------------------------------------------------------------------
// Key normalisation parameters for one key column (restates _initB/_initI/_initF,
// sort.cc:690-845, as a function evaluated on the fly inside the kernels).
//   x = NA ? na_value : (((desc ? edge - u : u - edge) >> cshift) + inc)
// where u is the raw integer (sign-extended) or the float's ordered image.
// ---------------------------------------------------------------------------
struct KeyNorm {
  const void* data;
  int32_t  stype;
  int32_t  desc;
  unsigned long long edge;      // min (ASC) or max (DESC)
  unsigned long long na_value;  // 0 (NA first) or range+1 (NA last)
  unsigned long long inc;       // 1 (NA first) or 0 (NA last)
  int32_t  cshift;              // constant low bits dropped
  int32_t  bits;                // significant bits of x
  int32_t  lshift;              // position of x inside the composite key
  int32_t  pad;
};

struct KeyPlan {
  int      nkeys;
  int      total_bits;          // bits of the composite key
  int      group_shift;         // composite >> group_shift = group key (by-columns only)
  KeyNorm  k[MAX_KEYS];
};

// ---------------------------------------------------------------------------
// Radix sort (replaces SortContext::radix_psort / _radix_recurse,
// sort.cc:1129-1353, with stable LSD single-sweep passes)
// ---------------------------------------------------------------------------
struct PassPlan {
  int npasses;
  int shift[MAX_PASSES];
  int bits[MAX_PASSES];
};

// Composite key materialisation for multi-column keys: out[i] = X(row idx[i]) (idx NULL = identity).
int launch_compose_keys(const KeyPlan& kp, int64_t n, const int32_t* idx, void* keys_out,
                        int key_bytes, cudaStream_t s);

struct PassIO {
  int         src_kind;     // 0 packed keys + idx_in (idx_in NULL = identity), 1 raw column (identity idx)
  const void* keys_in;      // packed keys (src_kind 0)
  const int32_t* idx_in;
  void*       keys_out;     // may be NULL on the last pass of a sort-only call
  int32_t*    idx_out;
  void*       keys_stage;   // src_kind 1 only, optional: buffer that receives the normalised keys in the
                            // count kernel; the scatter kernel of the pass then reads them from there
  // first pass over a raw column whose normalisation keeps the low bits (cshift == 0): per-tile histogram of
  // the low 8 bits of u from launch_col_stats_hist; the pass folds it (x = +-(u - edge) + inc, NA -> na_value)
  // into its digit counts and does not run its count kernel
  const unsigned short* raw_hist = nullptr;
  const unsigned short* raw_na = nullptr;
  int         narrow_out = 0;     // 64-bit keys, > 0: keys_out receives (key >> narrow_out) as uint32 (later passes run on 32-bit keys)
};

// One stable pass = count + scan + scatter kernels.  work: radix_pass_work_bytes(n) of scratch;
// hmax (optional, device): receives the largest digit count of the pass.
size_t radix_pass_work_bytes(int64_t n);
// after_counts (optional): recorded on `s` once the digit totals of the pass (hmax) are final.
// group_count (optional, last pass only): uint32 table indexed by (key >> group_shift), zeroed by the
// caller; receives the number of rows of every group key (see launch_offsets_from_counts).
int launch_radix_pass(const PassIO& io, const KeyPlan& kp, int key_bytes, int64_t n,
                      int shift, int bits, uint32_t* work, uint32_t* hmax, cudaStream_t s,
                      cudaEvent_t after_counts = nullptr, uint32_t* group_count = nullptr, int group_shift = 0);

// Groupby offsets from a per-group-key row count table (small key domains): offsets[] = exclusive
// scan of the non-zero counts, gkeys[g] = key of group g, *d_ngroups = number of groups.
// table must be a multiple of 1024 entries and at most 2^22; scratch: uint64[2 * table / 1024 + 2].
int launch_offsets_from_counts(const uint32_t* count, int64_t table, int64_t n, int32_t* offsets,
                               uint32_t* gkeys, unsigned long long* d_ngroups, unsigned long long* scratch,
                               cudaStream_t s);

// Dense per-key tables for the multi-GPU merge of per-group partials (dtb_dense_scatter / dtb_dense_compact).
int launch_dense_scatter(const void* keys, int key_bytes, const void* vals, int64_t n, int64_t kmin, int64_t size,
                         void* table, uint32_t* present, cudaStream_t s);
int launch_dense_emit(const uint32_t* gidx, const void* table, int64_t ng, int64_t kmin, int key_bytes,
                      void* out_keys, void* out_vals, cudaStream_t s);

// ---------------------------------------------------------------------------
// Group offsets (replaces GroupGatherer, sort_groups.cc:34-117): heads where
// (key >> group_shift) changes, compacted into offsets[] by a single-pass scan.
// ---------------------------------------------------------------------------
// scratch: uint64[ntiles + 2] zeroed by the caller.  ngroups_out: device int64.
int64_t offsets_num_tiles(int64_t n);
// key_bytes 4/8: heads from adjacent sorted keys; key_bytes 1: `sorted_keys` is a uint8 head-flag
// array (multi-round composites wider than 64 bits, see launch_mark_heads).
int launch_group_offsets(const void* sorted_keys, int key_bytes, int group_shift, int64_t n,
                         int32_t* offsets_out, unsigned long long* d_ngroups,
                         unsigned long long* scratch, cudaStream_t s);
// flags[i] |= (keys[i] >> shift) != (keys[i-1] >> shift)
int launch_mark_heads(const void* sorted_keys, int key_bytes, int group_shift, int64_t n,
                      uint8_t* flags, cudaStream_t s);

// ---------------------------------------------------------------------------
// Reducers / gather
// ---------------------------------------------------------------------------
// acc0/acc1: device scratch, ngroups uint64 each.  n = offsets[ngroups] (rows under the groups).
int launch_reduce_impl(int op, const void* value, int stype, int64_t nrows_value,
                       const void* order, int order_is64, const int32_t* offsets, int64_t ngroups,
                       int64_t n, unsigned long long* acc0, unsigned long long* acc1,
                       void* out, cudaStream_t s, void* extra = nullptr);
// device scratch `extra` that launch_reduce_impl needs for `op` (sd: m2[ng]; nunique: one flag byte per row)
size_t reduce_extra_bytes(int op, int64_t ng, int64_t n);
int reduce_out_stype_host(int op, int stype);
// *d_bad (device int, zeroed by the caller) = 1 + index of a group with offsets[g] >= offsets[g+1] (or offsets[0] != 0).
int launch_offsets_check(const int32_t* offsets, int64_t ng, int* d_bad, cudaStream_t s);

// Direct-address reducers over a small normalised key domain (see dtb_reduce.cu).
enum { DIRECT_PLAIN = 0,        // one L2 atomic per row into acc[x]
       DIRECT_SMALL = 1,        // <= 2048 accumulators: per-CTA shared-memory tables (map: uint16 x -> group, or NULL)
       DIRECT_HOT = 2,          // skewed group sizes: rows of hot keys (map: uint8 hot[x]) fold in shared memory
       DIRECT_DEVICE_HOT = 3 }; // legacy overlapped mode: hot-key folding decided on the device from hot_count
struct DirectPlan {
  int kind;
  const void* map;
  int64_t nslots;               // accumulators in use: table, or ngroups for a dense-mapped small table
  const uint32_t* hot_count;
  uint32_t hot_thresh;
};
size_t direct_map_bytes(int64_t table);
// Chooses the streaming mode from the group structure (gmax = rows of the largest group) and builds the
// map it needs in map_scratch (direct_map_bytes(table) bytes, device).
int plan_direct(int64_t table, const uint32_t* gkeys, const int32_t* offsets, int64_t ngroups, int64_t n,
                int64_t gmax, void* map_scratch, cudaStream_t s, DirectPlan& dp);
int launch_reduce_direct(int op, const KeyPlan& kp, const DirectPlan& dp, const void* value, int stype, int64_t n,
                         int64_t table, const uint32_t* gkeys, int64_t ngroups,
                         unsigned long long* acc0, unsigned long long* acc1, void* out, cudaStream_t s);
int launch_direct_accumulate(int op, const KeyPlan& kp, const DirectPlan& dp,
                             const void* value, int stype, int64_t n, int64_t table,
                             unsigned long long* acc0, unsigned long long* acc1, cudaStream_t s);
// gkeys == NULL: the accumulators are indexed by group (dense-mapped small table).
int launch_direct_init(int op, const DirectPlan& dp, int64_t table, unsigned long long* acc0, unsigned long long* acc1, cudaStream_t s);
int launch_direct_accumulate_rows(int op, const KeyPlan& kp, const DirectPlan& dp, const void* value, int stype, int64_t n,
                                  int64_t table, unsigned long long* acc0, unsigned long long* acc1, cudaStream_t s);
int launch_direct_finalize(int op, int stype, const unsigned long long* acc0, const unsigned long long* acc1,
                           const uint32_t* gkeys, int64_t ngroups, void* out, cudaStream_t s);
int launch_nrows(const int32_t* offsets, int64_t ngroups, void* out, cudaStream_t s);
int launch_group_keys(const void* sorted_keys, int key_bytes, const int32_t* offsets, int group_shift,
                      int64_t ngroups, uint32_t* gkeys, cudaStream_t s);

// Bucketed multi-reducer (dtb_bucket.cu): all reducers of one value column in one sweep over rows partitioned
// by group-key bucket, shared-memory accumulators.  Words a column can ask for:
enum { BK_SUMI = 0, BK_SUMF = 1, BK_CNT = 2, BK_MIN = 3, BK_MAX = 4, BK_CNTNA = 5, BK_NWORDS = 6 };
constexpr int BK_MAX_DBITS = 20, BK_MIN_DBITS = 12;
// rows per (slab of tiles, bucket) of the group keys xkeys[i] >> gshift: slab_starts u32[bucket_starts_bytes(n)/4]
// (first output slot of every slab inside every bucket), bstart u32[nb+1] (bucket boundaries)
size_t bucket_starts_bytes(int64_t n);
int launch_bucket_starts(const uint32_t* xkeys, int gshift, int64_t n, int nb, uint32_t* slab_starts, uint32_t* bstart, cudaStream_t s);
constexpr int BK_MAXCOLS = 4;                 // value columns partitioned in one sweep
size_t bucket_scratch_bytes(int64_t n, int sum_value_bytes, int ncols);
int launch_bucketed_reduce(const uint32_t* xkeys, int gshift, int dbits, int ncols, const void* const* values,
                           const int* stypes, int64_t n, const uint32_t* slab_starts, const uint32_t* start,
                           unsigned long long* const (*acc_w)[BK_NWORDS], void* scratch, cudaStream_t s);
void fill_u64(unsigned long long* p, int64_t n, unsigned long long v, cudaStream_t s);

int launch_gather(const void* src, int stype, int64_t nrows_src, const void* order,
                  int order_is64, int64_t n, void* out, cudaStream_t s);

// grouped cumulative / window functions (dtb_window.cu); scratch: window_scratch_bytes(n) of device memory
int window_out_stype_host(int op, int stype);
size_t window_scratch_bytes(int64_t n);
int launch_window(int op, int64_t param, const void* value, int stype, int64_t nrows_value, const int32_t* order,
                  const int32_t* offsets, int64_t ngroups, int64_t n, void* out, void* scratch, cudaStream_t s);

int launch_iota32(int32_t* out, int64_t n, cudaStream_t s);
int launch_widen_u32(const uint32_t* in, int64_t n, int64_t* out, cudaStream_t s);   // ARR32 bit patterns -> ARR64

// ---------------------------------------------------------------------------
// SURVEY.md 8(f) rows (dtb_next.cu): ordered reducers, set operations, mode, join
// ---------------------------------------------------------------------------
int launch_firstlast(const void* v, int stype, int64_t nv, const int32_t* order, const int32_t* offsets,
                     int64_t ng, int last, void* out, cudaStream_t s);
int launch_expand_gid(const int32_t* offsets, int64_t ng, int64_t n, int32_t* gid, cudaStream_t s);
// integer slice applied inside every group (dtb_slice_groups)
struct SliceParams { long long start, stop, step, nrows; int has_start, has_stop; };
size_t slice_scratch_bytes(int64_t ng);
int launch_slice_groups_plan(const int32_t* offsets, int64_t ng, const SliceParams& p, void* scratch, int32_t* offsets_out,
                             int32_t* gsel, unsigned long long* totals, cudaStream_t s);
int launch_slice_groups_emit(const int32_t* offsets, const SliceParams& p, const int32_t* offsets_out, const int32_t* gsel,
                             int64_t ng_out, int64_t nout, int32_t* gid, int32_t* rows_out, cudaStream_t s);
// sum/cnt: the MEAN accumulators of the same column; m2: double[ng], zeroed
int launch_sd(const void* v, int stype, int64_t nv, const int32_t* order, const int32_t* offsets, int64_t ng, int64_t n,
              const unsigned long long* sum, const unsigned long long* cnt, double* m2, void* out, cudaStream_t s);
int launch_median(const void* v, int stype, int64_t nv, const int32_t* order, const int32_t* offsets,
                  int64_t ng, void* out, cudaStream_t s);
int launch_distinct_flags(const void* v, int stype, int64_t nv, const int32_t* order, const int32_t* offsets,
                          int64_t ng, int64_t n, int8_t* flag, cudaStream_t s);
int launch_set_select(const int32_t* order, const int32_t* offsets, int64_t ng, const int64_t* d_sizes, int K,
                      int mode, uint8_t* flags, cudaStream_t s);
int launch_set_emit(const int32_t* pos, int64_t nsel, const int32_t* order, const int32_t* offsets, int32_t* out_rows,
                    cudaStream_t s);
int launch_largest_group(const int32_t* offsets, int64_t ng, int64_t skip, unsigned long long* d_result, cudaStream_t s);
int launch_lower_bound(const void* sorted, int stype, int64_t n, const void* values, int64_t m, int64_t* out, cudaStream_t s);
int launch_join(int nkeys, const void* const* xcols, const int* xst, const void* const* jcols, const int* jst,
                int64_t nx, int64_t nj, int32_t* out, cudaStream_t s);

}  // namespace dtb
