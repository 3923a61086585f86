/*
 * dtb200.h -- C-ABI of the B200-native groupby/sort engine that sits behind
 * h2oai/datatable's DT[i, j, by(), sort()] hot path.
 *
 * The reference has no FFI seam on this path (SURVEY.md 8b): the boundary is
 * its internal C++ function group() and the materialize() of its reducer /
 * view columns.  Every entry point below names the reference interface it
 * replaces (paths relative to /root/reference/src/core/).  INTEGRATION.md
 * shows the reference-side binding.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types cross this boundary.
 *   - every data pointer may be DEVICE memory or HOST memory (pinned or
 *     pageable); the engine detects which (cudaPointerGetAttributes).  Host
 *     inputs are staged to HBM, host outputs are copied back, inside the call.
 *   - `stream` is a cudaStream_t (NULL = legacy default stream).  Calls that
 *     return scalars (dtb_group*) block until their results are final; calls
 *     whose outputs are all in device memory (dtb_reduce, dtb_gather) only
 *     enqueue work on `stream`.  Host outputs are always complete on return.
 *   - return value 0 = success, negative = DTB_E*; dtb_last_error() gives the
 *     thread-local message (the reference throws dt::Error subclasses,
 *     utils/exceptions.h:43; a C ABI must not throw).
 *   - there is NO CPU fallback: without a usable CUDA device every compute
 *     call fails with DTB_ECUDA.
 */
#ifndef DTB200_H
#define DTB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DTB_ABI_VERSION 1

#if defined(__GNUC__)
#  define DTB_API __attribute__((visibility("default")))
#else
#  define DTB_API
#endif

/* stype codes == DtStype_* of src/datatable/include/datatable.h:32-42 */
#define DTB_STYPE_BOOL     1
#define DTB_STYPE_INT8     2
#define DTB_STYPE_INT16    3
#define DTB_STYPE_INT32    4
#define DTB_STYPE_INT64    5
#define DTB_STYPE_FLOAT32  6
#define DTB_STYPE_FLOAT64  7
#define DTB_STYPE_DATE32   17   /* sorted as int32, sort.cc:666 */
#define DTB_STYPE_TIME64   18   /* sorted as int64, sort.cc:668 */

/* SortFlag bits, sort.h:36-41 */
#define DTB_FLAG_NONE        0
#define DTB_FLAG_DESCENDING  2
#define DTB_FLAG_SORT_ONLY   4

/* NaPosition, sort.h:43-48 */
#define DTB_NA_FIRST   1
#define DTB_NA_LAST    2
#define DTB_NA_REMOVE  3

/* reducers: one per reference ColumnImpl */
#define DTB_OP_SUM      1   /* SumProd_ColumnImpl<T,true,..>  column/sumprod.h:30-62 */
#define DTB_OP_MEAN     2   /* Mean_ColumnImpl                column/mean.h:29-52    */
#define DTB_OP_MIN      3   /* MinMax_ColumnImpl<T,true>      column/minmax.h:29-62  */
#define DTB_OP_MAX      4   /* MinMax_ColumnImpl<T,false>                            */
#define DTB_OP_COUNT    5   /* CountUnary_ColumnImpl<T,false> column/count.h:31-56   */
#define DTB_OP_COUNTNA  6   /* CountUnary_ColumnImpl<T,true>                         */
#define DTB_OP_NROWS    7   /* CountNullary_ColumnImpl        column/count.h:60-89   */
/* within-group ordered reducers (SURVEY.md 8f; expr/head_reduce_unary.cc) */
#define DTB_OP_FIRST    8   /* FirstLast_ColumnImpl<true>     head_reduce_unary.cc:120-170: value of the group's first row */
#define DTB_OP_LAST     9   /* FirstLast_ColumnImpl<false>                                                                  */
#define DTB_OP_SD      10   /* sd_reducer                     head_reduce_unary.cc:197-219: sample sd, count <= 1 -> NA    */
#define DTB_OP_MEDIAN  11   /* Median_ColumnImpl              head_reduce_unary.cc:421-468: needs dtb_sort_grouped's order */
#define DTB_OP_NUNIQUE 12   /* op_nunique                     head_reduce_unary.cc:383-394: needs dtb_sort_grouped's order */

/* set operations, set_funcs.cc:126-456 */
#define DTB_SET_UNION      0
#define DTB_SET_INTERSECT  1
#define DTB_SET_SETDIFF    2
#define DTB_SET_SYMDIFF    3

/* error codes */
#define DTB_OK         0
#define DTB_EINVAL    -1   /* bad argument (ValueError / TypeError in the reference) */
#define DTB_ENOTIMPL  -2   /* unsupported stype (NotImplError, sort.cc:673): caller falls back outside the path */
#define DTB_ECUDA     -3   /* CUDA runtime failure or no device */
#define DTB_ENOMEM    -4
#define DTB_ENOSPACE  -5   /* caller-provided output too small; *ngroups_out still set */

typedef void* dtb_stream;           /* cudaStream_t */

/* A material fixed-width column: raw typed buffer with NA sentinels
 * (SentinelFw_ColumnImpl, column/sentinel_fw.h:34-78; NA constants stype.h:186-197). */
typedef struct dtb_col {
  const void* data;
  int32_t     stype;
  int32_t     reserved;
} dtb_col;

/* Thread-local message of the last failing call on this thread ("" if none). */
DTB_API const char* dtb_last_error(void);

/* DTB_ABI_VERSION of the loaded library (cf. DtABIVersion(), datatable.h:49). */
DTB_API int dtb_abi_version(void);

/* Bytes per element of an stype (0 = unsupported on this path). */
DTB_API int dtb_stype_size(int stype);

/* Output stype of reducer `op` applied to a column of `stype`
 * (expr/fexpr_sumprod.cc:50-66, fexpr_mean.cc:49-78, fexpr_minmax.cc:50-72,
 *  fexpr_count.cc:47-128); 0 if the combination is invalid. */
DTB_API int dtb_reduce_out_stype(int op, int stype);

/* Selects the CUDA device used by this thread's subsequent calls and creates
 * the engine context on it.  Optional: the first compute call does it for the
 * current device. */
DTB_API int dtb_init(int device);

/*
 * dtb_group -- replaces RiGb group(columns, flags, na_pos)  (sort.h:56-58,
 * sort.cc:1411-1495) for material bool/int/float key columns.
 *
 *   keys[nkeys], flags[nkeys] : key columns (by-columns first) and their
 *                               SortFlag bits
 *   na_pos                    : DTB_NA_*
 *   nrows                     : rows per column (<= INT32_MAX; more: dtb_group64)
 *   order_out                 : int32[nrows]  -- the ARR32 RowIndex payload
 *                               (sort.cc:598-608); with DTB_NA_REMOVE only the
 *                               first *norder_out entries are written
 *   offsets_out               : int32[offsets_cap] -- Groupby offsets,
 *                               offsets[0]=0 .. offsets[ng]=nrows
 *                               (groupby.h:41-47); may be NULL when flags[0]
 *                               has SORT_ONLY
 *   *ngroups_out              : number of groups; -1 when the reference
 *                               returns an empty Groupby (sort.cc:1491-1493)
 *   *norder_out               : valid entries in order_out
 *
 * Bit-exact with the reference for order and offsets.
 */
DTB_API int dtb_group(const dtb_col* keys, int nkeys, const int* flags, int na_pos,
              int64_t nrows, dtb_stream stream,
              void* order_out, void* offsets_out, int64_t offsets_cap,
              int64_t* ngroups_out, int64_t* norder_out);

/*
 * dtb_group64 -- dtb_group with the ARR64 layout: order_out is int64[nrows] (RowIndex ARR64,
 * rowindex_array.cc:50-60; the reference's new sorter emits it above INT32_MAX rows, sort/sorter.cc:74-81)
 * and offsets_out is int64[offsets_cap] (the reference's Groupby is int32-only, sort.h:119-124 "TODO: Add
 * support for 64-bit groups" -- this is the variant SURVEY.md 8b asks for).  nrows < 2^32 - 65536 on one
 * GPU (beyond that the frame is row-partitioned across GPUs, datatable_b200/dist.py); works for any
 * smaller nrows too.  Same ordering, groups and NA rules as dtb_group.
 */
DTB_API int dtb_group64(const dtb_col* keys, int nkeys, const int* flags, int na_pos,
              int64_t nrows, dtb_stream stream,
              void* order_out, void* offsets_out, int64_t offsets_cap,
              int64_t* ngroups_out, int64_t* norder_out);

/*
 * Handle variant: results stay resident in HBM (no worst-case caller buffers,
 * no host round trip before the reducers).  The handle owns order/offsets.
 */
typedef struct dtb_groupby dtb_groupby;

DTB_API int dtb_groupby_create(const dtb_col* keys, int nkeys, const int* flags,
                       int na_pos, int64_t nrows, dtb_stream stream,
                       dtb_groupby** out);
/*
 * Fused variant: group() plus `nreducers` per-group reducers in one call (the j-expressions of
 * DT[:, {sum(f.v), ...}, by(f.k)] are known before group() runs, expr/eval_context.cc:144-172).
 * When the group-key domain is small the reducers only need the key columns, so they run on an
 * engine-owned side stream concurrently with the sort passes.  Results are owned by the handle:
 * dtb_groupby_reduced(g, i) = device buffer of ngroups elements of stype
 * dtb_reduce_out_stype(op, value.stype).  Equivalent to dtb_groupby_create + dtb_groupby_reduce.
 */
typedef struct dtb_reduce_spec {
  int32_t op;          /* DTB_OP_* */
  int32_t reserved;
  dtb_col value;       /* ignored for DTB_OP_NROWS */
} dtb_reduce_spec;

DTB_API int dtb_groupby_create_reduce(const dtb_col* keys, int nkeys, const int* flags,
                       int na_pos, int64_t nrows, dtb_stream stream,
                       const dtb_reduce_spec* reducers, int nreducers, dtb_groupby** out);
DTB_API const void* dtb_groupby_reduced(const dtb_groupby* g, int i);

DTB_API int64_t     dtb_groupby_norder(const dtb_groupby* g);    /* RowIndex length               */
DTB_API int64_t     dtb_groupby_ngroups(const dtb_groupby* g);   /* -1 = no Groupby (sort only)   */
DTB_API const void* dtb_groupby_order(const dtb_groupby* g);     /* device int32[norder]          */
DTB_API const void* dtb_groupby_offsets(const dtb_groupby* g);   /* device int32[ngroups+1]/NULL  */
DTB_API int         dtb_groupby_destroy(dtb_groupby* g, dtb_stream stream);

/*
 * dtb_reduce -- replaces ColumnImpl::materialize() of the per-group reducer
 * columns (column/reduce_unary.h:30-68 driven by column/latent.cc:103-135 and
 * column/column_impl.cc:78-103): value column viewed through the RowIndex
 * `order` (NULL = identity), segmented by `offsets`.
 *
 *   out : ngroups elements of stype dtb_reduce_out_stype(op, value.stype);
 *         NA results are written as the stype's NA sentinel.
 *   nrows_value : rows in the value column (bounds the gather).
 *
 * SUM over integers/bool, MIN, MAX, COUNT*, NROWS are bit-exact.  Floating
 * SUM/MEAN are accumulated in float64 with an unspecified association order:
 * within 1e-6 relative of the reference's sequential sum (float32 SUM: the
 * reference accumulates sequentially in float32, so agreement is O(n*2^-24)).
 */
DTB_API int dtb_reduce(int op, dtb_col value, int64_t nrows_value,
               const void* order, int order_is64,
               const void* offsets, int64_t ngroups,
               dtb_stream stream, void* out);

/*
 * dtb_groupby_reduce -- dtb_reduce over the handle's RowIndex / offsets.  When the handle's
 * key domain is small (normalised group key < 2^22 values) and the key columns passed to
 * dtb_groupby_create live in device memory, the reducer streams the key and value columns in
 * storage order and accumulates with L2 atomics instead of gathering through the RowIndex;
 * the caller must keep those key columns alive and unchanged while the handle is used.
 * Results are identical to dtb_reduce (floating sums up to association order).
 */
DTB_API int dtb_groupby_reduce(dtb_groupby* g, int op, dtb_col value, int64_t nrows_value,
                       dtb_stream stream, void* out);

/*
 * The same reducer fed piecewise: the value column arrives in row ranges (e.g. the chunks of a host
 * column on their way over PCIe, each folded as soon as it is in HBM -- the reference's reducers,
 * column/sumprod.h / minmax.h / count.h, need the whole column before they start).  Streaming path only
 * (see dtb_groupby_reduce: small key domain, device key columns) and DTB_OP_SUM .. DTB_OP_COUNTNA;
 * otherwise _begin returns DTB_ENOTIMPL and the caller uses dtb_groupby_reduce on the whole column.
 *   _begin : allocates and initialises the accumulator tables
 *   _add   : value_rows = DEVICE pointer to rows [row0, row0 + nrows) of the value column, enqueued on `stream`
 *            (the caller orders it after the piece's upload); every row exactly once over all calls
 *   _end   : finalises into out (host or device, ngroups elements of dtb_reduce_out_stype) and frees the state
 *            (also on error).  Results as dtb_groupby_reduce.
 */
typedef struct dtb_reduce_state dtb_reduce_state;
DTB_API int dtb_groupby_reduce_begin(dtb_groupby* g, int op, int value_stype, dtb_stream stream, dtb_reduce_state** out);
DTB_API int dtb_groupby_reduce_add(dtb_reduce_state* st, const void* value_rows, int64_t row0, int64_t nrows, dtb_stream stream);
DTB_API int dtb_groupby_reduce_end(dtb_reduce_state* st, dtb_stream stream, void* out);

/*
 * dtb_gather -- replaces materialisation of ArrayView_ColumnImpl<int32/int64>
 * (column/view.cc:88-155): out[i] = order[i] < 0 ? NA : src[order[i]].
 */
DTB_API int dtb_gather(dtb_col src, int64_t nrows_src,
               const void* order, int order_is64, int64_t n,
               dtb_stream stream, void* out);

/*
 * dtb_window -- grouped cumulative and window functions: one output row per position of the grouped frame, in
 * group order.  Replaces the materialisation of the reference's per-row group functions (the GtoALL columns of
 * EvalContext):
 */
#define DTB_WIN_CUMSUM   1   /* CumSumProd_ColumnImpl<T,true,REV>      column/cumsumprod.h:48-95     */
#define DTB_WIN_CUMPROD  2   /* CumSumProd_ColumnImpl<T,false,REV>                                   */
#define DTB_WIN_CUMMIN   3   /* CumMinMax_ColumnImpl<T,true,REV>       column/cumminmax.h:48-110     */
#define DTB_WIN_CUMMAX   4
#define DTB_WIN_CUMCOUNT 5   /* CumcountNgroup_ColumnImpl<true,REV>    column/cumcountngroup.h:52-70 */
#define DTB_WIN_NGROUP   6
#define DTB_WIN_FILLNA   7   /* FExpr_FillNA::fill_rowindex            expr/fexpr_fillna.cc:86-118   */
#define DTB_WIN_SHIFT    8   /* compute_lag_rowindex                   expr/head_func_shift.cc:41-62 */
/*
 * Output stype of window op `op` over a value column of `stype`; 0 = invalid combination (TypeError in the
 * reference: cumsum / cumprod of date32 or time64).  cumsum / cumprod: bool, int8..int64 -> int64 (wraps mod 2^64),
 * float32 / float64 unchanged.  cummin / cummax / fillna / shift keep the stype.  cumcount / ngroup: int64.
 */
DTB_API int dtb_window_out_stype(int op, int stype);
/*
 *   value, nrows_value : the value column (ignored by CUMCOUNT / NGROUP), viewed through `order`
 *   order              : int32[offsets[ngroups]] RowIndex, or NULL = identity
 *   offsets            : int32[ngroups+1] Groupby (one group [0, n] for a frame without by())
 *   param              : `reverse` (0 / 1) for CUMSUM .. FILLNA; the shift n for SHIFT (int32 range, else
 *                        DTB_EINVAL): out[p] = v[order[p - n]] when p - n lies in p's group, else NA
 *   out                : offsets[ngroups] elements of dtb_window_out_stype(op, value.stype)
 * NA counts as 0 in CUMSUM and 1 in CUMPROD; CUMMIN / CUMMAX / FILLNA skip NAs (a leading NA stays NA) and break
 * ties toward the current row.  Integer sums and products are exact mod 2^64; float sums and products are
 * accumulated in float64 with an unspecified association order.  Everything else is bit-exact.
 */
DTB_API int dtb_window(int op, int64_t param, dtb_col value, int64_t nrows_value,
               const void* order, const void* offsets, int64_t ngroups, dtb_stream stream, void* out);

/*
 * dtb_slice_groups -- the `i` node of DT[i, j, by(), sort()] when i is an integer slice (or an integer: the
 * slice [i, i+1)); replaces FExpr_Literal_SliceInt::evaluate_iby (expr/fexpr_literal_sliceint.cc:82-170) and
 * FExpr_Literal_Int::evaluate_iby (expr/fexpr_literal_int.cc:146-192): the slice is applied inside every group
 * of the grouped frame.  offsets: int32[ngroups+1] (the Groupby; one group [0, n] under sort() alone).
 * start / stop / step: DTB_SLICE_NA for a missing member; step 0 = `stop` copies of row `start` (the reference's
 * repeat slice).  rows_out: int32 positions INTO THE ROWINDEX of group() (the caller composes: RowIndex product =
 * dtb_gather on the index buffer, eval_context.cc:154-163), at most rows_capacity of them (DTB_ENOSPACE with
 * *nrows_out = the number needed otherwise; the grouped frame's row count always suffices for step != 0);
 * offsets_out: int32[ngroups+1], the remaining groups -- groups that select nothing disappear.
 * Host or device pointers.
 */
#define DTB_SLICE_NA INT64_MIN
DTB_API int dtb_slice_groups(const void* offsets, int64_t ngroups, int64_t start, int64_t stop, int64_t step,
                     dtb_stream stream, void* rows_out, int64_t rows_capacity, void* offsets_out,
                     int64_t* ngroups_out, int64_t* nrows_out);

/*
 * dtb_sort_grouped -- replaces Column::sort_grouped (sort.cc:1499-1530): reorders the rows INSIDE every
 * group of (order, offsets) by `value` ascending, NA first, stable; the groups themselves stay where
 * they are.  order_out: int32[offsets[ngroups]].  DTB_OP_MEDIAN / DTB_OP_NUNIQUE expect this order
 * (the reference's Median_ColumnImpl calls sort_grouped in its pre_materialize_hook).
 */
DTB_API int dtb_sort_grouped(dtb_col value, int64_t nrows_value, const void* order, const void* offsets,
                     int64_t ngroups, dtb_stream stream, void* order_out);

/*
 * dtb_set_select -- the group-selection step of union / intersect / setdiff / symdiff
 * (set_funcs.cc:126-456).  The caller concatenated K single-column inputs (input k holds the rows
 * cum_sizes[k-1] .. cum_sizes[k]-1), grouped the result with dtb_group and passes its (order, offsets).
 * rows_out: int32[ngroups] receives, for every group that the operation keeps, the row index of the
 * group's first row (ascending group order); *nout = how many.  Gathering the concatenated column
 * through rows_out gives the result column.
 */
DTB_API int dtb_set_select(int mode, const void* order, const void* offsets, int64_t ngroups,
                   const int64_t* cum_sizes, int ninputs, dtb_stream stream, void* rows_out, int64_t* nout);

/*
 * dtb_largest_group -- the mode / nmodal scan of NumericStats<T>::compute_sorted_stats
 * (stats.cc:984-991): index and size of the first largest group among groups [skip, ngroups)
 * (skip = 1 when the first group holds the NA rows).  *index_out = -1 when there is no such group.
 */
DTB_API int dtb_largest_group(const void* offsets, int64_t ngroups, int64_t skip, dtb_stream stream,
                      int64_t* index_out, int64_t* size_out);

/*
 * dtb_join -- replaces natural_join(xdt, jdt) (frame/join.cc:392-470): for every row of X the index
 * of the row of the keyed frame J whose key columns all compare equal (FwCmp, join.cc:199-232: NA
 * matches NA; an X value that J's integer key type cannot represent matches nothing), or the NA
 * index INT32_MIN.  jkeys must be sorted ascending, NA first, with unique rows -- what setting a key
 * produces (DataTable::set_key, frame/key.cc:118-180 = dtb_group + uniqueness check + dtb_gather).
 * index_out: int32[nrows_x], the ARR32 RowIndex the reference applies to J's non-key columns.
 */
DTB_API int dtb_join(const dtb_col* xkeys, const dtb_col* jkeys, int nkeys, int64_t nrows_x, int64_t nrows_j,
             dtb_stream stream, void* index_out);

/*
 * Multi-GPU merge of per-group partials over a small group-key domain (one process per GPU; the
 * reference is single-process, SURVEY.md 8e -- this is north_star's "final NCCL reduce of per-group
 * partials").  Each rank scatters its (group key, 8-byte partial) list into a dense table indexed by
 * key - kmin; the caller all-reduces `table` (SUM, typed as the partials are) and `present` (uint32
 * SUM) in place with NCCL; dtb_dense_compact then lists the keys that occur on any rank, ascending,
 * with their merged partials.  Device buffers only.  table/present must be zeroed before the scatter;
 * table_size: multiple of 1024, at most 2^22.  key_stype: DTB_STYPE_INT32 or DTB_STYPE_INT64.
 */
DTB_API int dtb_dense_scatter(const void* keys, int key_stype, const void* vals, int64_t n, int64_t kmin,
                      int64_t table_size, void* table, void* present, dtb_stream stream);
DTB_API int dtb_dense_compact(const void* table, const void* present, int64_t table_size, int64_t kmin,
                      int key_stype, void* out_keys, void* out_vals, int64_t* ngroups_out, dtb_stream stream);

/*
 * dtb_lower_bound -- out[i] (int64) = number of rows of the ascending, NA-free column `sorted` that are
 * smaller than values[i]: the cut points of the key-range exchange between GPUs (no reference analogue;
 * SURVEY.md 8e).  Both columns share one stype.
 */
DTB_API int dtb_lower_bound(dtb_col sorted, int64_t nrows, dtb_col values, int64_t nvalues,
                    dtb_stream stream, void* out);

/*
 * Residency bracket for HOST buffers: between dtb_cache_begin() and the matching dtb_cache_end() (calls
 * nest; per thread) a host input staged into HBM by any entry point stays there and is reused by later
 * calls that pass the same (pointer, size); the RowIndex / offsets that dtb_group copied to host memory
 * are remembered too, so dtb_reduce / dtb_gather on them upload nothing.  The reference-side hook puts
 * the bracket around EvalContext::evaluate() (INTEGRATION.md): one upload per column per query, where the
 * reference's Buffers are host memory (buffer.cc:261-300).  The caller promises that the bracketed host
 * buffers do not change; dtb_cache_end() releases the copies.  dtb_last_call_stats().cache_hits counts the
 * cache hits of the last call.
 */
DTB_API int dtb_cache_begin(void);
DTB_API int dtb_cache_end(void);

/* Copies nbytes between any two host/device buffers on `stream`
 * (cudaMemcpyDefault) and waits for completion.  Lets a binding read the
 * HBM-resident results of a dtb_groupby without linking the CUDA runtime. */
DTB_API int dtb_memcpy(void* dst, const void* src, int64_t nbytes, dtb_stream stream);

/*
 * Engine options, the analogue of dt.options.sort.* (sort.cc:259-349).
 *   "radix_bits"   largest digit width of the LSD passes: 4..8, or 0 (default) = 8 bits (wider digits were
 *                  built and measured slower twice, DESIGN.md 4.2)
 *   "verbose"      1 = print the pass plan to stderr
 *   "profile"      1 = bracket every kernel with CUDA events on the call's stream (the calls do not wait for
 *                  them; dtb_profile_count / dtb_profile_reset do)
 *   "overlap_reducers" 1 = dtb_groupby_create_reduce runs the direct-address reducers on a side stream
 *                  concurrently with the sort passes (default 0: same stream, measured equally fast)
 *   "stage_keys"   0 (default) = the first count and scatter kernels of a single raw key column normalise it on
 *                  the fly (no normalised-key array is written); 1 = the first count kernel materialises the
 *                  normalised keys and the first scatter reads those (round-1 behaviour; measured at 1e9 rows:
 *                  +0.5 ms and +8 GB of DRAM traffic for int32 keys, +0.9 ms for float64)
 *   "fuse_stats_hist" 1 (default) = single-column keys: the statistics kernel also counts the low 8 bits of every
 *                  tile and the first radix pass folds that into its digit counts instead of reading the column
 *                  again (DESIGN.md 4.1); 0 = separate statistics and count kernels
 *   "bucketed_reducers" 1 (default) = value columns that would cost two or more L2 atomics per row (mean, or
 *                  several reducers of one column) take the bucketed multi-reducer (dtb_bucket.cu); 0 = always
 *                  one streaming pass per reducer
 *   "trim_scratch" (set only) release the calling thread's cached HBM scratch slab
 */
DTB_API int dtb_set_option(const char* name, int64_t value);
DTB_API int dtb_get_option(const char* name, int64_t* value);

/* Kernel timings collected while option "profile" is on (accumulated on the calling
 * thread until dtb_profile_reset): record i = (kernel family name, milliseconds).
 * dtb_profile_count waits for the recorded events of earlier calls before it answers. */
DTB_API int dtb_profile_count(void);
DTB_API int dtb_profile_get(int i, char* name, int cap, double* ms);
DTB_API int dtb_profile_reset(void);

/* Per-call statistics of the last dtb_group / dtb_groupby_create on this thread:
 * number of kernels launched, radix passes, significant key bits. */
typedef struct dtb_call_stats {
  int32_t kernels_launched;
  int32_t radix_passes;
  int32_t key_bits;
  int32_t cache_hits;        /* host inputs served from the dtb_cache_begin/end residency cache */
  int64_t scratch_bytes;
} dtb_call_stats;
DTB_API int dtb_last_call_stats(dtb_call_stats* out);

#ifdef __cplusplus
}
#endif
#endif /* DTB200_H */
