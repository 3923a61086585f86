// dtb_window.cu -- grouped cumulative and window functions: every row of the grouped frame keeps its place and gets
// a value that depends on the rows of its group before it (after it, under `reverse`).  The reference computes each
// one as a serial loop per group over the value column viewed through the RowIndex:
//
//   cumsum / cumprod      column/cumsumprod.h:48-95        NA counts as 0 / 1
//   cummin / cummax       column/cumminmax.h:48-110        NA skipped; a leading NA stays NA; ties -> current row
//   cumcount / ngroup     column/cumcountngroup.h:52-70    row number inside the group / group number
//   fillna                expr/fexpr_fillna.cc:86-118      last non-NA value so far
//   shift                 expr/head_func_shift.cc:41-62    value n rows earlier (n < 0: later) in the group, else NA
//
// Here the grouped frame is cut into tiles of WIN_TILE consecutive positions.  Every CTA finds the group of its
// tile's first and last positions by bisection of the offsets and walks the groups in between, so each row knows its
// group, the group's bounds and whether it is the group's head (its first row; its last row under `reverse`, where
// the tile maps positions from the end).  The scans read v[order[p]] with the gather fused in and run in three
// kernels, none of which waits on another CTA (the sort passes have the same rule, DESIGN.md 4.1):
//   1. win_scan_kernel   segmented scan inside the tile, written straight to `out`; the tile publishes the
//                        aggregate of its trailing open segment and the position of its first head
//   2. win_carry_kernel  one CTA: segmented scan over the tile aggregates = every tile's carry-in
//   3. win_fixup_kernel  the rows of a tile before its first head combine with the carry-in
// Bound: the random 8-byte gather v[order[p]] (one 32-byte sector per row), like gather_kernel.
#include <type_traits>
#include "dtb_common.cuh"

namespace dtb {

constexpr int WIN_THREADS = 256;
constexpr int WIN_IPT = 16;
constexpr int WIN_TILE = WIN_THREADS * WIN_IPT;               // 4096 positions
constexpr int CARRY_THREADS = 1024;

// ---- elements ----------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ bool is_valid(T x) {
  if constexpr (std::is_floating_point<T>::value) return !isnan(x);
  else return x != NaOf<T>::v();
}
template <typename T> __device__ __forceinline__ T na_of() {
  if constexpr (std::is_same<T, float>::value) return __int_as_float(0x7FC00000);
  else if constexpr (std::is_same<T, double>::value) return __longlong_as_double(0x7FF8000000000000ll);
  else return NaOf<T>::v();
}
template <typename A> __device__ __forceinline__ u64 to_bits(A a) {
  if constexpr (std::is_same<A, double>::value) return (u64)__double_as_longlong(a);
  else if constexpr (std::is_same<A, float>::value) return (u64)__float_as_uint(a);
  else return (u64)(typename std::make_unsigned<A>::type)a;
}
template <typename A> __device__ __forceinline__ A from_bits(u64 u) {
  if constexpr (std::is_same<A, double>::value) return __longlong_as_double((long long)u);
  else if constexpr (std::is_same<A, float>::value) return __uint_as_float((u32)u);
  else return (A)(typename std::make_unsigned<A>::type)u;
}

// ---- scan operators: Acc is the running state, combine(earlier, later) is associative -------------------
template <int OP, typename T> struct ScanOp;

// sum / product: integers (and bool) in uint64 (exact mod 2^64), floats in double, NA = the identity
template <int OP, typename T> struct SumProd {
  static constexpr bool F = std::is_floating_point<T>::value;
  typedef typename std::conditional<F, double, u64>::type Acc;
  typedef typename std::conditional<F, T, int64_t>::type Out;
  static __device__ __forceinline__ Acc identity() { return OP == DTB_WIN_CUMSUM ? (Acc)0 : (Acc)1; }
  static __device__ __forceinline__ Acc lift(T x) {
    if (!is_valid(x)) return identity();
    if constexpr (F) return (double)x; else return (u64)(int64_t)x;
  }
  static __device__ __forceinline__ Acc combine(Acc a, Acc b) { return OP == DTB_WIN_CUMSUM ? a + b : a * b; }
  static __device__ __forceinline__ Out store(Acc a) { return (Out)a; }
  static __device__ __forceinline__ Acc load(Out o) { return (Acc)o; }
  static __device__ __forceinline__ bool neutral(Acc) { return false; }
};
template <typename T> struct ScanOp<DTB_WIN_CUMSUM, T> : SumProd<DTB_WIN_CUMSUM, T> {};
template <typename T> struct ScanOp<DTB_WIN_CUMPROD, T> : SumProd<DTB_WIN_CUMPROD, T> {};

// min / max / last valid value: the stype itself, NA = "nothing yet".  Ties go to the later row
// (prev < val ? prev : val), which keeps the operator associative and the result bit-exact (+-0 included).
template <int OP, typename T> struct Select {
  typedef T Acc;
  typedef T Out;
  static __device__ __forceinline__ Acc identity() { return na_of<T>(); }
  static __device__ __forceinline__ Acc lift(T x) { return x; }
  static __device__ __forceinline__ Acc combine(Acc a, Acc b) {
    if (!is_valid(b)) return a;
    if (!is_valid(a) || OP == DTB_WIN_FILLNA) return b;
    if (OP == DTB_WIN_CUMMIN) return a < b ? a : b;
    return a > b ? a : b;
  }
  static __device__ __forceinline__ Out store(Acc a) { return a; }
  static __device__ __forceinline__ Acc load(Out o) { return o; }
  static __device__ __forceinline__ bool neutral(Acc a) { return !is_valid(a); }
};
template <typename T> struct ScanOp<DTB_WIN_CUMMIN, T> : Select<DTB_WIN_CUMMIN, T> {};
template <typename T> struct ScanOp<DTB_WIN_CUMMAX, T> : Select<DTB_WIN_CUMMAX, T> {};
template <typename T> struct ScanOp<DTB_WIN_FILLNA, T> : Select<DTB_WIN_FILLNA, T> {};

// segmented combine: (a, fa) then (b, fb) -- b restarts the segment when fb
template <typename Op>
__device__ __forceinline__ void seg_combine(typename Op::Acc& a, bool& fa, typename Op::Acc b, bool fb) {
  a = fb ? b : Op::combine(a, b);
  fa = fa || fb;
}

// ---- the tile walk -------------------------------------------------------------------------------------
// position of logical index q (reverse: counted from the end of the grouped frame)
template <bool REV> __device__ __forceinline__ int64_t pos_of(int64_t q, int64_t n) { return REV ? n - 1 - q : q; }

// largest g in [lo, hi] with offsets[g] <= p
__device__ __forceinline__ int64_t find_group(const int32_t* __restrict__ offsets, int64_t lo, int64_t hi, int64_t p) {
  hi += 1;
  while (hi - lo > 1) { const int64_t mid = (lo + hi) >> 1; if ((int64_t)offsets[mid] <= p) lo = mid; else hi = mid; }
  return lo;
}

// Groups of the tile's first and last positions (one bisection each over all groups); every thread then bisects
// only the few groups in between.
template <bool REV>
__device__ __forceinline__ void tile_groups(const int32_t* __restrict__ offsets, int64_t ng, int64_t n, int64_t q0,
                                            int64_t qlast, int64_t& lo, int64_t& hi) {
  __shared__ int64_t s_g[2];
  if (threadIdx.x == 0) s_g[0] = find_group(offsets, 0, ng - 1, pos_of<REV>(q0, n));
  if (threadIdx.x == 32) s_g[1] = find_group(offsets, 0, ng - 1, pos_of<REV>(qlast, n));
  __syncthreads();
  lo = REV ? s_g[1] : s_g[0];
  hi = REV ? s_g[0] : s_g[1];
}

// Exclusive segmented scan of one (acc, flag) per thread over the CTA; *total = inclusive result of the last thread.
template <typename Op, int NT>
__device__ __forceinline__ void block_seg_scan(typename Op::Acc acc, bool flag, typename Op::Acc& excl,
                                               typename Op::Acc& total, bool& total_flag) {
  typedef typename Op::Acc Acc;
  constexpr int NW = NT / 32;
  __shared__ u64 s_acc[NW];
  __shared__ int s_flag[NW];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  Acc inc = acc; bool f = flag;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const Acc o = from_bits<Acc>(__shfl_up_sync(0xFFFFFFFFu, to_bits(inc), d));
    const int of = __shfl_up_sync(0xFFFFFFFFu, (int)f, d);
    if (lane >= d) { if (!f) inc = Op::combine(o, inc); f = f || of; }
  }
  if (lane == 31) { s_acc[w] = to_bits(inc); s_flag[w] = f; }
  __syncthreads();
  Acc wp = Op::identity(); bool wf = false;                  // prefix of the warps before this one
  for (int k = 0; k < w; k++) seg_combine<Op>(wp, wf, from_bits<Acc>(s_acc[k]), s_flag[k] != 0);
  Acc le = from_bits<Acc>(__shfl_up_sync(0xFFFFFFFFu, to_bits(inc), 1));
  int lf = __shfl_up_sync(0xFFFFFFFFu, (int)f, 1);
  if (lane == 0) { le = Op::identity(); lf = 0; }
  Acc e = wp; bool ef = wf;
  seg_combine<Op>(e, ef, le, lf != 0);
  excl = e;
  Acc t = wp; bool tf = wf;
  seg_combine<Op>(t, tf, inc, f);
  total = t; total_flag = tf;
  __syncthreads();                                           // s_acc may be reused by the caller's next scan
}

// ===========================================================================
// 1. segmented scan inside every tile
// ===========================================================================
template <int OP, typename T, bool REV>
__global__ void __launch_bounds__(WIN_THREADS, 2)
win_scan_kernel(const T* __restrict__ v, int64_t nv, const int32_t* __restrict__ order,
                const int32_t* __restrict__ offsets, int64_t ng, int64_t n,
                typename ScanOp<OP, T>::Out* __restrict__ out, u64* __restrict__ tile_agg, int32_t* __restrict__ tile_head)
{
  typedef ScanOp<OP, T> Op;
  typedef typename Op::Acc Acc;
  __shared__ int s_head;
  const int64_t q0 = (int64_t)blockIdx.x * WIN_TILE;
  const int64_t qend = q0 + WIN_TILE < n ? q0 + WIN_TILE : n;
  if (threadIdx.x == 0) s_head = WIN_TILE;
  int64_t lo, hi;
  tile_groups<REV>(offsets, ng, n, q0, qend - 1, lo, hi);

  const int64_t qt = q0 + (int64_t)threadIdx.x * WIN_IPT;
  Acc val[WIN_IPT];
  unsigned heads = 0;
  {
    int64_t j[WIN_IPT];
    if (qt < qend) {
      int64_t p = pos_of<REV>(qt, n);
      int64_t g = find_group(offsets, lo, hi, p);
      int64_t gs = offsets[g], ge = offsets[g + 1];
#pragma unroll
      for (int i = 0; i < WIN_IPT; i++) {
        const int64_t q = qt + i;
        j[i] = -1;
        if (q < qend) {
          p = pos_of<REV>(q, n);
          if (REV) { while (p < gs) { g--; ge = gs; gs = offsets[g]; } }
          else     { while (p >= ge) { g++; gs = ge; ge = offsets[g + 1]; } }
          if (p == (REV ? ge - 1 : gs)) heads |= 1u << i;
          j[i] = order ? (int64_t)order[p] : p;
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < WIN_IPT; i++) j[i] = -1;
    }
#pragma unroll
    for (int i = 0; i < WIN_IPT; i++) val[i] = (j[i] >= 0 && j[i] < nv) ? Op::lift(v[j[i]]) : Op::identity();
  }
  // the thread's trailing open segment
  Acc agg = Op::identity();
#pragma unroll
  for (int i = 0; i < WIN_IPT; i++) agg = ((heads >> i) & 1) ? Op::combine(Op::identity(), val[i]) : Op::combine(agg, val[i]);
  if (heads) atomicMin(&s_head, (int)threadIdx.x * WIN_IPT + __ffs(heads) - 1);
  Acc run, total; bool total_flag;
  block_seg_scan<Op, WIN_THREADS>(agg, heads != 0, run, total, total_flag);
#pragma unroll
  for (int i = 0; i < WIN_IPT; i++) {
    run = Op::combine(((heads >> i) & 1) ? Op::identity() : run, val[i]);
    if (qt + i < qend) out[pos_of<REV>(qt + i, n)] = Op::store(run);
  }
  if (threadIdx.x == WIN_THREADS - 1) tile_agg[blockIdx.x] = to_bits(total);
  if (threadIdx.x == 0) tile_head[blockIdx.x] = s_head;     // s_head is final: block_seg_scan synchronised
}

// ===========================================================================
// 2. carry-in of every tile: exclusive segmented scan over the tile aggregates (one CTA)
// ===========================================================================
template <int OP, typename T>
__global__ void __launch_bounds__(CARRY_THREADS)
win_carry_kernel(const u64* __restrict__ tile_agg, const int32_t* __restrict__ tile_head, int64_t ntiles,
                 u64* __restrict__ carry)
{
  typedef ScanOp<OP, T> Op;
  typedef typename Op::Acc Acc;
  const int64_t per = (ntiles + CARRY_THREADS - 1) / CARRY_THREADS;
  const int64_t t0 = (int64_t)threadIdx.x * per, t1 = t0 + per < ntiles ? t0 + per : ntiles;
  Acc a = Op::identity(); bool f = false;
  for (int64_t t = t0; t < t1; t++) seg_combine<Op>(a, f, from_bits<Acc>(tile_agg[t]), tile_head[t] < WIN_TILE);
  Acc c, total; bool tf;
  block_seg_scan<Op, CARRY_THREADS>(a, f, c, total, tf);
  bool cf = false;
  for (int64_t t = t0; t < t1; t++) {
    carry[t] = to_bits(c);
    seg_combine<Op>(c, cf, from_bits<Acc>(tile_agg[t]), tile_head[t] < WIN_TILE);
  }
}

// ===========================================================================
// 3. rows before the first head of every tile: out = carry-in (+) out
// ===========================================================================
template <int OP, typename T, bool REV>
__global__ void __launch_bounds__(WIN_THREADS)
win_fixup_kernel(const u64* __restrict__ carry, const int32_t* __restrict__ tile_head, int64_t n,
                 typename ScanOp<OP, T>::Out* __restrict__ out)
{
  typedef ScanOp<OP, T> Op;
  typedef typename Op::Acc Acc;
  const int64_t b = blockIdx.x;
  const int h = tile_head[b];
  if (b == 0 || h == 0) return;
  const Acc c = from_bits<Acc>(carry[b]);
  if (Op::neutral(c)) return;
  const int64_t q0 = b * WIN_TILE;
  const int64_t qe = q0 + h < n ? q0 + h : n;
  for (int64_t q = q0 + threadIdx.x; q < qe; q += WIN_THREADS) {
    const int64_t p = pos_of<REV>(q, n);
    out[p] = Op::store(Op::combine(c, Op::load(out[p])));
  }
}

template <int OP, typename T>
static int run_scan(const void* v, int64_t nv, const int32_t* order, const int32_t* offsets, int64_t ng, int64_t n,
                    bool rev, void* out, void* scratch, cudaStream_t s)
{
  typedef typename ScanOp<OP, T>::Out Out;
  const int64_t ntiles = (n + WIN_TILE - 1) / WIN_TILE;
  u64* agg = (u64*)scratch;
  u64* carry = agg + ntiles;
  int32_t* head = (int32_t*)(carry + ntiles);
  prof_begin("window_scan", s);
  if (rev) win_scan_kernel<OP, T, true><<<(unsigned)ntiles, WIN_THREADS, 0, s>>>((const T*)v, nv, order, offsets, ng, n, (Out*)out, agg, head);
  else     win_scan_kernel<OP, T, false><<<(unsigned)ntiles, WIN_THREADS, 0, s>>>((const T*)v, nv, order, offsets, ng, n, (Out*)out, agg, head);
  prof_end(s);
  count_launch();
  if (ntiles > 1) {
    prof_begin("window_carry", s);
    win_carry_kernel<OP, T><<<1, CARRY_THREADS, 0, s>>>(agg, head, ntiles, carry);
    prof_end(s);
    prof_begin("window_fixup", s);
    if (rev) win_fixup_kernel<OP, T, true><<<(unsigned)ntiles, WIN_THREADS, 0, s>>>(carry, head, n, (Out*)out);
    else     win_fixup_kernel<OP, T, false><<<(unsigned)ntiles, WIN_THREADS, 0, s>>>(carry, head, n, (Out*)out);
    prof_end(s);
    count_launch(2);
  }
  DTB_CUDA_CHECK(cudaGetLastError());
  return DTB_OK;
}

// ===========================================================================
// elementwise ops on the same walk: cumcount, ngroup (int64, no value read), shift (raw element copy)
// ===========================================================================
template <int OP, typename E>
__global__ void __launch_bounds__(WIN_THREADS)
win_elem_kernel(const E* __restrict__ v, int64_t nv, const int32_t* __restrict__ order,
                const int32_t* __restrict__ offsets, int64_t ng, int64_t n, int64_t param, E na, void* __restrict__ out)
{
  const int64_t q0 = (int64_t)blockIdx.x * WIN_TILE;
  const int64_t qend = q0 + WIN_TILE < n ? q0 + WIN_TILE : n;
  int64_t lo, hi;
  tile_groups<false>(offsets, ng, n, q0, qend - 1, lo, hi);
  const int64_t qt = q0 + (int64_t)threadIdx.x * WIN_IPT;
  if (qt >= qend) return;
  int64_t g = find_group(offsets, lo, hi, qt);
  int64_t gs = offsets[g], ge = offsets[g + 1];
  if (OP == DTB_WIN_SHIFT) {
    int64_t j[WIN_IPT];
#pragma unroll
    for (int i = 0; i < WIN_IPT; i++) {
      const int64_t p = qt + i;
      j[i] = -1;
      if (p < qend) {
        while (p >= ge) { g++; gs = ge; ge = offsets[g + 1]; }
        const int64_t src = p - param;
        if (src >= gs && src < ge) j[i] = order ? (int64_t)order[src] : src;
      }
    }
#pragma unroll
    for (int i = 0; i < WIN_IPT; i++)
      if (qt + i < qend) ((E*)out)[qt + i] = (j[i] >= 0 && j[i] < nv) ? v[j[i]] : na;
  } else {
#pragma unroll
    for (int i = 0; i < WIN_IPT; i++) {
      const int64_t p = qt + i;
      if (p < qend) {
        while (p >= ge) { g++; gs = ge; ge = offsets[g + 1]; }
        int64_t r;
        if (OP == DTB_WIN_CUMCOUNT) r = param ? ge - 1 - p : p - gs;
        else                        r = param ? ng - 1 - g : g;
        ((int64_t*)out)[p] = r;
      }
    }
  }
}

template <int OP, typename E>
static int run_elem(const void* v, int64_t nv, const int32_t* order, const int32_t* offsets, int64_t ng, int64_t n,
                    int64_t param, E na, void* out, cudaStream_t s)
{
  const int64_t ntiles = (n + WIN_TILE - 1) / WIN_TILE;
  prof_begin(OP == DTB_WIN_SHIFT ? "window_shift" : "window_count", s);
  win_elem_kernel<OP, E><<<(unsigned)ntiles, WIN_THREADS, 0, s>>>((const E*)v, nv, order, offsets, ng, n, param, na, out);
  prof_end(s);
  count_launch();
  DTB_CUDA_CHECK(cudaGetLastError());
  return DTB_OK;
}

size_t window_scratch_bytes(int64_t n) {
  const int64_t ntiles = (n + WIN_TILE - 1) / WIN_TILE;
  return (size_t)ntiles * (2 * sizeof(u64) + sizeof(int32_t));
}

int window_out_stype_host(int op, int stype) {
  const bool known = stype_bytes(stype) != 0;
  switch (op) {
    case DTB_WIN_CUMCOUNT: case DTB_WIN_NGROUP:
      return DTB_STYPE_INT64;
    case DTB_WIN_CUMSUM: case DTB_WIN_CUMPROD:
      if (stype == DTB_STYPE_FLOAT32 || stype == DTB_STYPE_FLOAT64) return stype;
      if (stype == DTB_STYPE_BOOL || (stype >= DTB_STYPE_INT8 && stype <= DTB_STYPE_INT64)) return DTB_STYPE_INT64;
      return 0;                                           // date32 / time64: TypeError (fexpr_cumsumprod.cc)
    case DTB_WIN_CUMMIN: case DTB_WIN_CUMMAX: case DTB_WIN_FILLNA: case DTB_WIN_SHIFT:
      return known ? stype : 0;
  }
  return 0;
}

#define DTB_WIN_DISPATCH(st, CALL)                                             \
  switch (st) {                                                                \
    case DTB_STYPE_BOOL: case DTB_STYPE_INT8:    return CALL(int8_t);          \
    case DTB_STYPE_INT16:                        return CALL(int16_t);         \
    case DTB_STYPE_INT32: case DTB_STYPE_DATE32: return CALL(int32_t);         \
    case DTB_STYPE_INT64: case DTB_STYPE_TIME64: return CALL(int64_t);         \
    case DTB_STYPE_FLOAT32:                      return CALL(float);           \
    case DTB_STYPE_FLOAT64:                      return CALL(double);          \
  }

int launch_window(int op, int64_t param, const void* v, int stype, int64_t nv, const int32_t* order,
                  const int32_t* offsets, int64_t ng, int64_t n, void* out, void* scratch, cudaStream_t s)
{
  if (n == 0 || ng == 0) return DTB_OK;
  const bool rev = param != 0;
  switch (op) {
#define WIN_SCAN_CALL(OPC, T) run_scan<OPC, T>(v, nv, order, offsets, ng, n, rev, out, scratch, s)
    case DTB_WIN_CUMSUM: {
#define C(T) WIN_SCAN_CALL(DTB_WIN_CUMSUM, T)
      DTB_WIN_DISPATCH(stype, C)
#undef C
      break;
    }
    case DTB_WIN_CUMPROD: {
#define C(T) WIN_SCAN_CALL(DTB_WIN_CUMPROD, T)
      DTB_WIN_DISPATCH(stype, C)
#undef C
      break;
    }
    case DTB_WIN_CUMMIN: {
#define C(T) WIN_SCAN_CALL(DTB_WIN_CUMMIN, T)
      DTB_WIN_DISPATCH(stype, C)
#undef C
      break;
    }
    case DTB_WIN_CUMMAX: {
#define C(T) WIN_SCAN_CALL(DTB_WIN_CUMMAX, T)
      DTB_WIN_DISPATCH(stype, C)
#undef C
      break;
    }
    case DTB_WIN_FILLNA: {
#define C(T) WIN_SCAN_CALL(DTB_WIN_FILLNA, T)
      DTB_WIN_DISPATCH(stype, C)
#undef C
      break;
    }
#undef WIN_SCAN_CALL
    case DTB_WIN_CUMCOUNT:
      return run_elem<DTB_WIN_CUMCOUNT, uint8_t>(nullptr, 0, order, offsets, ng, n, param, 0, out, s);
    case DTB_WIN_NGROUP:
      return run_elem<DTB_WIN_NGROUP, uint8_t>(nullptr, 0, order, offsets, ng, n, param, 0, out, s);
    case DTB_WIN_SHIFT:
      switch (stype_bytes(stype)) {
        case 1: return run_elem<DTB_WIN_SHIFT, uint8_t>(v, nv, order, offsets, ng, n, param, (uint8_t)0x80, out, s);
        case 2: return run_elem<DTB_WIN_SHIFT, uint16_t>(v, nv, order, offsets, ng, n, param, (uint16_t)0x8000, out, s);
        case 4: return run_elem<DTB_WIN_SHIFT, u32>(v, nv, order, offsets, ng, n, param,
                                                    stype == DTB_STYPE_FLOAT32 ? 0x7FC00000u : 0x80000000u, out, s);
        case 8: return run_elem<DTB_WIN_SHIFT, u64>(v, nv, order, offsets, ng, n, param,
                                                    stype == DTB_STYPE_FLOAT64 ? 0x7FF8000000000000ull : 0x8000000000000000ull, out, s);
      }
      break;
  }
  set_error("window op " + std::to_string(op) + " is not defined for stype " + std::to_string(stype));
  return DTB_EINVAL;
}

}  // namespace dtb
