// dtb_api.cu -- the C-ABI (include/dtb200.h): call planning, HBM scratch,
// host<->device staging and error reporting.  No compute happens on the host:
// without a CUDA device every entry point fails with DTB_ECUDA.
#include <stdio.h>
#include <chrono>
#include <string.h>
#include <list>
#include <mutex>
#include <string>
#include <vector>
#include "dtb_common.cuh"

namespace dtb {

// ---------------------------------------------------------------------------
// thread-local state
// ---------------------------------------------------------------------------
static thread_local std::string t_error;
static thread_local dtb_call_stats t_stats = {0, 0, 0, 0, 0};

void set_error(const std::string& msg) { t_error = msg; }
void count_launch(int n) { t_stats.kernels_launched += n; }

// ---------------------------------------------------------------------------
// options (analogue of dt.options.sort.*, sort.cc:259-349)
// ---------------------------------------------------------------------------
static int64_t opt_radix_bits = 0;     // 0 = default (8-bit digits); 4..8 = largest digit width
static int64_t opt_verbose = 0;
static int64_t opt_profile = 0;
static thread_local int opt_trust_offsets = 0;  // internal: dtb_groupby_reduce passes the handle's own offsets to dtb_reduce
static int64_t opt_fuse_hist = 1;      // 1 = single-column keys: statistics and the first pass's histogram from one read of the column
static int64_t opt_stage_keys = 0;     // 1 = the first count kernel also materialises the normalised keys of a raw key column (round-1 behaviour)
static int64_t opt_bucketed = 1;       // 1 = columns with >= 2 L2 atomics per row take the bucketed multi-reducer (dtb_bucket.cu)
static int64_t opt_overlap = 0;        // 1 = run fused direct reducers on a side stream under the sort passes

// ---------------------------------------------------------------------------
// optional per-kernel timing with CUDA events on the launching stream
// (option "profile"): the reference only times whole calls (call_logger.cc:153-174)
// ---------------------------------------------------------------------------
struct ProfRec { const char* name; cudaEvent_t a, b; };
static thread_local std::vector<ProfRec> t_prof_open;
static thread_local std::vector<std::pair<std::string, double>> t_prof_done;

struct ProfScope {
  bool on; cudaStream_t s; ProfRec r;
  ProfScope(const char* name, cudaStream_t stream) : on(opt_profile != 0), s(stream) {
    if (!on) return;
    r.name = name;
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    cudaEventRecord(r.a, s);
  }
  ~ProfScope() { if (on) { cudaEventRecord(r.b, s); t_prof_open.push_back(r); } }
};

static thread_local ProfRec t_prof_cur;
static thread_local bool t_prof_cur_on = false;
void prof_begin(const char* name, cudaStream_t s) {
  if (!opt_profile) return;
  t_prof_cur.name = name;
  cudaEventCreate(&t_prof_cur.a); cudaEventCreate(&t_prof_cur.b);
  cudaEventRecord(t_prof_cur.a, s);
  t_prof_cur_on = true;
}
void prof_end(cudaStream_t s) {
  if (!t_prof_cur_on) return;
  cudaEventRecord(t_prof_cur.b, s);
  t_prof_open.push_back(t_prof_cur);
  t_prof_cur_on = false;
}

// Lazy: the calls only record events; the first query (dtb_profile_count / _reset) waits for them.  (A sync at the
// end of every profiled call kept the host from running ahead and cost ~0.4 ms per C2 step in bench.py's timed region.)
static void prof_collect() {
  for (auto& r : t_prof_open) {
    float ms = 0.f;
    if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess)
      t_prof_done.emplace_back(r.name, (double)ms);
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  t_prof_open.clear();
}

// ---------------------------------------------------------------------------
// per-device context: the stream-ordered memory pool keeps scratch resident
// ---------------------------------------------------------------------------
static std::mutex g_ctx_mutex;
static bool g_ctx_ready[64] = {false};

static double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
#define DTB_TL(label) do { if (opt_verbose >= 2) fprintf(stderr, "[dtb200]   t=%9.3f ms  %s\n", now_ms() - tl0, label); } while (0)

// Waits for the stream by polling.  cudaStreamSynchronize parks the thread (the context is usually created by the
// host framework with the default scheduling policy) and wakes it 50-100 us after the stream drained; group() has
// two such waits on its critical path (the statistics, the number of groups) with the GPU idle behind them.
static cudaError_t stream_wait(cudaStream_t s) {
  cudaError_t e;
  while ((e = cudaStreamQuery(s)) == cudaErrorNotReady) {}
  return e;
}

static int ensure_context() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    set_error(std::string("no usable CUDA device: ") + cudaGetErrorString(e));
    return DTB_ECUDA;
  }
  if (dev < 0 || dev >= 64) { set_error("device ordinal out of range"); return DTB_EINVAL; }
  if (g_ctx_ready[dev]) return DTB_OK;
  std::lock_guard<std::mutex> lock(g_ctx_mutex);
  if (g_ctx_ready[dev]) return DTB_OK;
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) {
    set_error(std::string("no usable CUDA device: ") + cudaGetErrorString(e));
    return DTB_ECUDA;
  }
  if (prop.major != 10) {
    set_error("dtb200 is built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) +
              std::to_string(prop.minor));
    return DTB_ECUDA;
  }
  cudaMemPool_t pool;
  DTB_CUDA_CHECK(cudaDeviceGetDefaultMemPool(&pool, dev));
  uint64_t thresh = UINT64_MAX;          // keep freed scratch cached in the pool
  DTB_CUDA_CHECK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thresh));
  g_ctx_ready[dev] = true;
  return DTB_OK;
}

// ---------------------------------------------------------------------------
// Scratch arena.  Every API call carves its temporaries out of one HBM slab that the
// calling thread keeps between calls: after the first call of a given size there are
// no allocator calls at all on the hot path (cudaMallocAsync of multi-GB blocks costs
// milliseconds even when the pool already holds the memory).  The slab only grows.
// ---------------------------------------------------------------------------
struct Arena {
  struct Slab { char* p; size_t cap; };
  std::vector<Slab> slabs;
  size_t cur = 0, off = 0;
  int depth = 0;
  int device = -1;              // the slabs (and last_stream) belong to this device
  cudaStream_t last_stream = nullptr;
  bool have_last = false;

  int begin(cudaStream_t s) {
    if (depth++ > 0) return DTB_OK;
    // A thread may move between devices (dtb_init(d) / cudaSetDevice): scratch carved out of another
    // device's slab would be an illegal address, so the arena follows the thread's current device and
    // gives the old device's slabs back first.
    int dev = 0;
    DTB_CUDA_CHECK(cudaGetDevice(&dev));
    if (device != dev) {
      if (device >= 0 && (!slabs.empty() || have_last)) {
        DTB_CUDA_CHECK(cudaSetDevice(device));
        trim();
        DTB_CUDA_CHECK(cudaSetDevice(dev));
      }
      device = dev; have_last = false; last_stream = nullptr;
    }
    // work enqueued by the previous call may still be using the slab on another stream
    if (have_last && last_stream != s) DTB_CUDA_CHECK(cudaStreamSynchronize(last_stream));
    last_stream = s; have_last = true;
    if (slabs.size() > 1) {                         // coalesce what the last call needed into one slab
      size_t total = 0;
      for (auto& sl : slabs) total += sl.cap;
      DTB_CUDA_CHECK(cudaDeviceSynchronize());
      for (auto& sl : slabs) cudaFree(sl.p);
      slabs.clear();
      char* p = nullptr;
      cudaError_t e = cudaMalloc(&p, total);
      if (e != cudaSuccess) { cudaGetLastError(); }   // fall back to growing on demand
      else slabs.push_back({p, total});
    }
    cur = 0; off = 0;
    return DTB_OK;
  }
  void end() { if (depth > 0) depth--; }
  int take(size_t bytes, void** out) {
    bytes = (bytes + 255) & ~(size_t)255;
    while (cur < slabs.size()) {
      if (off + bytes <= slabs[cur].cap) { *out = slabs[cur].p + off; off += bytes; return DTB_OK; }
      cur++; off = 0;
    }
    size_t cap = bytes < ((size_t)64 << 20) ? ((size_t)64 << 20) : bytes;
    char* p = nullptr;
    cudaError_t e = cudaMalloc(&p, cap);
    if (e != cudaSuccess) {
      set_error("cudaMalloc(" + std::to_string(cap) + " bytes): " + cudaGetErrorString(e));
      cudaGetLastError();
      return e == cudaErrorMemoryAllocation ? DTB_ENOMEM : DTB_ECUDA;
    }
    slabs.push_back({p, cap});
    cur = slabs.size() - 1; off = bytes;
    *out = p;
    return DTB_OK;
  }
  void trim() {
    cudaDeviceSynchronize();
    for (auto& sl : slabs) cudaFree(sl.p);
    slabs.clear(); cur = 0; off = 0;
  }
};
static thread_local Arena t_arena;

struct ArenaScope {
  int rc;
  explicit ArenaScope(cudaStream_t s) { rc = t_arena.begin(s); }
  ~ArenaScope() { t_arena.end(); }
};

// Device buffer: arena scratch by default (lives until the end of the API call), or an owned
// stream-ordered allocation for results that outlive the call (RowIndex / offsets of a handle).
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  cudaStream_t s = nullptr;
  bool owned = false;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  int alloc(size_t nbytes, cudaStream_t stream) {
    release();
    s = stream; bytes = nbytes ? nbytes : 16; owned = false;
    t_stats.scratch_bytes += (int64_t)bytes;
    return t_arena.take(bytes, &p);
  }
  int alloc_owned(size_t nbytes, cudaStream_t stream) {
    release();
    s = stream; bytes = nbytes ? nbytes : 16; owned = true;
    cudaError_t e = cudaMallocAsync(&p, bytes, s);
    if (e != cudaSuccess) {
      p = nullptr;
      set_error("cudaMallocAsync(" + std::to_string(bytes) + " bytes): " + cudaGetErrorString(e));
      cudaGetLastError();
      return e == cudaErrorMemoryAllocation ? DTB_ENOMEM : DTB_ECUDA;
    }
    return DTB_OK;
  }
  void release() { if (p && owned) cudaFreeAsync(p, s); p = nullptr; }
  void* detach() { void* q = p; p = nullptr; return q; }
  template <typename T> T* as() { return reinterpret_cast<T*>(p); }
};

static bool is_device_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// Host inputs kept resident in HBM between the calls of one query (dtb_cache_begin / dtb_cache_end): the
// reference-side hook calls dtb_group on the key columns and then dtb_reduce / dtb_gather on the value
// columns and on the RowIndex it just received, all inside one EvalContext::evaluate(); without the cache
// every call uploads its host buffers again.  Entries are keyed by (host pointer, bytes) and are only valid
// while the caller guarantees the host buffers do not change -- the bracket is the caller's promise.
struct InputCache {
  struct Entry { const void* host; size_t bytes; void* dev; int device; };
  std::vector<Entry> entries;
  int depth = 0;
  void* find(const void* p, size_t bytes, int dev) const {
    for (const Entry& e : entries) if (e.host == p && e.bytes == bytes && e.device == dev) return e.dev;
    return nullptr;
  }
  void clear() {
    for (Entry& e : entries) { int cur = 0; cudaGetDevice(&cur); if (cur != e.device) cudaSetDevice(e.device); cudaFree(e.dev); if (cur != e.device) cudaSetDevice(cur); }
    entries.clear();
  }
};
static thread_local InputCache t_cache;

// Input that may live on the host: staged into HBM when needed.
struct DevIn {
  const void* dptr = nullptr;
  DevBuf buf;
  int bind(const void* p, size_t bytes, cudaStream_t s) {
    if (!p || bytes == 0) { dptr = p; return DTB_OK; }
    if (is_device_ptr(p)) { dptr = p; return DTB_OK; }
    if (t_cache.depth > 0) {
      int dev = 0; DTB_CUDA_CHECK(cudaGetDevice(&dev));
      if (void* d = t_cache.find(p, bytes, dev)) { dptr = d; t_stats.cache_hits += 1; return DTB_OK; }
      void* d = nullptr;
      cudaError_t e = cudaMalloc(&d, bytes);
      if (e == cudaSuccess) {
        DTB_CUDA_CHECK(cudaMemcpyAsync(d, p, bytes, cudaMemcpyHostToDevice, s));
        t_cache.entries.push_back({p, bytes, d, dev});
        dptr = d;
        return DTB_OK;
      }
      cudaGetLastError();                           // no room to keep it: stage it for this call only
    }
    DTB_TRY(buf.alloc(bytes, s));
    DTB_CUDA_CHECK(cudaMemcpyAsync(buf.p, p, bytes, cudaMemcpyHostToDevice, s));
    dptr = buf.p;
    return DTB_OK;
  }
};

// Output that may live on the host: computed in HBM, copied back by finish().
struct DevOut {
  void* dptr = nullptr;
  void* host = nullptr;
  size_t bytes = 0;
  DevBuf buf;
  int bind(void* p, size_t nbytes, cudaStream_t s) {
    bytes = nbytes;
    if (!p) { dptr = nullptr; return DTB_OK; }
    if (is_device_ptr(p)) { dptr = p; return DTB_OK; }
    host = p;
    DTB_TRY(buf.alloc(nbytes, s));
    dptr = buf.p;
    return DTB_OK;
  }
  bool staged() const { return host != nullptr; }
  int finish(size_t nbytes, cudaStream_t s) {
    if (host && nbytes) DTB_CUDA_CHECK(cudaMemcpyAsync(host, dptr, nbytes, cudaMemcpyDeviceToHost, s));
    return DTB_OK;
  }
  // inside a cache bracket: keep a device copy of a result that went to the host (the hook hands the RowIndex
  // of dtb_group straight back to dtb_reduce / dtb_gather)
  static void remember(const void* host_ptr, const void* dev_src, size_t nbytes, cudaStream_t s) {
    if (t_cache.depth <= 0 || !host_ptr || !nbytes) return;
    int dev = 0; if (cudaGetDevice(&dev) != cudaSuccess) return;
    if (t_cache.find(host_ptr, nbytes, dev)) return;
    void* d = nullptr;
    if (cudaMalloc(&d, nbytes) != cudaSuccess) { cudaGetLastError(); return; }
    if (cudaMemcpyAsync(d, dev_src, nbytes, cudaMemcpyDeviceToDevice, s) != cudaSuccess) { cudaGetLastError(); cudaFree(d); return; }
    t_cache.entries.push_back({host_ptr, nbytes, d, dev});
  }
};

static int bitlen(u64 v) { int b = 0; while (v) { b++; v >>= 1; } return b; }
static int ctz64(u64 v) { int c = 0; while (!(v & 1)) { v >>= 1; c++; } return c; }

static bool stype_supported(int st) { return stype_bytes(st) != 0; }

// ---------------------------------------------------------------------------
// group(): plan + launch
// ---------------------------------------------------------------------------
// Reducers evaluated inside the group() call (dtb_groupby_create_reduce).
struct FusedReducers {
  const dtb_reduce_spec* spec = nullptr;
  int n = 0;
  std::vector<void*> out;       // owned device buffers, ngroups elements each
};

// Side stream on which the direct-address reducers run while the sort passes occupy `s`.
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  int device = -1;
  int ensure() {
    int dev = 0;
    DTB_CUDA_CHECK(cudaGetDevice(&dev));
    if (stream && device != dev) {               // the thread moved to another device: new stream there
      cudaSetDevice(device);
      cudaStreamDestroy(stream); cudaEventDestroy(fork); cudaEventDestroy(join);
      cudaSetDevice(dev);
      stream = nullptr;
    }
    device = dev;
    if (stream) return DTB_OK;
    int lo = 0, hi = 0;
    DTB_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    DTB_CUDA_CHECK(cudaStreamCreateWithPriority(&stream, cudaStreamNonBlocking, hi));
    DTB_CUDA_CHECK(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
    DTB_CUDA_CHECK(cudaEventCreateWithFlags(&join, cudaEventDisableTiming));
    return DTB_OK;
  }
};
static thread_local SideStream t_side;

struct GroupResult {
  DevBuf order;          // int32[n]
  DevBuf offsets;        // int32[ng+1] (capacity n+1) when groups were requested
  int64_t n = 0;
  int64_t nskip = 0;     // leading NA rows to drop (na_position = remove)
  int64_t ngroups = -1;
  // direct-address reducer support (small key domains, device-resident key columns)
  bool    direct = false;
  int64_t direct_gmax = 0;   // rows of the largest group
  KeyPlan direct_kp;
  int64_t direct_table = 0;
  DevBuf  gkeys;         // uint32[ngroups]
};

// Builds the per-column normalisation from device-computed stats.
static int plan_keys(const dtb_col* keys, const void* const* dptrs, int nkeys, const int* flags,
                     int na_pos, const ColStats* st, KeyPlan& kp, int64_t& nacount_last)
{
  kp.nkeys = nkeys;
  int total = 0;
  // the last key is the least significant part of the composite
  for (int c = nkeys - 1; c >= 0; c--) {
    KeyNorm& k = kp.k[c];
    const ColStats& cs = st[c];
    k.data = dptrs[c];
    k.stype = keys[c].stype;
    k.desc = (flags[c] & DTB_FLAG_DESCENDING) ? 1 : 0;
    k.pad = 0;
    u64 lo = cs.lo, hi = cs.hi;
    if (cs.nvalid == 0) { lo = hi = 0; }
    const u64 vary = cs.nvalid ? (cs.bits_or ^ cs.bits_and) : 0;
    k.cshift = vary ? ctz64(vary) : 0;
    const u64 rng = (hi - lo) >> k.cshift;                 // values span 0..rng after the shift
    k.edge = k.desc ? hi : lo;
    if (cs.nacount == 0) {                                 // no NA slot needed
      k.inc = 0; k.na_value = 0; k.bits = bitlen(rng);
    } else if (na_pos == DTB_NA_LAST) {                    // sort.cc:749-751: NA -> max-min+1, increment 0
      k.inc = 0; k.na_value = rng + 1; k.bits = bitlen(rng + 1);
    } else {                                               // NA -> 0, values shifted up by one
      k.inc = 1; k.na_value = 0; k.bits = bitlen(rng + 1);
    }
    if (cs.nvalid == 0) { k.bits = 0; k.na_value = 0; }    // all-NA column is constant
    k.lshift = total;
    total += k.bits;
    if (c == nkeys - 1) nacount_last = (int64_t)cs.nacount;
  }
  kp.total_bits = total;
  // groups are defined by the leading by-columns only (sort.cc:1471-1482)
  int gs = 0;
  for (int c = nkeys - 1; c >= 0 && (flags[c] & DTB_FLAG_SORT_ONLY); c--) gs = kp.k[c].lshift + kp.k[c].bits;
  kp.group_shift = gs;
  return DTB_OK;
}

static void plan_passes(int total_bits, int width, PassPlan& pp) {
  int np = (total_bits + width - 1) / width;
  if (np < 1) np = 1;
  pp.npasses = np;
  int base = total_bits / np, extra = total_bits % np, sh = 0;
  for (int p = 0; p < np; p++) {
    int b = base + (p < extra ? 1 : 0);
    if (b < 1) b = 1;
    pp.shift[p] = sh; pp.bits[p] = b; sh += b;
  }
}

static int group_core(const dtb_col* keys, int nkeys, const int* flags, int na_pos, int64_t n,
                      cudaStream_t s, int32_t* order_dev /*optional caller buffer*/,
                      int32_t* offsets_dev /*optional caller buffer, n+1*/, GroupResult& res,
                      bool want_direct = false, FusedReducers* fr = nullptr, bool wide = false)
{
  // wide == dtb_group64: up to 2^32 - 1 rows.  The passes carry row ids and output slots as 32-bit words
  // whose arithmetic is unsigned throughout, so ids >= 2^31 are just bit patterns in the int32 buffers;
  // the caller zero-extends order / offsets to int64 (ARR64, rowindex_array.cc:50-60).
  // want_direct == the handle path: the RowIndex outlives the call and must be an owned allocation
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  const double tl0 = now_ms();
  if (nkeys < 1 || nkeys > MAX_KEYS) { set_error("number of key columns must be in 1.." + std::to_string(MAX_KEYS)); return DTB_EINVAL; }
  if (!keys || !flags) { set_error("keys/flags must not be NULL"); return DTB_EINVAL; }
  if (na_pos < DTB_NA_FIRST || na_pos > DTB_NA_REMOVE) { set_error("na position value is not supported"); return DTB_EINVAL; }
  if (n < 0) { set_error("nrows must be non-negative"); return DTB_EINVAL; }
  for (int c = 0; c < nkeys; c++) {
    if (!stype_supported(keys[c].stype)) {
      set_error("Unable to sort Column of stype " + std::to_string(keys[c].stype));   // sort.cc:673
      return DTB_ENOTIMPL;
    }
    if (n > 0 && !keys[c].data) { set_error("key column data is NULL"); return DTB_EINVAL; }
  }
  if (n > (int64_t)INT32_MAX && !wide) { set_error("nrows > INT32_MAX needs an ARR64 RowIndex: use dtb_group64"); return DTB_ENOTIMPL; }
  if (n > (int64_t)0xFFFFFFFFll - 65536) { set_error("nrows >= 2^32 is beyond one GPU's passes (32-bit output slots): partition the frame"); return DTB_ENOTIMPL; }
  if (wide && (want_direct || fr)) { set_error("internal: the ARR64 path has no fused reducers"); return DTB_EINVAL; }
  DTB_TRY(ensure_context());

  const bool do_groups = !(flags[0] & DTB_FLAG_SORT_ONLY);
  res.n = n; res.nskip = 0; res.ngroups = do_groups ? 0 : -1;

  int32_t* order = order_dev;
  if (!order) {
    if (want_direct) DTB_TRY(res.order.alloc_owned(sizeof(int32_t) * (size_t)n, s));
    else             DTB_TRY(res.order.alloc(sizeof(int32_t) * (size_t)n, s));
    order = res.order.as<int32_t>();
  }
  int32_t* offsets = offsets_dev;
  if (do_groups && !offsets) {
    DTB_TRY(res.offsets.alloc(sizeof(int32_t) * (size_t)(n + 1), s)); offsets = res.offsets.as<int32_t>();
  }

  if (n == 0) {                                           // sort.cc:1431-1434
    if (do_groups) DTB_CUDA_CHECK(cudaMemsetAsync(offsets, 0, sizeof(int32_t), s));
    res.ngroups = do_groups ? 0 : -1;
    return DTB_OK;
  }

  // ---- stage host inputs, column statistics -------------------------------------
  std::vector<DevIn> in(nkeys);
  const void* dptrs[MAX_KEYS];
  for (int c = 0; c < nkeys; c++) {
    DTB_TRY(in[c].bind(keys[c].data, (size_t)n * stype_bytes(keys[c].stype), s));
    dptrs[c] = in[c].dptr;
  }
  DevBuf d_stats; DTB_TRY(d_stats.alloc(sizeof(ColStats) * nkeys, s));
  // single key column: the statistics kernel also counts the low 8 bits of every tile, which becomes the first
  // pass's histogram once edge / inc are known (no count kernel, one read of the column less)
  const bool fuse_hist = nkeys == 1 && opt_fuse_hist && !opt_stage_keys;
  DevBuf rawhist, rawna;
  if (fuse_hist) {
    DTB_TRY(rawhist.alloc(stats_hist_bytes(n), s));
    DTB_TRY(rawna.alloc(stats_na_bytes(n), s));
    ProfScope ps("col_stats", s);
    DTB_TRY(launch_col_stats_hist(dptrs[0], keys[0].stype, n, d_stats.as<ColStats>(), rawhist.as<unsigned short>(),
                                  rawna.as<unsigned short>(), s));
  } else for (int c = 0; c < nkeys; c++) {
    ProfScope ps("col_stats", s);
    DTB_TRY(launch_col_stats(dptrs[c], keys[c].stype, n, d_stats.as<ColStats>() + c, s));
  }
  ColStats h_stats[MAX_KEYS];
  DTB_CUDA_CHECK(cudaMemcpyAsync(h_stats, d_stats.p, sizeof(ColStats) * nkeys, cudaMemcpyDeviceToHost, s));
  DTB_CUDA_CHECK(stream_wait(s));

  DTB_TL("stats synced");
  KeyPlan kp; memset(&kp, 0, sizeof(kp));
  int64_t nacount_last = 0;
  DTB_TRY(plan_keys(keys, dptrs, nkeys, flags, na_pos, h_stats, kp, nacount_last));
  if (na_pos == DTB_NA_REMOVE) res.nskip = nacount_last;   // sort.cc:598-605
  t_stats.key_bits = kp.total_bits;
  if (kp.total_bits == 0) {
    // every key column is constant: identity order, one group (cf. sort.cc:1435-1439)
    DTB_TRY(launch_iota32(order, n, s));
    if (do_groups) {
      int32_t h[2] = {0, (int32_t)n};
      DTB_CUDA_CHECK(cudaMemcpyAsync(offsets, h, sizeof(h), cudaMemcpyHostToDevice, s));
      DTB_CUDA_CHECK(cudaStreamSynchronize(s));
      res.ngroups = 1;
    }
    return DTB_OK;
  }

  // by-columns that are all constant (0 bits) while sort columns vary: one group, and no kernel may
  // shift a key by its full width (composite >> group_shift with group_shift == key width is undefined)
  int by_bits = 0;
  for (int c = 0; c < nkeys; c++) if (!(flags[c] & DTB_FLAG_SORT_ONLY)) by_bits += kp.k[c].bits;
  const bool groups_k = do_groups && by_bits > 0;          // group boundaries come from the kernels

  // ---- rounds: a composite wider than 64 bits is sorted in several stable rounds,
  //      least significant key columns first (the reference refines column by column,
  //      sort.cc:561-595; here a round covers as many columns as fit in 64 bits) ----------
  struct Round { KeyPlan kp; bool has_by; };
  std::vector<Round> rounds;
  {
    int c = nkeys - 1;
    while (c >= 0) {
      int cols[MAX_KEYS], nc = 0, bits = 0;
      while (c >= 0 && bits + kp.k[c].bits <= 64) { cols[nc++] = c; bits += kp.k[c].bits; c--; }
      Round r; memset(&r.kp, 0, sizeof(r.kp)); r.has_by = false;
      int sh = 0, gs = 0;
      for (int j = 0; j < nc; j++) {
        KeyNorm kn = kp.k[cols[j]];
        kn.lshift = sh; sh += kn.bits;
        r.kp.k[nc - 1 - j] = kn;
        if (flags[cols[j]] & DTB_FLAG_SORT_ONLY) gs = sh; else r.has_by = true;
      }
      r.kp.nkeys = nc; r.kp.total_bits = sh; r.kp.group_shift = gs;
      if (sh > 0) rounds.push_back(r);
    }
  }
  const int nrounds = (int)rounds.size();
  const bool fused_raw = (nrounds == 1 && rounds[0].kp.nkeys == 1);   // normalise on the fly
  int max_bits = 0;
  for (auto& r : rounds) if (r.kp.total_bits > max_bits) max_bits = r.kp.total_bits;
  const int buf_key_bytes = max_bits <= 32 ? 4 : 8;

  if (opt_verbose) {
    fprintf(stderr, "[dtb200] group: n=%lld keys=%d bits=%d rounds=%d\n", (long long)n, nkeys, kp.total_bits, nrounds);
    for (int c = 0; c < nkeys; c++)
      fprintf(stderr, "[dtb200]   key %d: stype=%d desc=%d bits=%d cshift=%d lshift=%d na=%llu\n", c,
              kp.k[c].stype, kp.k[c].desc, kp.k[c].bits, kp.k[c].cshift, kp.k[c].lshift,
              (unsigned long long)h_stats[c].nacount);
  }

  DevBuf keyA, keyB, idxA, idxB, idxR0, idxR1;
  DTB_TRY(keyA.alloc((size_t)n * buf_key_bytes, s));
  DTB_TRY(keyB.alloc((size_t)n * buf_key_bytes, s));
  DTB_TRY(idxA.alloc((size_t)n * 4, s));
  DTB_TRY(idxB.alloc((size_t)n * 4, s));
  if (nrounds > 1) { DTB_TRY(idxR0.alloc((size_t)n * 4, s)); }
  if (nrounds > 2) { DTB_TRY(idxR1.alloc((size_t)n * 4, s)); }

  DTB_TL("scratch allocated");

  // ---- fused reducers: when the group key domain is small the reducers only need the key
  //      columns, not the RowIndex: they stream the rows in storage order once the groups are known
  //      (the streaming mode -- plain / shared-memory table / hot-key cache -- depends on the number of
  //      groups and the size of the largest one, see plan_direct).  Option "overlap_reducers" runs
  //      them on a side stream WHILE the sort passes run instead (hot keys guessed on the device). ----
  bool staged_keys = false;
  for (int c = 0; c < nkeys; c++) staged_keys = staged_keys || (in[c].buf.p != nullptr);
  const int dbits0 = (nrounds == 1) ? rounds[0].kp.total_bits - rounds[0].kp.group_shift : 99;
  bool fused_direct = fr && fr->n > 0 && groups_k && nrounds == 1 && !staged_keys && dbits0 <= 22 &&
                      na_pos != DTB_NA_REMOVE;
  if (fused_direct)
    for (int i = 0; i < fr->n; i++)
      fused_direct = fused_direct && fr->spec[i].op <= DTB_OP_NROWS &&           // streaming modes exist for sum..nrows only
                     (fr->spec[i].op == DTB_OP_NROWS || is_device_ptr(fr->spec[i].value.data));
  // Small key domain + handle path: the last pass counts rows per group key instead of writing
  // the sorted keys, and the offsets come from a scan over that table.
  const bool count_table = want_direct && groups_k && nrounds == 1 && !staged_keys && dbits0 <= 22 &&
                           na_pos != DTB_NA_REMOVE;
  int64_t ctable = 0;
  DevBuf gcount;
  if (count_table) {
    ctable = (int64_t)1 << (dbits0 < 10 ? 10 : dbits0);
    DTB_TRY(gcount.alloc(sizeof(u32) * (size_t)ctable, s));
    DTB_CUDA_CHECK(cudaMemsetAsync(gcount.p, 0, sizeof(u32) * (size_t)ctable, s));
  }
  DevBuf facc;
  DevBuf bxk;                                          // bucketed reducers: the rows' composite keys, kept
  bool bucket_wanted = false;                          // some value column costs >= 2 L2 atomics per row
  if (fused_direct && opt_bucketed && dbits0 >= BK_MIN_DBITS && dbits0 <= BK_MAX_DBITS)
    for (int i = 0; i < fr->n && !bucket_wanted; i++) {
      if (fr->spec[i].op == DTB_OP_NROWS) continue;
      int cost = 0;
      for (int j = 0; j < fr->n; j++)
        if (fr->spec[j].op != DTB_OP_NROWS && fr->spec[j].value.data == fr->spec[i].value.data)
          cost += fr->spec[j].op == DTB_OP_MEAN ? 2 : 1;
      bucket_wanted = cost >= 2;
    }
  const int64_t ftable = fused_direct ? ((int64_t)1 << dbits0) : 0;
  // Measured on C2: under the sort passes the accumulation gains ~2 % (both want the same SMs) and
  // inflates every scatter launch by ~40 %, so by default it runs on `s` after the offsets stage;
  // option "overlap_reducers" moves it to the side stream.
  cudaStream_t rs = s;
  if (fused_direct) {
    if (opt_overlap) { DTB_TRY(t_side.ensure()); rs = t_side.stream; }
    DTB_TRY(facc.alloc(sizeof(u64) * (size_t)ftable * 2 * (size_t)fr->n, s));
  }
  const int32_t* idx_cur = nullptr;        // rows in the order established by the previous rounds
  void* sorted_keys = nullptr;             // last round's sorted composite keys
  int last_key_bytes = 4;
  idx_cur = nullptr; sorted_keys = nullptr;
  for (int ri = 0; ri < nrounds; ri++) {
    const KeyPlan& rk = rounds[ri].kp;
    const bool last_round = (ri == nrounds - 1);
    const int key_bytes = rk.total_bits <= 32 ? 4 : 8;
    int width = (int)opt_radix_bits;                            // digits of at most 8 bits (256 bins), see dtb_radix.cu
    if (width <= 0 || width > 8) width = 8;
    if (width < 4) width = 4;                                   // 64 bits / 4 = MAX_PASSES
    PassPlan pp; plan_passes(rk.total_bits, width, pp);
    const bool want_sorted_keys = last_round && groups_k && rounds[ri].has_by && !count_table;
    // 64-bit keys whose sorted values are not needed afterwards: the passes over the low T-32 bits run
    // on 64-bit keys, the last of them writes only the upper 32 bits, and the remaining passes run on
    // 32-bit keys (8 instead of 12 bytes per row and pass in flight).  Never more passes than before.
    int narrow_after = -1;                                     // index of the pass that narrows
    if (key_bytes == 8 && !want_sorted_keys && !count_table && width == 8 && rk.total_bits > 32) {
      PassPlan lo, hi;
      plan_passes(rk.total_bits - 32, width, lo);
      plan_passes(32, width, hi);
      if (lo.npasses + hi.npasses <= pp.npasses) {
        pp.npasses = lo.npasses + hi.npasses;
        for (int p = 0; p < lo.npasses; p++) { pp.shift[p] = lo.shift[p]; pp.bits[p] = lo.bits[p]; }
        for (int p = 0; p < hi.npasses; p++) { pp.shift[lo.npasses + p] = hi.shift[p]; pp.bits[lo.npasses + p] = hi.bits[p]; }
        narrow_after = lo.npasses - 1;
      }
    }
    t_stats.radix_passes += pp.npasses;

    int src_kind = 1;
    // multi-column keys whose reducers will take the bucketed path (dtb_bucket.cu): the composite keys are
    // composed ONCE into a buffer the passes only read, and the bucket kernels read them again afterwards
    const bool keep_composite = bucket_wanted && !fused_raw && nrounds == 1 && key_bytes == 4;
    if (keep_composite) DTB_TRY(bxk.alloc(sizeof(u32) * (size_t)n, s));
    if (!fused_raw) {
      ProfScope ps("compose_keys", s);
      DTB_TRY(launch_compose_keys(rk, n, idx_cur, keep_composite ? bxk.p : keyA.p, key_bytes, s)); src_kind = 0;
    }

    // per-pass scratch: chunk x digit counts + digit totals/bases; largest digit count per pass
    DevBuf work; DTB_TRY(work.alloc(radix_pass_work_bytes(n), s));
    DevBuf hmax; DTB_TRY(hmax.alloc(sizeof(u32) * MAX_PASSES, s));

    int32_t* round_out = last_round ? order : ((ri & 1) ? idxR1.as<int32_t>() : idxR0.as<int32_t>());
    // raw single column: the first count kernel materialises the normalised keys into keyA
    void* kin = keep_composite ? bxk.p : keyA.p; void* kout = keyB.p;
    const int32_t* iin = idx_cur;
    for (int p = 0; p < pp.npasses; p++) {
      const bool last = (p == pp.npasses - 1);
      PassIO io;
      io.src_kind = (p == 0) ? src_kind : 0;
      io.keys_in = kin;
      io.keys_stage = (p == 0 && src_kind == 1 && opt_stage_keys) ? keyA.p : nullptr;
      io.narrow_out = (p == narrow_after) ? (rk.total_bits - 32) : 0;
      if (fuse_hist && ri == 0 && p == 0 && src_kind == 1 && pp.shift[0] == 0 && rk.k[0].cshift == 0 && rk.k[0].lshift == 0) {
        io.raw_hist = rawhist.as<unsigned short>(); io.raw_na = rawna.as<unsigned short>();
      }
      const int kb = (narrow_after >= 0 && p > narrow_after) ? 4 : key_bytes;   // key width this pass reads
      io.idx_in = iin;
      io.keys_out = (last && !want_sorted_keys) ? nullptr : kout;
      int32_t* iout = last ? round_out : ((p & 1) ? idxB.as<int32_t>() : idxA.as<int32_t>());
      io.idx_out = iout;
      const bool fork_here = fused_direct && rs != s && ri == 0 && p == 0;
      DTB_TRY(launch_radix_pass(io, rk, kb, n, pp.shift[p], pp.bits[p], work.as<u32>(),
                                hmax.as<u32>() + p, s, fork_here ? t_side.fork : nullptr,
                                (count_table && last) ? gcount.as<u32>() : nullptr, rk.group_shift));
      if (fork_here) {
        // the digit totals of pass 0 exist (hmax): the reducers decide about hot keys on the device
        DTB_CUDA_CHECK(cudaStreamWaitEvent(rs, t_side.fork, 0));
        DirectPlan dp = {DIRECT_DEVICE_HOT, nullptr, ftable, hmax.as<u32>(), (u32)(0.02 * (double)n)};
        for (int i = 0; i < fr->n; i++) {
          if (fr->spec[i].op == DTB_OP_NROWS) continue;
          ProfScope ps("reduce_direct_overlapped", rs);
          DTB_TRY(launch_direct_accumulate(fr->spec[i].op, rk, dp, fr->spec[i].value.data,
                                           fr->spec[i].value.stype, n, ftable,
                                           facc.as<u64>() + (size_t)ftable * 2 * i,
                                           facc.as<u64>() + (size_t)ftable * (2 * i + 1), rs));
        }
        DTB_CUDA_CHECK(cudaEventRecord(t_side.join, rs));
      }
      if (last && want_sorted_keys) { sorted_keys = kout; last_key_bytes = key_bytes; }
      kin = kout;
      kout = (kout == keyA.p) ? keyB.p : keyA.p;
      iin = iout;
    }
    idx_cur = round_out;
  }

  DTB_TL("passes enqueued");
  // ---- group offsets -----------------------------------------------------------------
  if (do_groups && !groups_k) {
    int32_t h[2] = {0, (int32_t)n};
    DTB_CUDA_CHECK(cudaMemcpyAsync(offsets, h, sizeof(h), cudaMemcpyHostToDevice, s));
    DTB_CUDA_CHECK(cudaStreamSynchronize(s));
    res.ngroups = 1;
  }
  if (groups_k) {
    const int64_t otiles = offsets_num_tiles(n);
    DevBuf oscr; DTB_TRY(oscr.alloc(sizeof(u64) * (size_t)(otiles + 4), s));
    DTB_CUDA_CHECK(cudaMemsetAsync(oscr.p, 0, oscr.bytes, s));
    u64* d_ng = oscr.as<u64>() + otiles + 2;
    DevBuf headflags;
    if (count_table) {
      ProfScope ps("group_offsets_from_counts", s);
      DTB_TRY(res.gkeys.alloc_owned(sizeof(u32) * (size_t)(ctable + 1), s));   // trimmed by the handle's lifetime
      DevBuf cscr; DTB_TRY(cscr.alloc(sizeof(u64) * (size_t)(2 * ctable / 1024 + 2), s));
      DTB_TRY(launch_offsets_from_counts(gcount.as<u32>(), ctable, n, offsets, res.gkeys.as<u32>(), d_ng,
                                         cscr.as<u64>(), s));
    } else if (nrounds == 1) {
      ProfScope ps("group_offsets", s);
      DTB_TRY(launch_group_offsets(sorted_keys, last_key_bytes, rounds[0].kp.group_shift, n, offsets, d_ng,
                                   oscr.as<u64>(), s));
    } else {
      // heads = rows where any by-column differs from the previous row: OR the per-round
      // comparisons; earlier rounds' keys are re-composed through the final RowIndex.
      DTB_TRY(headflags.alloc((size_t)n + 32, s));
      DTB_CUDA_CHECK(cudaMemsetAsync(headflags.p, 0, headflags.bytes, s));
      for (int ri = 0; ri < nrounds; ri++) {
        if (!rounds[ri].has_by) continue;
        const KeyPlan& rk = rounds[ri].kp;
        const int key_bytes = rk.total_bits <= 32 ? 4 : 8;
        const void* ks = sorted_keys;
        if (ri != nrounds - 1 || !sorted_keys) {
          void* tmp = (sorted_keys == keyA.p) ? keyB.p : keyA.p;
          DTB_TRY(launch_compose_keys(rk, n, order, tmp, key_bytes, s));
          ks = tmp;
        }
        DTB_TRY(launch_mark_heads(ks, key_bytes, rk.group_shift, n, headflags.as<uint8_t>(), s));
      }
      DTB_TRY(launch_group_offsets(headflags.p, 1, 0, n, offsets, d_ng, oscr.as<u64>(), s));
    }
    u64 h_ng[2] = {0, 0};                    // {groups, rows of the largest group (count-table path only)}
    DTB_CUDA_CHECK(cudaMemcpyAsync(h_ng, d_ng, 2 * sizeof(u64), cudaMemcpyDeviceToHost, s));
    DTB_CUDA_CHECK(stream_wait(s));
    res.ngroups = (int64_t)h_ng[0];
    // group key of every group, for the direct-address reducers
    bool staged = false;
    for (int c = 0; c < nkeys; c++) staged = staged || (in[c].buf.p != nullptr);
    const int dbits = (nrounds == 1) ? rounds[0].kp.total_bits - rounds[0].kp.group_shift : 99;
    if ((want_direct || fused_direct) && nrounds == 1 && !staged && dbits <= 22 && na_pos != DTB_NA_REMOVE) {
      if (!count_table) {
        DTB_TRY(res.gkeys.alloc_owned(sizeof(u32) * (size_t)(res.ngroups + 1), s));
        DTB_TRY(launch_group_keys(sorted_keys, last_key_bytes, offsets, rounds[0].kp.group_shift, res.ngroups,
                                  res.gkeys.as<u32>(), s));
      }
      res.direct = true;
      res.direct_gmax = count_table ? (int64_t)h_ng[1] : n;       // unknown: assume the worst
      res.direct_kp = rounds[0].kp;
      res.direct_table = (int64_t)1 << dbits;
    }
  }
  DTB_TL("offsets synced");

  // ---- fused reducers: finalize (direct) or evaluate through the RowIndex (general) ------------
  if (fr && fr->n > 0 && do_groups) {
    const int64_t ng = res.ngroups;
    fr->out.assign(fr->n, nullptr);
    if (fused_direct && rs != s) DTB_CUDA_CHECK(cudaStreamWaitEvent(s, t_side.join, 0));
    DirectPlan dp = {DIRECT_PLAIN, nullptr, ftable, nullptr, 0};
    DevBuf dmap;
    if (fused_direct && rs == s && ng > 0) {
      DTB_TRY(dmap.alloc(direct_map_bytes(ftable), s));
      DTB_TRY(plan_direct(ftable, res.gkeys.as<u32>(), offsets, ng, n, res.direct_gmax, dmap.p, s, dp));
    }
    DevBuf gacc;
    if (!fused_direct) DTB_TRY(gacc.alloc(sizeof(u64) * (size_t)(ng > 0 ? ng : 1) * 2, s));

    // ---- bucketed multi-reducer: value columns that would cost two or more L2 atomics per row (mean = sum +
    //      count; several reducers of one column) are partitioned by key bucket once and folded in shared
    //      memory, all their reducers together (dtb_bucket.cu).  Spread-out keys only: few groups and hot keys
    //      have their own streaming modes (plan_direct). --------------------------------------------------
    struct BucketCol { const void* data; int stype; u64* w[BK_NWORDS]; };
    std::vector<BucketCol> bcols;
    std::vector<int> bcol_of(fr->n, -1);
    std::list<DevBuf> bbufs;                                   // accumulator tables (live until the finalizes ran)
    DevBuf bstart, bscr;
    if (fused_direct && rs == s && ng > 0 && dp.kind == DIRECT_PLAIN && opt_bucketed &&
        dbits0 >= BK_MIN_DBITS && dbits0 <= BK_MAX_DBITS) {
      auto natomics = [](int op) { return op == DTB_OP_MEAN ? 2 : (op >= DTB_OP_SUM && op <= DTB_OP_COUNTNA ? 1 : 0); };
      for (int i = 0; i < fr->n; i++) {
        const dtb_reduce_spec& sp = fr->spec[i];
        if (sp.op == DTB_OP_NROWS || bcol_of[i] >= 0 || !reduce_out_stype_host(sp.op, sp.value.stype)) continue;
        int cost = 0;
        for (int j = i; j < fr->n; j++)
          if (fr->spec[j].op != DTB_OP_NROWS && fr->spec[j].value.data == sp.value.data && fr->spec[j].value.stype == sp.value.stype)
            cost += natomics(fr->spec[j].op);
        if (cost < 2) continue;
        BucketCol bc; bc.data = sp.value.data; bc.stype = sp.value.stype;
        for (int w = 0; w < BK_NWORDS; w++) bc.w[w] = nullptr;
        bool want[BK_NWORDS] = {false, false, false, false, false, false};
        const bool vflt = sp.value.stype == DTB_STYPE_FLOAT32 || sp.value.stype == DTB_STYPE_FLOAT64;
        for (int j = i; j < fr->n; j++) {
          const dtb_reduce_spec& sj = fr->spec[j];
          if (sj.op == DTB_OP_NROWS || sj.value.data != sp.value.data || sj.value.stype != sp.value.stype) continue;
          bcol_of[j] = (int)bcols.size();
          switch (sj.op) {
            case DTB_OP_SUM:  want[vflt ? BK_SUMF : BK_SUMI] = true; break;
            case DTB_OP_MEAN: want[BK_SUMF] = want[BK_CNT] = true; break;
            case DTB_OP_MIN:  want[BK_MIN] = true; break;
            case DTB_OP_MAX:  want[BK_MAX] = true; break;
            case DTB_OP_COUNT: want[BK_CNT] = true; break;
            case DTB_OP_COUNTNA: want[BK_CNTNA] = true; break;
          }
        }
        for (int w = 0; w < BK_NWORDS; w++) {
          if (!want[w]) continue;
          bbufs.emplace_back();
          DTB_TRY(bbufs.back().alloc(sizeof(u64) * (size_t)ftable, s));
          bc.w[w] = bbufs.back().as<u64>();
          fill_u64(bc.w[w], ftable, w == BK_MIN ? ~0ull : 0ull, s);
        }
        bcols.push_back(bc);
      }
      if (!bcols.empty()) {
        const int nb = 1 << (dbits0 > 11 ? dbits0 - 11 : 0);
        // sweeps of up to BK_MAXCOLS columns / 32 value bytes per row (the partitioned copies live in scratch)
        std::vector<std::pair<int, int>> sweeps;           // [first, last) into bcols
        size_t scr = 0;
        for (int c = 0; c < (int)bcols.size();) {
          int e = c, bytes = 0;
          while (e < (int)bcols.size() && e - c < BK_MAXCOLS && (e == c || bytes + stype_bytes(bcols[e].stype) <= 32))
            bytes += stype_bytes(bcols[e++].stype);
          const size_t need = bucket_scratch_bytes(n, bytes, e - c);
          scr = need > scr ? need : scr;
          sweeps.push_back({c, e});
          c = e;
        }
        DTB_TRY(bstart.alloc(bucket_starts_bytes(n) + sizeof(u32) * (size_t)(nb + 8), s));
        DTB_TRY(bscr.alloc(scr, s));
        if (!bxk.p) {                                  // single raw key column: its normalised keys, once
          DTB_TRY(bxk.alloc(sizeof(u32) * (size_t)n, s));
          ProfScope ps("compose_keys", s); DTB_TRY(launch_compose_keys(rounds[0].kp, n, nullptr, bxk.p, 4, s));
        }
        u32* slab_starts = bstart.as<u32>(); u32* start = slab_starts + bucket_starts_bytes(n) / sizeof(u32);
        DTB_TRY(launch_bucket_starts(bxk.as<u32>(), rounds[0].kp.group_shift, n, nb, slab_starts, start, s));
        for (auto& sw : sweeps) {
          const void* vals[BK_MAXCOLS]; int sts[BK_MAXCOLS]; unsigned long long* words[BK_MAXCOLS][BK_NWORDS];
          const int nc = sw.second - sw.first;
          for (int c = 0; c < nc; c++) {
            const BucketCol& bc = bcols[sw.first + c];
            vals[c] = bc.data; sts[c] = bc.stype;
            for (int w = 0; w < BK_NWORDS; w++) words[c][w] = bc.w[w];
          }
          DTB_TRY(launch_bucketed_reduce(bxk.as<u32>(), rounds[0].kp.group_shift, dbits0, nc, vals, sts, n, slab_starts,
                                         start, words, bscr.p, s));
        }
      }
    }
    for (int i = 0; i < fr->n; i++) {
      const dtb_reduce_spec& sp = fr->spec[i];
      const int out_st = (sp.op == DTB_OP_NROWS) ? DTB_STYPE_INT64 : reduce_out_stype_host(sp.op, sp.value.stype);
      if (!out_st) {
        set_error("Invalid column of stype " + std::to_string(sp.value.stype) + " in reducer " + std::to_string(sp.op));
        return stype_supported(sp.value.stype) ? DTB_EINVAL : DTB_ENOTIMPL;
      }
      DevBuf ob; DTB_TRY(ob.alloc_owned((size_t)(ng > 0 ? ng : 1) * stype_bytes(out_st), s));
      if (sp.op == DTB_OP_NROWS) {
        DTB_TRY(launch_nrows(offsets, ng, ob.p, s));
      } else if (bcol_of[i] >= 0) {
        const BucketCol& bc = bcols[bcol_of[i]];
        const bool vflt = sp.value.stype == DTB_STYPE_FLOAT32 || sp.value.stype == DTB_STYPE_FLOAT64;
        const u64* a0 = nullptr; const u64* a1 = nullptr;
        switch (sp.op) {
          case DTB_OP_SUM:  a0 = bc.w[vflt ? BK_SUMF : BK_SUMI]; break;
          case DTB_OP_MEAN: a0 = bc.w[BK_SUMF]; a1 = bc.w[BK_CNT]; break;
          case DTB_OP_MIN:  a0 = bc.w[BK_MIN]; break;
          case DTB_OP_MAX:  a0 = bc.w[BK_MAX]; break;
          case DTB_OP_COUNT: a0 = bc.w[BK_CNT]; break;
          default: a0 = bc.w[BK_CNTNA]; break;
        }
        DTB_TRY(launch_direct_finalize(sp.op, sp.value.stype, a0, a1, res.gkeys.as<u32>(), ng, ob.p, s));
      } else if (fused_direct) {
        u64* a0 = facc.as<u64>() + (size_t)ftable * 2 * i;
        u64* a1 = facc.as<u64>() + (size_t)ftable * (2 * i + 1);
        if (rs == s && ng > 0) {
          ProfScope ps("reduce_direct", s);
          DTB_TRY(launch_direct_accumulate(sp.op, rounds[0].kp, dp, sp.value.data, sp.value.stype, n, ftable, a0, a1, s));
        }
        DTB_TRY(launch_direct_finalize(sp.op, sp.value.stype, a0, a1,
                                       (dp.kind == DIRECT_SMALL && dp.map) ? nullptr : res.gkeys.as<u32>(), ng, ob.p, s));
      } else {
        DevIn dv; DTB_TRY(dv.bind(sp.value.data, (size_t)n * stype_bytes(sp.value.stype), s));
        DevBuf extra;
        const size_t xb = reduce_extra_bytes(sp.op, ng, n);
        if (xb) DTB_TRY(extra.alloc(xb, s));
        ProfScope ps("reduce", s);
        DTB_TRY(launch_reduce_impl(sp.op, dv.dptr, sp.value.stype, n, order + res.nskip, 0, offsets, ng,
                                   ng > 0 ? (int64_t)(n - res.nskip) : 0, gacc.as<u64>(), gacc.as<u64>() + ng, ob.p, s,
                                   xb ? extra.p : nullptr));
      }
      fr->out[i] = ob.detach();
    }
  }
  return DTB_OK;
}

}  // namespace dtb

using namespace dtb;

// ===========================================================================
// extern "C"
// ===========================================================================
struct dtb_groupby {
  void* order = nullptr;      // device int32[norder] (view into order_base)
  void* order_base = nullptr;
  void* offsets = nullptr;    // device int32[ngroups+1]
  int64_t norder = 0;
  int64_t ngroups = -1;
  int64_t nrows = 0;
  // direct-address reducers: valid while the caller keeps the key columns alive and unchanged
  bool direct = false;
  int64_t gmax = 0;           // rows of the largest group
  dtb::KeyPlan kp;
  int64_t table = 0;
  void* gkeys = nullptr;      // device uint32[ngroups]
  std::vector<void*> reduced; // outputs of the reducers evaluated by dtb_groupby_create_reduce
};

// A reducer fed piecewise (dtb_groupby_reduce_begin / _add / _end): the accumulator tables live across calls.
struct dtb_reduce_state {
  dtb_groupby* g = nullptr;
  int op = 0, stype = 0, out_stype = 0;
  void* acc = nullptr;        // device u64[2 * table]
  void* dmap = nullptr;       // plan_direct's map (shared-memory table / hot-key modes)
  dtb::DirectPlan dp;
  int64_t rows_added = 0;
};

extern "C" {

const char* dtb_last_error(void) { return t_error.c_str(); }
int dtb_abi_version(void) { return DTB_ABI_VERSION; }
int dtb_stype_size(int stype) { return stype_bytes(stype); }
int dtb_reduce_out_stype(int op, int stype) { return reduce_out_stype_host(op, stype); }

int dtb_init(int device) {
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) {
    set_error(std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    return DTB_ECUDA;
  }
  return ensure_context();
}

int dtb_memcpy(void* dst, const void* src, int64_t nbytes, dtb_stream stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (nbytes < 0 || (nbytes > 0 && (!dst || !src))) { set_error("bad dtb_memcpy arguments"); return DTB_EINVAL; }
  if (nbytes == 0) return DTB_OK;
  DTB_CUDA_CHECK(cudaMemcpyAsync(dst, src, (size_t)nbytes, cudaMemcpyDefault, s));
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  return DTB_OK;
}

int dtb_set_option(const char* name, int64_t value) {
  if (!name) { set_error("option name is NULL"); return DTB_EINVAL; }
  if (!strcmp(name, "radix_bits")) {
    if (value != 0 && (value < 4 || value > 8)) { set_error("radix_bits must be 0 (default) or 4..8"); return DTB_EINVAL; }
    opt_radix_bits = value; return DTB_OK;
  }
  if (!strcmp(name, "verbose")) { opt_verbose = value; return DTB_OK; }
  if (!strcmp(name, "profile")) { opt_profile = value; return DTB_OK; }
  if (!strcmp(name, "overlap_reducers")) { opt_overlap = value; return DTB_OK; }
  if (!strcmp(name, "bucketed_reducers")) { opt_bucketed = value ? 1 : 0; return DTB_OK; }
  if (!strcmp(name, "stage_keys")) { opt_stage_keys = value ? 1 : 0; return DTB_OK; }
  if (!strcmp(name, "fuse_stats_hist")) { opt_fuse_hist = value ? 1 : 0; return DTB_OK; }
  if (!strcmp(name, "trim_scratch")) {
    if (t_arena.depth == 0 && t_arena.device >= 0) {
      int cur = 0; cudaGetDevice(&cur);
      if (cur != t_arena.device) cudaSetDevice(t_arena.device);
      t_arena.trim();
      if (cur != t_arena.device) cudaSetDevice(cur);
    }
    return DTB_OK;
  }
  set_error(std::string("unknown option ") + name);
  return DTB_EINVAL;
}

int dtb_profile_count(void) { prof_collect(); return (int)t_prof_done.size(); }

int dtb_profile_get(int i, char* name, int cap, double* ms) {
  if (i < 0 || i >= (int)t_prof_done.size() || !name || cap < 1 || !ms) { set_error("bad dtb_profile_get arguments"); return DTB_EINVAL; }
  strncpy(name, t_prof_done[i].first.c_str(), (size_t)cap - 1);
  name[cap - 1] = 0;
  *ms = t_prof_done[i].second;
  return DTB_OK;
}

int dtb_profile_reset(void) { prof_collect(); t_prof_done.clear(); return DTB_OK; }

int dtb_get_option(const char* name, int64_t* value) {
  if (!name || !value) { set_error("NULL argument"); return DTB_EINVAL; }
  if (!strcmp(name, "radix_bits")) { *value = opt_radix_bits; return DTB_OK; }
  if (!strcmp(name, "verbose")) { *value = opt_verbose; return DTB_OK; }
  if (!strcmp(name, "profile")) { *value = opt_profile; return DTB_OK; }
  if (!strcmp(name, "overlap_reducers")) { *value = opt_overlap; return DTB_OK; }
  if (!strcmp(name, "bucketed_reducers")) { *value = opt_bucketed; return DTB_OK; }
  if (!strcmp(name, "stage_keys")) { *value = opt_stage_keys; return DTB_OK; }
  if (!strcmp(name, "fuse_stats_hist")) { *value = opt_fuse_hist; return DTB_OK; }
  set_error(std::string("unknown option ") + name);
  return DTB_EINVAL;
}

int dtb_last_call_stats(dtb_call_stats* out) {
  if (!out) { set_error("NULL argument"); return DTB_EINVAL; }
  *out = t_stats;
  return DTB_OK;
}

int dtb_group(const dtb_col* keys, int nkeys, const int* flags, int na_pos, int64_t nrows,
              dtb_stream stream, void* order_out, void* offsets_out, int64_t offsets_cap,
              int64_t* ngroups_out, int64_t* norder_out)
{
  cudaStream_t s = (cudaStream_t)stream;
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  if (!order_out && nrows > 0) { set_error("order_out is NULL"); return DTB_EINVAL; }
  if (nkeys >= 1 && flags && !(flags[0] & DTB_FLAG_SORT_ONLY) && !offsets_out) {
    set_error("offsets_out is NULL but groups were requested"); return DTB_EINVAL;
  }
  GroupResult res;
  // compute straight into the caller's device buffers when they are large enough
  int32_t* order_dev = (nrows > 0 && is_device_ptr(order_out) && na_pos != DTB_NA_REMOVE) ? (int32_t*)order_out : nullptr;
  int32_t* offsets_dev = (offsets_out && is_device_ptr(offsets_out) && offsets_cap >= nrows + 1) ? (int32_t*)offsets_out : nullptr;
  int rc = group_core(keys, nkeys, flags, na_pos, nrows, s, order_dev, offsets_dev, res);
  if (rc != DTB_OK) return rc;
  const int64_t norder = res.n - res.nskip;
  if (norder_out) *norder_out = norder;
  if (ngroups_out) *ngroups_out = res.ngroups;
  if (!order_dev && norder > 0) {
    const int32_t* src = res.order.as<int32_t>() + res.nskip;
    DTB_CUDA_CHECK(cudaMemcpyAsync(order_out, src, sizeof(int32_t) * (size_t)norder, cudaMemcpyDefault, s));
    if (!is_device_ptr(order_out)) DevOut::remember(order_out, src, sizeof(int32_t) * (size_t)norder, s);
  }
  if (res.ngroups >= 0 && !offsets_dev) {
    if (offsets_cap < res.ngroups + 1) {
      cudaStreamSynchronize(s);
      set_error("offsets_out holds " + std::to_string(offsets_cap) + " entries, need " + std::to_string(res.ngroups + 1));
      return DTB_ENOSPACE;
    }
    DTB_CUDA_CHECK(cudaMemcpyAsync(offsets_out, res.offsets.p, sizeof(int32_t) * (size_t)(res.ngroups + 1), cudaMemcpyDefault, s));
    if (!is_device_ptr(offsets_out)) DevOut::remember(offsets_out, res.offsets.p, sizeof(int32_t) * (size_t)(res.ngroups + 1), s);
  }
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  return DTB_OK;
}

int dtb_groupby_create(const dtb_col* keys, int nkeys, const int* flags, int na_pos, int64_t nrows,
                       dtb_stream stream, dtb_groupby** out)
{
  return dtb_groupby_create_reduce(keys, nkeys, flags, na_pos, nrows, stream, nullptr, 0, out);
}

int dtb_groupby_create_reduce(const dtb_col* keys, int nkeys, const int* flags, int na_pos, int64_t nrows,
                              dtb_stream stream, const dtb_reduce_spec* reducers, int nreducers,
                              dtb_groupby** out)
{
  cudaStream_t s = (cudaStream_t)stream;
  if (!out) { set_error("out is NULL"); return DTB_EINVAL; }
  *out = nullptr;
  if (nreducers < 0 || (nreducers > 0 && !reducers)) { set_error("bad reducer list"); return DTB_EINVAL; }
  if (nreducers > 0 && flags && nkeys > 0 && (flags[0] & DTB_FLAG_SORT_ONLY)) {
    set_error("reducers need a Groupby: the first key column must not be SORT_ONLY"); return DTB_EINVAL;
  }
  for (int i = 0; i < nreducers; i++)
    if (reducers[i].op == DTB_OP_MEDIAN || reducers[i].op == DTB_OP_NUNIQUE) {
      set_error("median/nunique read rows sorted inside their group: use dtb_sort_grouped + dtb_reduce"); return DTB_EINVAL;
    }
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  GroupResult res;
  FusedReducers fr; fr.spec = reducers; fr.n = nreducers;
  int rc = group_core(keys, nkeys, flags, na_pos, nrows, s, nullptr, nullptr, res, true, nreducers ? &fr : nullptr);
  if (rc != DTB_OK) { for (void* p : fr.out) if (p) cudaFreeAsync(p, s); return rc; }
  dtb_groupby* g = new dtb_groupby();
  g->reduced = fr.out;
  g->norder = res.n - res.nskip;
  g->ngroups = res.ngroups;
  g->nrows = res.n;
  if (res.direct) { g->direct = true; g->gmax = res.direct_gmax; g->kp = res.direct_kp; g->table = res.direct_table; g->gkeys = res.gkeys.detach(); }
  if (res.ngroups >= 0) {
    // shrink the worst-case offsets buffer to ngroups+1 entries
    DevBuf exact;
    // on failure the handle already owns the detached group keys and the fused reducer outputs:
    // dtb_groupby_destroy releases them (res.order is still owned by `res`)
    rc = exact.alloc_owned(sizeof(int32_t) * (size_t)(res.ngroups + 1), s);
    if (rc != DTB_OK) { dtb_groupby_destroy(g, stream); return rc; }
    cudaError_t e = cudaMemcpyAsync(exact.p, res.offsets.p, sizeof(int32_t) * (size_t)(res.ngroups + 1),
                                    cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) { set_error(cudaGetErrorString(e)); dtb_groupby_destroy(g, stream); return DTB_ECUDA; }
    g->offsets = exact.detach();
  }
  g->order_base = res.order.detach();
  g->order = (int32_t*)g->order_base + res.nskip;
  *out = g;
  return DTB_OK;
}

int64_t dtb_groupby_norder(const dtb_groupby* g) { return g ? g->norder : 0; }
int64_t dtb_groupby_ngroups(const dtb_groupby* g) { return g ? g->ngroups : -1; }
const void* dtb_groupby_order(const dtb_groupby* g) { return g ? g->order : nullptr; }
const void* dtb_groupby_offsets(const dtb_groupby* g) { return g ? g->offsets : nullptr; }
const void* dtb_groupby_reduced(const dtb_groupby* g, int i) {
  return (g && i >= 0 && i < (int)g->reduced.size()) ? g->reduced[i] : nullptr;
}

int dtb_groupby_destroy(dtb_groupby* g, dtb_stream stream) {
  if (!g) return DTB_OK;
  cudaStream_t s = (cudaStream_t)stream;
  if (g->order_base) cudaFreeAsync(g->order_base, s);
  if (g->offsets) cudaFreeAsync(g->offsets, s);
  if (g->gkeys) cudaFreeAsync(g->gkeys, s);
  for (void* p : g->reduced) if (p) cudaFreeAsync(p, s);
  delete g;
  return DTB_OK;
}

int dtb_reduce(int op, dtb_col value, int64_t nrows_value, const void* order, int order_is64,
               const void* offsets, int64_t ngroups, dtb_stream stream, void* out)
{
  cudaStream_t s = (cudaStream_t)stream;
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  if (ngroups < 0) { set_error("ngroups must be non-negative"); return DTB_EINVAL; }
  if (!offsets) { set_error("offsets is NULL"); return DTB_EINVAL; }
  if (!out && ngroups > 0) { set_error("out is NULL"); return DTB_EINVAL; }
  const int out_st = (op == DTB_OP_NROWS) ? DTB_STYPE_INT64 : reduce_out_stype_host(op, value.stype);
  if (!out_st) {
    set_error("Invalid column of stype " + std::to_string(value.stype) + " in reducer " + std::to_string(op));
    return stype_supported(value.stype) ? DTB_EINVAL : DTB_ENOTIMPL;
  }
  if (op != DTB_OP_NROWS && !value.data && nrows_value > 0) { set_error("value column data is NULL"); return DTB_EINVAL; }
  DTB_TRY(ensure_context());
  if (ngroups == 0) return DTB_OK;

  DevIn d_off; DTB_TRY(d_off.bind(offsets, sizeof(int32_t) * (size_t)(ngroups + 1), s));
  // caller-supplied offsets must be a Groupby: offsets[0] = 0, strictly increasing (groupby.h:41-47)
  int32_t n32 = 0;
  int bad = 0;
  if (is_device_ptr(offsets)) {
    DevBuf d_bad; DTB_TRY(d_bad.alloc(sizeof(int), s));
    DTB_CUDA_CHECK(cudaMemsetAsync(d_bad.p, 0, sizeof(int), s));
    if (!opt_trust_offsets) DTB_TRY(launch_offsets_check((const int32_t*)offsets, ngroups, d_bad.as<int>(), s));
    DTB_CUDA_CHECK(cudaMemcpyAsync(&n32, (const int32_t*)offsets + ngroups, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    DTB_CUDA_CHECK(cudaMemcpyAsync(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  } else {
    const int32_t* ho = (const int32_t*)offsets;
    n32 = ho[ngroups];
    if (ho[0] != 0) bad = 1;
    for (int64_t g = 0; g < ngroups && !bad; g++) if (ho[g] >= ho[g + 1]) bad = (int)(g < INT32_MAX ? g + 1 : INT32_MAX);
  }
  if (bad) {
    set_error("offsets is not a Groupby: offsets[0] must be 0 and offsets strictly increasing (group " +
              std::to_string(bad - 1) + " is empty or out of order)");
    return DTB_EINVAL;
  }
  const int64_t n = n32;
  DevIn d_val, d_ord;
  if (op != DTB_OP_NROWS) {
    DTB_TRY(d_val.bind(value.data, (size_t)nrows_value * stype_bytes(value.stype), s));
    DTB_TRY(d_ord.bind(order, (size_t)n * (order_is64 ? 8 : 4), s));
  }
  DevOut d_out; DTB_TRY(d_out.bind(out, (size_t)ngroups * stype_bytes(out_st), s));
  DevBuf acc; DTB_TRY(acc.alloc(sizeof(u64) * (size_t)ngroups * 2, s));
  DevBuf extra;
  const size_t xb = reduce_extra_bytes(op, ngroups, n);
  if (xb) DTB_TRY(extra.alloc(xb, s));
  {
    ProfScope ps("reduce", s);
    DTB_TRY(launch_reduce_impl(op, d_val.dptr, value.stype, nrows_value, d_ord.dptr, order_is64,
                               (const int32_t*)d_off.dptr, ngroups, n, acc.as<u64>(),
                               acc.as<u64>() + ngroups, d_out.dptr, s, xb ? extra.p : nullptr));
  }
  if (d_out.staged()) {
    DTB_TRY(d_out.finish((size_t)ngroups * stype_bytes(out_st), s));
    DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  }
  return DTB_OK;
}

int dtb_groupby_reduce(dtb_groupby* g, int op, dtb_col value, int64_t nrows_value, dtb_stream stream, void* out)
{
  cudaStream_t s = (cudaStream_t)stream;
  if (!g) { set_error("groupby handle is NULL"); return DTB_EINVAL; }
  if (g->ngroups < 0) { set_error("the handle holds no Groupby (sort-only call)"); return DTB_EINVAL; }
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  const bool device_value = (op == DTB_OP_NROWS) || is_device_ptr(value.data);
  if (!g->direct || op == DTB_OP_NROWS || op >= DTB_OP_FIRST || !device_value || nrows_value != g->nrows) {
    opt_trust_offsets = 1;                         // the handle's own offsets come from group()
    const int rc = dtb_reduce(op, value, nrows_value, g->order, 0, g->offsets, g->ngroups, stream, out);
    opt_trust_offsets = 0;
    return rc;
  }
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  const int out_st = reduce_out_stype_host(op, value.stype);
  if (!out_st) {
    set_error("Invalid column of stype " + std::to_string(value.stype) + " in reducer " + std::to_string(op));
    return stype_supported(value.stype) ? DTB_EINVAL : DTB_ENOTIMPL;
  }
  if (!out && g->ngroups > 0) { set_error("out is NULL"); return DTB_EINVAL; }
  DTB_TRY(ensure_context());
  if (g->ngroups == 0) return DTB_OK;
  DevOut d_out; DTB_TRY(d_out.bind(out, (size_t)g->ngroups * stype_bytes(out_st), s));
  DevBuf acc; DTB_TRY(acc.alloc(sizeof(u64) * (size_t)g->table * 2, s));
  DevBuf dmap; DTB_TRY(dmap.alloc(direct_map_bytes(g->table), s));
  DirectPlan dp;
  DTB_TRY(plan_direct(g->table, (const uint32_t*)g->gkeys, (const int32_t*)g->offsets, g->ngroups, g->nrows,
                      g->gmax, dmap.p, s, dp));
  {
    ProfScope ps("reduce_direct", s);
    DTB_TRY(launch_reduce_direct(op, g->kp, dp, value.data, value.stype, g->nrows, g->table,
                                 (const uint32_t*)g->gkeys, g->ngroups, acc.as<u64>(),
                                 acc.as<u64>() + g->table, d_out.dptr, s));
  }
  if (d_out.staged()) {
    DTB_TRY(d_out.finish((size_t)g->ngroups * stype_bytes(out_st), s));
    DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  }
  return DTB_OK;
}

int dtb_groupby_reduce_begin(dtb_groupby* g, int op, int value_stype, dtb_stream stream, dtb_reduce_state** out)
{
  cudaStream_t s = (cudaStream_t)stream;
  if (!g || !out) { set_error("groupby handle / out is NULL"); return DTB_EINVAL; }
  *out = nullptr;
  if (g->ngroups < 0) { set_error("the handle holds no Groupby (sort-only call)"); return DTB_EINVAL; }
  if (!g->direct || op < DTB_OP_SUM || op >= DTB_OP_NROWS) {
    set_error("piecewise reducers exist for the streaming path only (small key domain, device key columns, sum..countna)");
    return DTB_ENOTIMPL;
  }
  const int out_st = reduce_out_stype_host(op, value_stype);
  if (!out_st) {
    set_error("Invalid column of stype " + std::to_string(value_stype) + " in reducer " + std::to_string(op));
    return stype_supported(value_stype) ? DTB_EINVAL : DTB_ENOTIMPL;
  }
  DTB_TRY(ensure_context());
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  dtb_reduce_state* st = new dtb_reduce_state();
  st->g = g; st->op = op; st->stype = value_stype; st->out_stype = out_st;
  const size_t acc_bytes = sizeof(u64) * (size_t)g->table * 2, map_bytes = direct_map_bytes(g->table);
  if (cudaMalloc(&st->acc, acc_bytes ? acc_bytes : 8) != cudaSuccess || cudaMalloc(&st->dmap, map_bytes ? map_bytes : 8) != cudaSuccess) {
    cudaGetLastError(); cudaFree(st->acc); delete st; set_error("out of device memory"); return DTB_ENOMEM;
  }
  int rc = DTB_OK;
  if (g->ngroups > 0) {
    rc = plan_direct(g->table, (const uint32_t*)g->gkeys, (const int32_t*)g->offsets, g->ngroups, g->nrows, g->gmax, st->dmap, s, st->dp);
    if (rc == DTB_OK) rc = launch_direct_init(op, st->dp, g->table, (u64*)st->acc, (u64*)st->acc + g->table, s);
  }
  if (rc != DTB_OK) { cudaFree(st->acc); cudaFree(st->dmap); delete st; return rc; }
  *out = st;
  return DTB_OK;
}

int dtb_groupby_reduce_add(dtb_reduce_state* st, const void* value_rows, int64_t row0, int64_t nrows, dtb_stream stream)
{
  cudaStream_t s = (cudaStream_t)stream;
  if (!st || !st->g) { set_error("reducer state is NULL"); return DTB_EINVAL; }
  dtb_groupby* g = st->g;
  if (row0 < 0 || nrows < 0 || row0 + nrows > g->nrows) { set_error("row range outside the frame"); return DTB_EINVAL; }
  if (nrows == 0 || g->ngroups == 0) return DTB_OK;
  if (!value_rows || !is_device_ptr(value_rows)) { set_error("piecewise reducers take device rows"); return DTB_EINVAL; }
  KeyPlan kp = g->kp;                               // the key columns, advanced to row0
  for (int c = 0; c < kp.nkeys; c++)
    kp.k[c].data = (const char*)kp.k[c].data + (size_t)row0 * stype_bytes(kp.k[c].stype);
  ProfScope ps("reduce_direct", s);
  DTB_TRY(launch_direct_accumulate_rows(st->op, kp, st->dp, value_rows, st->stype, nrows, g->table,
                                        (u64*)st->acc, (u64*)st->acc + g->table, s));
  st->rows_added += nrows;
  return DTB_OK;
}

int dtb_groupby_reduce_end(dtb_reduce_state* st, dtb_stream stream, void* out)
{
  cudaStream_t s = (cudaStream_t)stream;
  if (!st || !st->g) { set_error("reducer state is NULL"); return DTB_EINVAL; }
  dtb_groupby* g = st->g;
  int rc = DTB_OK;
  if (g->ngroups > 0) {
    if (!out) { set_error("out is NULL"); rc = DTB_EINVAL; }
    else if (st->rows_added != g->nrows) { set_error("the pieces do not cover the frame's rows exactly once"); rc = DTB_EINVAL; }
    else {
      ArenaScope scope(s);
      rc = scope.rc;
      DevOut d_out;
      if (rc == DTB_OK) rc = d_out.bind(out, (size_t)g->ngroups * stype_bytes(st->out_stype), s);
      if (rc == DTB_OK)
        rc = launch_direct_finalize(st->op, st->stype, (const u64*)st->acc, (const u64*)st->acc + g->table,
                                    (st->dp.kind == DIRECT_SMALL && st->dp.map) ? nullptr : (const uint32_t*)g->gkeys,
                                    g->ngroups, d_out.dptr, s);
      if (rc == DTB_OK && d_out.staged()) rc = d_out.finish((size_t)g->ngroups * stype_bytes(st->out_stype), s);
      if (rc == DTB_OK && cudaStreamSynchronize(s) != cudaSuccess) { set_error("cudaStreamSynchronize failed"); rc = DTB_ECUDA; }
    }
  }
  if (rc != DTB_OK) cudaStreamSynchronize(s);       // the tables may still be in use
  cudaFree(st->acc); cudaFree(st->dmap);
  delete st;
  return rc;
}

int dtb_gather(dtb_col src, int64_t nrows_src, const void* order, int order_is64, int64_t n,
               dtb_stream stream, void* out)
{
  cudaStream_t s = (cudaStream_t)stream;
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  const int esz = stype_bytes(src.stype);
  if (!esz) { set_error("Unable to gather Column of stype " + std::to_string(src.stype)); return DTB_ENOTIMPL; }
  if (n < 0 || nrows_src < 0) { set_error("negative size"); return DTB_EINVAL; }
  if (n > 0 && (!order || !out)) { set_error("order/out is NULL"); return DTB_EINVAL; }
  DTB_TRY(ensure_context());
  if (n == 0) return DTB_OK;
  DevIn d_src, d_ord;
  DTB_TRY(d_src.bind(src.data, (size_t)nrows_src * esz, s));
  DTB_TRY(d_ord.bind(order, (size_t)n * (order_is64 ? 8 : 4), s));
  DevOut d_out; DTB_TRY(d_out.bind(out, (size_t)n * esz, s));
  DTB_TRY(launch_gather(d_src.dptr, src.stype, nrows_src, d_ord.dptr, order_is64, n, d_out.dptr, s));
  if (d_out.staged()) {
    DTB_TRY(d_out.finish((size_t)n * esz, s));
    DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  }
  return DTB_OK;
}

int dtb_window_out_stype(int op, int stype) { return window_out_stype_host(op, stype); }

int dtb_window(int op, int64_t param, dtb_col value, int64_t nrows_value, const void* order, const void* offsets,
               int64_t ngroups, dtb_stream stream, void* out)
{
  cudaStream_t s = (cudaStream_t)stream;
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  if (op < DTB_WIN_CUMSUM || op > DTB_WIN_SHIFT) { set_error("unknown window op " + std::to_string(op)); return DTB_EINVAL; }
  const bool uses_value = op != DTB_WIN_CUMCOUNT && op != DTB_WIN_NGROUP;
  const int out_st = window_out_stype_host(op, value.stype);
  if (!out_st) {
    set_error("Invalid column of stype " + std::to_string(value.stype) + " in window op " + std::to_string(op));
    return stype_supported(value.stype) ? DTB_EINVAL : DTB_ENOTIMPL;
  }
  if (op == DTB_WIN_SHIFT && (param < INT32_MIN || param > INT32_MAX)) {
    set_error("Value is too large to fit in an int32"); return DTB_EINVAL;
  }
  if (ngroups < 0 || nrows_value < 0) { set_error("negative size"); return DTB_EINVAL; }
  if (!offsets) { set_error("offsets is NULL"); return DTB_EINVAL; }
  if (uses_value && !value.data && nrows_value > 0) { set_error("value column data is NULL"); return DTB_EINVAL; }
  DTB_TRY(ensure_context());
  if (ngroups == 0) return DTB_OK;

  DevIn d_off; DTB_TRY(d_off.bind(offsets, sizeof(int32_t) * (size_t)(ngroups + 1), s));
  // caller-supplied offsets must be a Groupby: offsets[0] = 0, strictly increasing (groupby.h:41-47)
  int32_t n32 = 0;
  int bad = 0;
  {
    DevBuf d_bad; DTB_TRY(d_bad.alloc(sizeof(int), s));
    DTB_CUDA_CHECK(cudaMemsetAsync(d_bad.p, 0, sizeof(int), s));
    DTB_TRY(launch_offsets_check((const int32_t*)d_off.dptr, ngroups, d_bad.as<int>(), s));
    DTB_CUDA_CHECK(cudaMemcpyAsync(&n32, (const int32_t*)d_off.dptr + ngroups, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    DTB_CUDA_CHECK(cudaMemcpyAsync(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  }
  if (bad) {
    set_error("offsets is not a Groupby: offsets[0] must be 0 and offsets strictly increasing (group " +
              std::to_string(bad - 1) + " is empty or out of order)");
    return DTB_EINVAL;
  }
  const int64_t n = n32;
  if (!out && n > 0) { set_error("out is NULL"); return DTB_EINVAL; }
  DevIn d_val, d_ord;
  if (uses_value) DTB_TRY(d_val.bind(value.data, (size_t)nrows_value * stype_bytes(value.stype), s));
  DTB_TRY(d_ord.bind(order, (size_t)n * sizeof(int32_t), s));
  DevOut d_out; DTB_TRY(d_out.bind(out, (size_t)n * stype_bytes(out_st), s));
  DevBuf scratch; DTB_TRY(scratch.alloc(window_scratch_bytes(n), s));
  DTB_TRY(launch_window(op, param, d_val.dptr, value.stype, uses_value ? nrows_value : 0, (const int32_t*)d_ord.dptr,
                        (const int32_t*)d_off.dptr, ngroups, n, d_out.dptr, scratch.p, s));
  if (d_out.staged()) {
    DTB_TRY(d_out.finish((size_t)n * stype_bytes(out_st), s));
    DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  }
  return DTB_OK;
}

int dtb_dense_scatter(const void* keys, int key_stype, const void* vals, int64_t n, int64_t kmin, int64_t table_size,
                      void* table, void* present, dtb_stream stream)
{
  cudaStream_t s = (cudaStream_t)stream;
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  const int kb = (key_stype == DTB_STYPE_INT32) ? 4 : (key_stype == DTB_STYPE_INT64 ? 8 : 0);
  if (!kb) { set_error("dense merge: group keys must be int32 or int64"); return DTB_ENOTIMPL; }
  if (n < 0 || table_size < 1 || (n > 0 && (!keys || !vals)) || !table || !present) { set_error("bad dtb_dense_scatter arguments"); return DTB_EINVAL; }
  if (!is_device_ptr(table) || !is_device_ptr(present) || (n > 0 && (!is_device_ptr(keys) || !is_device_ptr(vals)))) {
    set_error("dense merge works on device buffers (they are NCCL all-reduced in place)"); return DTB_EINVAL;
  }
  DTB_TRY(ensure_context());
  return launch_dense_scatter(keys, kb, vals, n, kmin, table_size, table, (uint32_t*)present, s);
}

int dtb_dense_compact(const void* table, const void* present, int64_t table_size, int64_t kmin, int key_stype,
                      void* out_keys, void* out_vals, int64_t* ngroups_out, dtb_stream stream)
{
  cudaStream_t s = (cudaStream_t)stream;
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  const int kb = (key_stype == DTB_STYPE_INT32) ? 4 : (key_stype == DTB_STYPE_INT64 ? 8 : 0);
  if (!kb) { set_error("dense merge: group keys must be int32 or int64"); return DTB_ENOTIMPL; }
  if (!table || !present || !out_keys || !out_vals || !ngroups_out) { set_error("NULL argument"); return DTB_EINVAL; }
  if (table_size < 1024 || table_size % 1024 || table_size > ((int64_t)1 << 22)) {
    set_error("dense merge: table size must be a multiple of 1024 and at most 2^22"); return DTB_EINVAL;
  }
  if (!is_device_ptr(table) || !is_device_ptr(present) || !is_device_ptr(out_keys) || !is_device_ptr(out_vals)) {
    set_error("dense merge works on device buffers"); return DTB_EINVAL;
  }
  DTB_TRY(ensure_context());
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  DevBuf offs, gidx, scr;
  DTB_TRY(offs.alloc(sizeof(int32_t) * (size_t)(table_size + 1), s));
  DTB_TRY(gidx.alloc(sizeof(u32) * (size_t)(table_size + 1), s));
  DTB_TRY(scr.alloc(sizeof(u64) * (size_t)(2 * table_size / 1024 + 4), s));
  u64* d_ng = scr.as<u64>() + 2 * table_size / 1024 + 2;
  DTB_CUDA_CHECK(cudaMemsetAsync(d_ng, 0, 2 * sizeof(u64), s));
  DTB_TRY(launch_offsets_from_counts((const u32*)present, table_size, 0, offs.as<int32_t>(), gidx.as<u32>(), d_ng, scr.as<u64>(), s));
  u64 h_ng = 0;
  DTB_CUDA_CHECK(cudaMemcpyAsync(&h_ng, d_ng, sizeof(u64), cudaMemcpyDeviceToHost, s));
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  *ngroups_out = (int64_t)h_ng;
  DTB_TRY(launch_dense_emit(gidx.as<u32>(), table, (int64_t)h_ng, kmin, kb, out_keys, out_vals, s));
  return DTB_OK;
}

int dtb_sort_grouped(dtb_col value, int64_t nrows_value, const void* order, const void* offsets, int64_t ngroups,
                     dtb_stream stream, void* order_out)
{
  cudaStream_t s = (cudaStream_t)stream;
  const int esz = stype_bytes(value.stype);
  if (!esz) { set_error("Unable to sort Column of stype " + std::to_string(value.stype)); return DTB_ENOTIMPL; }
  if (ngroups < 0 || !offsets) { set_error("bad dtb_sort_grouped arguments"); return DTB_EINVAL; }
  DTB_TRY(ensure_context());
  if (ngroups == 0) return DTB_OK;
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  DevIn d_off; DTB_TRY(d_off.bind(offsets, sizeof(int32_t) * (size_t)(ngroups + 1), s));
  int32_t n32 = 0;
  DTB_CUDA_CHECK(cudaMemcpyAsync(&n32, (const int32_t*)d_off.dptr + ngroups, sizeof(int32_t), cudaMemcpyDefault, s));
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  const int64_t n = n32;
  if (n == 0) return DTB_OK;
  if (!order_out) { set_error("order_out is NULL"); return DTB_EINVAL; }
  DevIn d_val, d_ord;
  DTB_TRY(d_val.bind(value.data, (size_t)nrows_value * esz, s));
  DTB_TRY(d_ord.bind(order, (size_t)n * 4, s));
  DevOut d_out; DTB_TRY(d_out.bind(order_out, (size_t)n * 4, s));
  // sort by (group id, value): the group id of every sorted position and the value seen through the RowIndex
  DevBuf gid, vg, iota;
  DTB_TRY(gid.alloc((size_t)n * 4, s));
  DTB_TRY(vg.alloc((size_t)n * esz, s));
  DTB_TRY(launch_expand_gid((const int32_t*)d_off.dptr, ngroups, n, gid.as<int32_t>(), s));
  const void* ord = d_ord.dptr;
  if (!ord) { DTB_TRY(iota.alloc((size_t)n * 4, s)); DTB_TRY(launch_iota32(iota.as<int32_t>(), n, s)); ord = iota.p; }
  DTB_TRY(launch_gather(d_val.dptr, value.stype, nrows_value, ord, 0, n, vg.p, s));
  dtb_col keys[2] = {{gid.p, DTB_STYPE_INT32, 0}, {vg.p, value.stype, 0}};
  const int flags[2] = {DTB_FLAG_SORT_ONLY, DTB_FLAG_SORT_ONLY};
  GroupResult res;
  DTB_TRY(group_core(keys, 2, flags, DTB_NA_FIRST, n, s, nullptr, nullptr, res));
  // positions -> rows
  DTB_TRY(launch_gather(ord, DTB_STYPE_INT32, n, res.order.p, 0, n, d_out.dptr, s));
  if (d_out.staged()) DTB_TRY(d_out.finish((size_t)n * 4, s));
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  return DTB_OK;
}

int dtb_set_select(int mode, const void* order, const void* offsets, int64_t ngroups, const int64_t* cum_sizes,
                   int ninputs, dtb_stream stream, void* rows_out, int64_t* nout)
{
  cudaStream_t s = (cudaStream_t)stream;
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  if (mode < DTB_SET_UNION || mode > DTB_SET_SYMDIFF) { set_error("unknown set operation"); return DTB_EINVAL; }
  if (ngroups < 0 || !nout || ninputs < 1 || ninputs > 64 || !cum_sizes) { set_error("bad dtb_set_select arguments"); return DTB_EINVAL; }
  *nout = 0;
  DTB_TRY(ensure_context());
  if (ngroups == 0) return DTB_OK;
  if (!order || !offsets || !rows_out) { set_error("NULL argument"); return DTB_EINVAL; }
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  const int64_t n = cum_sizes[ninputs - 1];
  DevIn d_ord, d_off;
  DTB_TRY(d_ord.bind(order, (size_t)n * 4, s));
  DTB_TRY(d_off.bind(offsets, sizeof(int32_t) * (size_t)(ngroups + 1), s));
  DevOut d_out; DTB_TRY(d_out.bind(rows_out, (size_t)ngroups * 4, s));
  DevBuf d_sizes, flags, pos, oscr;
  DTB_TRY(d_sizes.alloc(sizeof(int64_t) * (size_t)ninputs, s));
  DTB_CUDA_CHECK(cudaMemcpyAsync(d_sizes.p, cum_sizes, sizeof(int64_t) * (size_t)ninputs, cudaMemcpyHostToDevice, s));
  const int64_t m = ngroups + 1;                          // flags[0] = sentinel head for the compaction
  DTB_TRY(flags.alloc((size_t)m + 64, s));
  DTB_CUDA_CHECK(cudaMemsetAsync(flags.p, 0, (size_t)m + 64, s));
  DTB_TRY(launch_set_select((const int32_t*)d_ord.dptr, (const int32_t*)d_off.dptr, ngroups, d_sizes.as<int64_t>(),
                            ninputs, mode, flags.as<uint8_t>(), s));
  const int64_t otiles = offsets_num_tiles(m);
  DTB_TRY(pos.alloc(sizeof(int32_t) * (size_t)(m + 1), s));
  DTB_TRY(oscr.alloc(sizeof(u64) * (size_t)(otiles + 4), s));
  DTB_CUDA_CHECK(cudaMemsetAsync(oscr.p, 0, oscr.bytes, s));
  u64* d_ng = oscr.as<u64>() + otiles + 2;
  DTB_TRY(launch_group_offsets(flags.p, 1, 0, m, pos.as<int32_t>(), d_ng, oscr.as<u64>(), s));
  u64 h_ng = 0;
  DTB_CUDA_CHECK(cudaMemcpyAsync(&h_ng, d_ng, sizeof(u64), cudaMemcpyDeviceToHost, s));
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  const int64_t nsel = (int64_t)h_ng - 1;                 // without the sentinel
  DTB_TRY(launch_set_emit(pos.as<int32_t>(), nsel, (const int32_t*)d_ord.dptr, (const int32_t*)d_off.dptr,
                          (int32_t*)d_out.dptr, s));
  if (d_out.staged()) DTB_TRY(d_out.finish((size_t)nsel * 4, s));
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  *nout = nsel;
  return DTB_OK;
}

int dtb_largest_group(const void* offsets, int64_t ngroups, int64_t skip, dtb_stream stream, int64_t* index_out,
                      int64_t* size_out)
{
  cudaStream_t s = (cudaStream_t)stream;
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  if (!index_out || !size_out || ngroups < 0 || skip < 0) { set_error("bad dtb_largest_group arguments"); return DTB_EINVAL; }
  *index_out = -1; *size_out = 0;
  DTB_TRY(ensure_context());
  if (ngroups <= skip) return DTB_OK;
  if (!offsets) { set_error("offsets is NULL"); return DTB_EINVAL; }
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  DevIn d_off; DTB_TRY(d_off.bind(offsets, sizeof(int32_t) * (size_t)(ngroups + 1), s));
  DevBuf r; DTB_TRY(r.alloc(sizeof(u64), s));
  DTB_CUDA_CHECK(cudaMemsetAsync(r.p, 0, sizeof(u64), s));
  DTB_TRY(launch_largest_group((const int32_t*)d_off.dptr, ngroups, skip, r.as<u64>(), s));
  u64 h = 0;
  DTB_CUDA_CHECK(cudaMemcpyAsync(&h, r.p, sizeof(u64), cudaMemcpyDeviceToHost, s));
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  if (h) { *size_out = (int64_t)(h >> 32); *index_out = (int64_t)(0xffffffffu - (u32)(h & 0xffffffffu)); }
  return DTB_OK;
}

int dtb_slice_groups(const void* offsets, int64_t ngroups, int64_t start, int64_t stop, int64_t step,
                     dtb_stream stream, void* rows_out, int64_t rows_capacity, void* offsets_out,
                     int64_t* ngroups_out, int64_t* nrows_out)
{
  cudaStream_t s = (cudaStream_t)stream;
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  if (!ngroups_out || !nrows_out || ngroups < 0 || rows_capacity < 0) { set_error("bad dtb_slice_groups arguments"); return DTB_EINVAL; }
  *ngroups_out = 0; *nrows_out = 0;
  if (ngroups > 0 && (!offsets || !offsets_out)) { set_error("offsets / offsets_out is NULL"); return DTB_EINVAL; }
  if (step == DTB_SLICE_NA) step = 1;                                   // fexpr_literal_sliceint.cc:86
  if (step != (int64_t)(int32_t)step) { set_error("slice step does not fit int32"); return DTB_EINVAL; }
  if (step == 0 && (start == DTB_SLICE_NA || stop == DTB_SLICE_NA || stop <= 0 || stop > (int64_t)INT32_MAX)) {
    set_error("a slice with step 0 needs a start and a positive count"); return DTB_EINVAL;    // the reference asserts it (:150-152)
  }
  DTB_TRY(ensure_context());
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  if (ngroups == 0) {
    if (offsets_out) {
      DevOut z; DTB_TRY(z.bind(offsets_out, sizeof(int32_t), s));
      DTB_CUDA_CHECK(cudaMemsetAsync(z.dptr, 0, sizeof(int32_t), s));
      DTB_TRY(z.finish(sizeof(int32_t), s));
      DTB_CUDA_CHECK(cudaStreamSynchronize(s));
    }
    return DTB_OK;
  }
  DevIn d_off; DTB_TRY(d_off.bind(offsets, sizeof(int32_t) * (size_t)(ngroups + 1), s));
  DevOut d_oo; DTB_TRY(d_oo.bind(offsets_out, sizeof(int32_t) * (size_t)(ngroups + 1), s));
  int32_t h_last = 0;                                                   // rows of the grouped frame
  DTB_CUDA_CHECK(cudaMemcpyAsync(&h_last, (const int32_t*)d_off.dptr + ngroups, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  SliceParams p;
  p.has_start = start != DTB_SLICE_NA; p.has_stop = stop != DTB_SLICE_NA;
  p.start = p.has_start ? start : 0; p.stop = p.has_stop ? stop : 0; p.step = step; p.nrows = (long long)(u32)h_last;
  DevBuf scr, gsel, tot;
  DTB_TRY(scr.alloc(slice_scratch_bytes(ngroups), s));
  DTB_TRY(gsel.alloc(sizeof(int32_t) * (size_t)ngroups, s));
  DTB_TRY(tot.alloc(2 * sizeof(u64), s));
  DTB_TRY(launch_slice_groups_plan((const int32_t*)d_off.dptr, ngroups, p, scr.p, (int32_t*)d_oo.dptr, gsel.as<int32_t>(),
                                   tot.as<u64>(), s));
  u64 h_tot[2] = {0, 0};
  DTB_CUDA_CHECK(cudaMemcpyAsync(h_tot, tot.p, sizeof(h_tot), cudaMemcpyDeviceToHost, s));
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  const int64_t nout = (int64_t)h_tot[0], ng_out = (int64_t)h_tot[1];
  *nrows_out = nout; *ngroups_out = ng_out;
  if (nout > (int64_t)INT32_MAX) { set_error("the slice selects more than INT32_MAX rows"); return DTB_ENOTIMPL; }
  if (nout > rows_capacity) { set_error("rows_out is too small: " + std::to_string(nout) + " rows selected"); return DTB_ENOSPACE; }
  const int32_t h_end = (int32_t)nout;
  DTB_CUDA_CHECK(cudaMemcpyAsync((int32_t*)d_oo.dptr + ng_out, &h_end, sizeof(int32_t), cudaMemcpyHostToDevice, s));
  if (nout > 0) {
    if (!rows_out) { set_error("rows_out is NULL"); return DTB_EINVAL; }
    DevOut d_rows; DTB_TRY(d_rows.bind(rows_out, sizeof(int32_t) * (size_t)nout, s));
    DevBuf gid; DTB_TRY(gid.alloc(sizeof(int32_t) * (size_t)nout, s));
    DTB_TRY(launch_slice_groups_emit((const int32_t*)d_off.dptr, p, (const int32_t*)d_oo.dptr, gsel.as<int32_t>(), ng_out, nout,
                                     gid.as<int32_t>(), (int32_t*)d_rows.dptr, s));
    DTB_TRY(d_rows.finish(sizeof(int32_t) * (size_t)nout, s));
  }
  DTB_TRY(d_oo.finish(sizeof(int32_t) * (size_t)(ng_out + 1), s));
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  return DTB_OK;
}

int dtb_join(const dtb_col* xkeys, const dtb_col* jkeys, int nkeys, int64_t nrows_x, int64_t nrows_j,
             dtb_stream stream, void* index_out)
{
  cudaStream_t s = (cudaStream_t)stream;
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  if (nkeys < 1 || nkeys > MAX_KEYS || !xkeys || !jkeys) { set_error("number of key columns must be in 1.." + std::to_string(MAX_KEYS)); return DTB_EINVAL; }
  if (nrows_x < 0 || nrows_j < 0 || nrows_j > (int64_t)INT32_MAX) { set_error("bad row counts"); return DTB_EINVAL; }
  for (int c = 0; c < nkeys; c++) {
    if (!stype_supported(xkeys[c].stype) || !stype_supported(jkeys[c].stype)) {
      set_error("join keys of stype " + std::to_string(xkeys[c].stype) + " / " + std::to_string(jkeys[c].stype) + " are not supported");
      return DTB_ENOTIMPL;
    }
    const bool xd = xkeys[c].stype == DTB_STYPE_DATE32 || xkeys[c].stype == DTB_STYPE_TIME64;
    const bool jd = jkeys[c].stype == DTB_STYPE_DATE32 || jkeys[c].stype == DTB_STYPE_TIME64;
    if ((xd || jd) && xkeys[c].stype != jkeys[c].stype) {       // join.cc:384-385: date/time only join their own type
      set_error("a date/time key column can only be joined to a column of the same type"); return DTB_EINVAL;
    }
  }
  DTB_TRY(ensure_context());
  if (nrows_x == 0) return DTB_OK;
  if (!index_out) { set_error("index_out is NULL"); return DTB_EINVAL; }
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  std::vector<DevIn> xin(nkeys), jin(nkeys);
  const void* xp[MAX_KEYS]; const void* jp[MAX_KEYS]; int xst[MAX_KEYS], jst[MAX_KEYS];
  for (int c = 0; c < nkeys; c++) {
    DTB_TRY(xin[c].bind(xkeys[c].data, (size_t)nrows_x * stype_bytes(xkeys[c].stype), s));
    DTB_TRY(jin[c].bind(jkeys[c].data, (size_t)nrows_j * stype_bytes(jkeys[c].stype), s));
    xp[c] = xin[c].dptr; jp[c] = jin[c].dptr; xst[c] = xkeys[c].stype; jst[c] = jkeys[c].stype;
  }
  DevOut d_out; DTB_TRY(d_out.bind(index_out, (size_t)nrows_x * 4, s));
  DTB_TRY(launch_join(nkeys, xp, xst, jp, jst, nrows_x, nrows_j, (int32_t*)d_out.dptr, s));
  if (d_out.staged()) { DTB_TRY(d_out.finish((size_t)nrows_x * 4, s)); DTB_CUDA_CHECK(cudaStreamSynchronize(s)); }
  return DTB_OK;
}

int dtb_cache_begin(void) {
  t_cache.depth++;
  return DTB_OK;
}

int dtb_cache_end(void) {
  if (t_cache.depth > 0 && --t_cache.depth == 0) { cudaDeviceSynchronize(); t_cache.clear(); }
  return DTB_OK;
}

int dtb_group64(const dtb_col* keys, int nkeys, const int* flags, int na_pos, int64_t nrows, dtb_stream stream,
                void* order_out, void* offsets_out, int64_t offsets_cap, int64_t* ngroups_out, int64_t* norder_out)
{
  cudaStream_t s = (cudaStream_t)stream;
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  if (!order_out && nrows > 0) { set_error("order_out is NULL"); return DTB_EINVAL; }
  if (nkeys >= 1 && flags && !(flags[0] & DTB_FLAG_SORT_ONLY) && !offsets_out) {
    set_error("offsets_out is NULL but groups were requested"); return DTB_EINVAL;
  }
  GroupResult res;
  int rc = group_core(keys, nkeys, flags, na_pos, nrows, s, nullptr, nullptr, res, false, nullptr, /*wide=*/true);
  if (rc != DTB_OK) return rc;
  const int64_t norder = res.n - res.nskip;
  if (norder_out) *norder_out = norder;
  if (ngroups_out) *ngroups_out = res.ngroups;
  // zero-extend the 32-bit row ids / offsets to the int64 layout of an ARR64 RowIndex and int64 offsets
  if (norder > 0) {
    DevOut d_ord; DTB_TRY(d_ord.bind(order_out, sizeof(int64_t) * (size_t)norder, s));
    DTB_TRY(launch_widen_u32((const uint32_t*)res.order.p + res.nskip, norder, (int64_t*)d_ord.dptr, s));
    if (d_ord.staged()) DTB_TRY(d_ord.finish(sizeof(int64_t) * (size_t)norder, s));
  }
  if (res.ngroups >= 0) {
    if (offsets_cap < res.ngroups + 1) {
      cudaStreamSynchronize(s);
      set_error("offsets_out holds " + std::to_string(offsets_cap) + " entries, need " + std::to_string(res.ngroups + 1));
      return DTB_ENOSPACE;
    }
    DevOut d_off; DTB_TRY(d_off.bind(offsets_out, sizeof(int64_t) * (size_t)(res.ngroups + 1), s));
    DTB_TRY(launch_widen_u32((const uint32_t*)res.offsets.p, res.ngroups + 1, (int64_t*)d_off.dptr, s));
    if (d_off.staged()) DTB_TRY(d_off.finish(sizeof(int64_t) * (size_t)(res.ngroups + 1), s));
  }
  DTB_CUDA_CHECK(cudaStreamSynchronize(s));
  return DTB_OK;
}

int dtb_lower_bound(dtb_col sorted, int64_t nrows, dtb_col values, int64_t nvalues, dtb_stream stream, void* out)
{
  cudaStream_t s = (cudaStream_t)stream;
  t_stats = dtb_call_stats{0, 0, 0, 0, 0};
  if (sorted.stype != values.stype || !stype_supported(sorted.stype)) { set_error("lower_bound: columns must share a supported stype"); return DTB_EINVAL; }
  if (nrows < 0 || nvalues < 0 || (nvalues > 0 && (!values.data || !out))) { set_error("bad dtb_lower_bound arguments"); return DTB_EINVAL; }
  DTB_TRY(ensure_context());
  if (nvalues == 0) return DTB_OK;
  ArenaScope scope(s); if (scope.rc != DTB_OK) return scope.rc;
  const int esz = stype_bytes(sorted.stype);
  DevIn d_s, d_v;
  DTB_TRY(d_s.bind(sorted.data, (size_t)nrows * esz, s));
  DTB_TRY(d_v.bind(values.data, (size_t)nvalues * esz, s));
  DevOut d_out; DTB_TRY(d_out.bind(out, (size_t)nvalues * 8, s));
  DTB_TRY(launch_lower_bound(d_s.dptr, sorted.stype, nrows, d_v.dptr, nvalues, (int64_t*)d_out.dptr, s));
  if (d_out.staged()) { DTB_TRY(d_out.finish((size_t)nvalues * 8, s)); DTB_CUDA_CHECK(cudaStreamSynchronize(s)); }
  return DTB_OK;
}

}  // extern "C"
