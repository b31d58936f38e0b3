// libogbsampler.so -- host runtime + C-ABI (include/ogb_sampler.h) of the B200 replay sampler.
//
// Layering: ogb_dataset = the reference's Dataset (fields resident in HBM); ogb_sampler = GCDataset/HGCDataset
// (trajectory tables, key plan, Philox stream); ogb_batch = the dict sample() returns (one device block, one
// sub-array per key).  The kernels are in relabel_rows.cuh and gather_frames.cuh.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/ogb_sampler.h"
#include "gather_frames.cuh"
#include "relabel_rows.cuh"

namespace {

thread_local std::string g_error;

// Switches read once from the environment.  None of them is needed in production: each forces, for every input, a path
// that some real inputs take anyway, so that the tests can reach it with any dataset (test_gpu_rows.py runs each one in
// a process of its own against the default's batches).  Results are identical under every setting.
struct AbSwitches {
  bool no_records;       // OGB_NO_RECORDS      one array per field instead of the packed record table
  int fuse;              // OGB_FUSE=0|1        force the fused kernel off / on (-1: the built-in policy)
  bool gather_lsu;       // OGB_GATHER=lsu      register-staged gather kernel instead of the cp.async rings
  bool no_tiny_groups;   // OGB_NO_TINY_GROUPS  small fields copied one by one instead of grouped record loads
  bool timeline;         // OGB_TIMELINE        record an event per phase for ogb_debug_timeline
};

const AbSwitches& ab() {
  static const AbSwitches sw = [] {
    auto flag = [](const char* name) { return getenv(name) != nullptr; };
    const char* gather = getenv("OGB_GATHER");
    const char* fuse = getenv("OGB_FUSE");
    AbSwitches a;
    a.no_records = flag("OGB_NO_RECORDS");
    a.fuse = fuse ? atoi(fuse) : -1;
    a.gather_lsu = gather != nullptr && strcmp(gather, "lsu") == 0;
    a.no_tiny_groups = flag("OGB_NO_TINY_GROUPS");
    a.timeline = flag("OGB_TIMELINE");
    return a;
  }();
  return sw;
}
std::vector<cudaEvent_t> g_timeline;   // OGB_TIMELINE=1: four events per sample() call (index begin/end, gather begin/end)

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_error = buf;
  return code;
}

// No C++ exception may cross the C boundary (the callers are ctypes / cgo-style bindings): every entry point is a
// function-try-block that turns an exception into a status code and a message for ogb_last_error().
int fail_from_exception() {
  try {
    throw;
  } catch (const std::bad_alloc&) {
    return fail(OGB_ERR_UNSUPPORTED, "out of host memory");
  } catch (const std::exception& e) {
    return fail(OGB_ERR_INVALID, "internal error: %s", e.what());
  } catch (...) {
    return fail(OGB_ERR_INVALID, "internal error: unknown exception");
  }
}
#define OGB_CATCH_ALL catch (...) { return fail_from_exception(); }

#define OGB_CUDA(expr)                                                                                   \
  do {                                                                                                   \
    cudaError_t err_ = (expr);                                                                           \
    if (err_ != cudaSuccess) return fail(OGB_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(err_), \
                                         __FILE__, __LINE__);                                            \
  } while (0)

// The calling thread's current device is the caller's business: entry points switch to the dataset's device for their
// own calls and put the previous one back on the way out (a process that drives several GPUs from one thread --
// or a garbage-collected batch of another device's sampler -- must not find its device changed underfoot).
struct DeviceGuard {
  int previous = -1;
  cudaError_t status = cudaSuccess;
  explicit DeviceGuard(int device) {
    status = cudaGetDevice(&previous);
    if (status != cudaSuccess) { previous = -1; status = cudaSetDevice(device); return; }
    if (previous == device) previous = -1;          // nothing to switch, nothing to restore
    else status = cudaSetDevice(device);
  }
  ~DeviceGuard() {
    if (previous >= 0) cudaSetDevice(previous);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

#define OGB_TRY(expr)        \
  do {                       \
    int rc_ = (expr);        \
    if (rc_ != 0) return rc_; \
  } while (0)

size_t dtype_size(int dtype) {
  switch (dtype) {
    case OGB_U8: case OGB_I8: case OGB_BOOL: return 1;
    case OGB_I16: case OGB_F16: case OGB_U16: return 2;
    case OGB_I32: case OGB_F32: case OGB_U32: return 4;
    case OGB_I64: case OGB_F64: case OGB_U64: return 8;
    default: return 0;
  }
}

size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int largest_vec_log2(size_t a, size_t b) {  // largest power of two <= 16 dividing both
  int v = 4;
  while (v > 0 && ((a % ((size_t)1 << v)) != 0 || (b % ((size_t)1 << v)) != 0)) --v;
  return v;
}

// Row gathers: rows per item, the largest power of two whose rows fit the stage budget, so that the items of a 32-row
// tile are equal (an uneven split, e.g. 28 + 4 rows, makes the short item hold a pipeline slot for little data).
size_t rows_per_item(size_t pitch, size_t budget) {
  size_t r = 32;
  while (r > 1 && r * pitch > budget) r >>= 1;
  return r;
}

// Stage budget of a row-gather launch whose widest span is max_pitch bytes: 4 KB stages (2 CTAs per SM) for rows up to
// 256 bytes, 6 KB (16-row items, 1 CTA per SM) beyond -- C3's 384/288-byte spans run 15 % faster with 16-row items than
// with 8-row ones.
size_t stage_budget(size_t max_pitch) {
  return std::max<size_t>(max_pitch > 256 ? 6144 : 4096, max_pitch);
}

bool positive_at(const void* data, int dtype, int64_t i) {
  switch (dtype) {
    case OGB_U8: case OGB_BOOL: return ((const uint8_t*)data)[i] > 0;
    case OGB_I8: return ((const int8_t*)data)[i] > 0;
    case OGB_I16: return ((const int16_t*)data)[i] > 0;
    case OGB_U16: return ((const uint16_t*)data)[i] > 0;
    case OGB_I32: return ((const int32_t*)data)[i] > 0;
    case OGB_U32: return ((const uint32_t*)data)[i] > 0;
    case OGB_I64: return ((const int64_t*)data)[i] > 0;
    case OGB_U64: return ((const uint64_t*)data)[i] > 0;
    case OGB_F32: return ((const float*)data)[i] > 0.0f;
    case OGB_F64: return ((const double*)data)[i] > 0.0;
    default: return false;
  }
}

struct Field {
  std::string name;
  int dtype = 0;
  int ndim = 0;
  int64_t shape[OGB_MAX_NDIM] = {0};
  size_t itemsize = 0;
  size_t row_bytes = 0;
  size_t stride = 0;
  uint8_t* dptr = nullptr;
  bool in_record = false;  // dptr points into the dataset's packed record table (stride = record stride)
  size_t rec_off = 0;      // byte offset of this field inside a record
};

int shift_for(int64_t key_range, int64_t table_len) {
  // bucket width ~ half the mean gap between table entries, bounded so the bucket table stays <= 2^17 entries
  int shift = 4;
  const int64_t mean_gap = table_len > 0 ? std::max<int64_t>(1, key_range / table_len) : key_range;
  while (((int64_t)1 << (shift + 1)) < mean_gap / 2) ++shift;
  while ((key_range >> shift) > (1 << 17)) ++shift;
  return shift;
}

// bucket[b] = lower_bound(table, b << shift) for b in [0, (max_key >> shift) + 1]
std::vector<int32_t> build_buckets(const std::vector<int32_t>& table, int64_t max_key, int shift) {
  const int64_t nb = (max_key >> shift) + 2;
  std::vector<int32_t> bucket((size_t)nb);
  for (int64_t b = 0; b < nb; ++b) {
    const int64_t key = b << shift;
    bucket[(size_t)b] = (int32_t)(std::lower_bound(table.begin(), table.end(), key,
                                                  [](int32_t v, int64_t k) { return (int64_t)v < k; }) - table.begin());
  }
  return bucket;
}

template <typename T>
int upload_vector(const std::vector<T>& host, T** dptr, cudaStream_t stream = 0) {
  *dptr = nullptr;
  const size_t bytes = std::max<size_t>(host.size(), 1) * sizeof(T);
  OGB_CUDA(cudaMalloc((void**)dptr, bytes));
  if (!host.empty()) OGB_CUDA(cudaMemcpy(*dptr, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
  return 0;
}

// shadow[r] = observations[min(r + 1, n_rows - 1)] inside the record table (datasets.py:82), rows [row_begin, row_end)
__global__ void shadow_next_kernel(uint8_t* record_base, size_t stride, uint32_t obs_off, uint32_t shadow_off, uint32_t row_bytes,
                                   int64_t n_rows, int64_t row_begin, int64_t row_end) {
  const int64_t n = (row_end - row_begin) * row_bytes;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = row_begin + e / row_bytes, c = e % row_bytes;
    const int64_t src = r + 1 < n_rows ? r + 1 : n_rows - 1;
    record_base[(size_t)r * stride + shadow_off + c] = record_base[(size_t)src * stride + obs_off + c];
  }
}

__global__ void repad_rows_kernel(const uint8_t* __restrict__ dense, uint8_t* __restrict__ padded, int64_t n_rows,
                                  uint32_t row_bytes, uint32_t stride, int vec_log2) {
  const uint32_t epr = row_bytes >> vec_log2;
  const int64_t total = n_rows * epr;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / epr;
    const uint32_t c = (uint32_t)(e - r * epr);
    const uint8_t* s = dense + (size_t)e * ((size_t)1 << vec_log2);
    uint8_t* d = padded + (size_t)r * stride + ((size_t)c << vec_log2);
    switch (vec_log2) {
      case 2: *reinterpret_cast<uint32_t*>(d) = *reinterpret_cast<const uint32_t*>(s); break;
      case 1: *reinterpret_cast<uint16_t*>(d) = *reinterpret_cast<const uint16_t*>(s); break;
      default: *d = *s; break;
    }
  }
}

// ogb_sampler_write_ring: dense source rows [0, n_rows) of every field to rows (dst0 + i) mod ring_rows of the dataset's
// layout.  The host picks each field's access width (2^vec_log2 bytes, up to 16) so that the source, the destination base,
// the destination stride and the row length are all multiples of it.  n_rows <= ring_rows: every row is written once.
constexpr int kRingMaxFields = 64;
struct RingField {
  const uint8_t* src;
  uint8_t* dst;
  uint64_t stride;
  uint32_t row_bytes;
  uint32_t vec_log2;
};
struct RingParams {
  RingField f[kRingMaxFields];
  int n_fields;
};

template <typename T>
__device__ __forceinline__ void ring_copy_rows(const RingField& f, int64_t n_rows, int64_t dst0, int64_t ring_rows) {
  const uint32_t upr = f.row_bytes / (uint32_t)sizeof(T);
  const int64_t total = n_rows * upr;
  const T* src = reinterpret_cast<const T*>(f.src);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t r;
    uint32_t c;
    if (total <= 0x7fffffff) {               // (32-bit division for every launch short of 2^31 accesses per field)
      r = (uint32_t)e / upr;
      c = (uint32_t)e - (uint32_t)r * upr;
    } else {
      r = e / upr;
      c = (uint32_t)(e - r * upr);
    }
    int64_t d = dst0 + r;
    if (d >= ring_rows) d -= ring_rows;
    reinterpret_cast<T*>(f.dst + (size_t)d * f.stride)[c] = src[e];
  }
}

__global__ void ring_scatter_kernel(const __grid_constant__ RingParams p, int64_t n_rows, int64_t dst0, int64_t ring_rows) {
  for (int i = 0; i < p.n_fields; ++i) {
    const RingField& f = p.f[i];
    switch (f.vec_log2) {
      case 4: ring_copy_rows<uint4>(f, n_rows, dst0, ring_rows); break;
      case 3: ring_copy_rows<uint2>(f, n_rows, dst0, ring_rows); break;
      case 2: ring_copy_rows<uint32_t>(f, n_rows, dst0, ring_rows); break;
      case 1: ring_copy_rows<uint16_t>(f, n_rows, dst0, ring_rows); break;
      default: ring_copy_rows<uint8_t>(f, n_rows, dst0, ring_rows); break;
    }
  }
}

__global__ void searchsorted_warp_kernel(const int64_t* __restrict__ table, int64_t n, const int64_t* __restrict__ keys, int64_t m,
                                         int side_right, int64_t* __restrict__ out) {
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t k = warp; k < m; k += n_warps) {
    const int64_t pos = ogb::warp_searchsorted<int64_t>(table, n, keys[k], side_right != 0);
    if ((threadIdx.x & 31) == 0) out[k] = pos;
  }
}

__global__ void philox_fill_kernel(const __grid_constant__ ogb::RngKey key, uint64_t batch, uint32_t purpose, int64_t n, uint4* out) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x)
    out[r] = ogb::draw4(key, batch, (uint32_t)r, purpose);
}

// test helper: the float32 fast path of the geometric inversion against the float64 expression it stands for
__global__ void geometric_check_kernel(const __grid_constant__ ogb::RngKey key, double log_1mp, float abs_margin, int64_t n,
                                       unsigned long long* mismatches) {
  unsigned long long bad = 0;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const uint4 w = ogb::draw4(key, (uint64_t)(r >> 32), (uint32_t)r, 0);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t a = h ? w.z : w.x, b = h ? w.w : w.y;
      const double x = ceil(log(1.0 - ogb::unit_double(a, b)) / log_1mp);
      const int64_t want = x < 1.0 ? 1 : (int64_t)x;
      if (ogb::geometric_from_words(a, b, log_1mp, abs_margin) != want) ++bad;
    }
  }
  if (bad) atomicAdd(mismatches, bad);
}

enum Route { ROUTE_ROW = 0, ROUTE_FRAMES = 1, ROUTE_SCALAR = 2 };
enum ScalarKind {
  SC_MASKS = 0, SC_REWARDS, SC_HV_OFFSETS, SC_HV_STEPS, SC_HV_MASKS, SC_HV_REWARDS, SC_LV_STEPS, SC_LV_MASKS, SC_LV_REWARDS,
  SC_TRL_OFFSETS, SC_TRL_MID_OFFSETS, SC_COUNT
};

struct KeyPlan {
  std::string name;
  int route = ROUTE_ROW;
  int field = -1;
  int slot = 0;
  int fs = 1;
  bool crop = false;
  int scalar = -1;
  int dtype = 0;
  int ndim_tail = 0;
  int64_t tail[OGB_MAX_NDIM] = {0};
  size_t row_bytes = 0;
  int alias_of = -1;
};

struct DLDevice_ { int32_t device_type; int32_t device_id; };
struct DLDataType_ { uint8_t code; uint8_t bits; uint16_t lanes; };
struct DLTensor_ {
  void* data; DLDevice_ device; int32_t ndim; DLDataType_ dtype; int64_t* shape; int64_t* strides; uint64_t byte_offset;
};
struct DLManagedTensor_ {
  DLTensor_ dl_tensor; void* manager_ctx; void (*deleter)(struct DLManagedTensor_*);
};

}  // namespace

// ----------------------------------------------------------------------------------------------------------------
// Pinned double buffer of ogb_dataset_write_rows: block k is packed into host[k & 1] while block k - 1 is still on its way
// to dev[k & 1 ^ 1] (copy stream) or being repadded into the records (pack stream).
struct WriteStage {
  size_t bytes = 0;
  uint8_t* host[2] = {nullptr, nullptr};
  uint8_t* dev[2] = {nullptr, nullptr};
  cudaEvent_t copied[2] = {nullptr, nullptr}, packed[2] = {nullptr, nullptr};
  cudaStream_t copy = nullptr, pack = nullptr;
  uint64_t block = 0;
  ~WriteStage() {
    if (copy) cudaStreamSynchronize(copy);
    if (pack) cudaStreamSynchronize(pack);
    for (int b = 0; b < 2; ++b) {
      if (host[b]) cudaFreeHost(host[b]);
      if (dev[b]) cudaFree(dev[b]);
      if (copied[b]) cudaEventDestroy(copied[b]);
      if (packed[b]) cudaEventDestroy(packed[b]);
    }
    if (copy) cudaStreamDestroy(copy);
    if (pack) cudaStreamDestroy(pack);
  }
};

namespace {
// Two pinned host blocks and two device blocks of `bytes` each, their events, and a copy stream (and a pack stream when the
// blocks are unpacked on one of the stage's own).
int make_write_stage(size_t bytes, bool with_pack, std::unique_ptr<WriteStage>* out) {
  std::unique_ptr<WriteStage> st(new WriteStage());
  st->bytes = bytes;
  for (int b = 0; b < 2; ++b) {
    OGB_CUDA(cudaHostAlloc((void**)&st->host[b], bytes, cudaHostAllocDefault));
    OGB_CUDA(cudaMalloc((void**)&st->dev[b], bytes));
    OGB_CUDA(cudaEventCreateWithFlags(&st->copied[b], cudaEventDisableTiming));
    OGB_CUDA(cudaEventCreateWithFlags(&st->packed[b], cudaEventDisableTiming));
  }
  OGB_CUDA(cudaStreamCreateWithFlags(&st->copy, cudaStreamNonBlocking));
  if (with_pack) OGB_CUDA(cudaStreamCreateWithFlags(&st->pack, cudaStreamNonBlocking));
  *out = std::move(st);
  return 0;
}
}  // namespace

struct ogb_dataset {
  std::atomic<int> refs{1};
  int device = 0;
  int64_t capacity = 0;     // rows allocated
  int64_t size = 0;         // rows of the dataset (== capacity except for a dataset sealed with fewer rows)
  int64_t active_rows = 0;  // rows that hold data (== size except for a ReplayBuffer that is still filling up)
  // ogb_dataset_create_empty: the tables below are built by ogb_dataset_seal; no sampler is created before that
  bool sealed = true;
  std::unique_ptr<WriteStage> stage;
  // A view (ogb_dataset_view) shares the rows [row0, row0 + size) of `parent`'s memory -- its field pointers and
  // record_base are offset by row0 rows -- and holds a reference on it; its terminal and valid tables are its own.
  ogb_dataset* parent = nullptr;
  std::vector<Field> fields;    // the caller's fields, then (hidden, index >= n_public) the shadow field if there is one
  size_t n_public = 0;
  // Shadow copy of the NEXT row's observation inside every record (row r holds observations[min(r + 1, size - 1)],
  // datasets.py:82), kept for datasets whose observation row is <= 16 bytes and fits the record's padding: the
  // transition's next_observations then comes out of the record that is loaded anyway instead of costing a scattered
  // sector of its own (point-maze: 4 -> 3 sectors per transition).  -1: none.
  int shadow_next_field = -1;
  size_t record_used = 0;       // bytes of a record the fields occupy (before padding)
  int obs_field = -1, terminals_field = -1, valids_field = -1, next_obs_field = -1, oracle_field = -1;
  // valid rows
  int valid_mode = 0;  // 0 none, 1 table, 2 gaps
  int64_t n_valid = -1;
  int32_t* d_valid_table = nullptr;
  int32_t* d_gap_c = nullptr;
  int32_t* d_gap_bucket = nullptr;
  int gap_shift = 0;
  std::vector<int32_t> gaps_host;       // c[m] of valid_mode 2, kept for the sampler's segment table
  size_t table_bytes = 0;               // device bytes of the valid-row tables (part of resident_bytes)
  uint8_t* record_base = nullptr;       // packed record table: one record per row holding every small field
  size_t record_stride = 0;
  std::vector<uint8_t> terminals_host;  // terminals > 0, one byte per row (tiny next to the data)
  std::vector<uint8_t> valid_host;      // valids > 0 (empty when the dataset has no 'valids')
  size_t resident_bytes = 0;
  int sm_count = 148;

  // Pytree fields (the reference maps every gather over arbitrary pytrees, datasets.py:13,80,344,365-366): the host
  // wrapper flattens a nested dict into one field per leaf named "<key>/<path>".  Every leaf under "observations/" is an
  // observation: obs_field is the first of them (or the plain "observations" field), obs_extra the others.
  std::vector<int> obs_extra;

  int find(const char* name) const {
    for (size_t i = 0; i < fields.size(); ++i)
      if (fields[i].name == name) return (int)i;
    return -1;
  }
  static bool under(const std::string& field_name, const char* key) {   // the field is `key` itself or a leaf below it
    const size_t n = strlen(key);
    return field_name.compare(0, n, key) == 0 && (field_name.size() == n || field_name[n] == '/');
  }
  int find_under(const char* key) const {
    const int exact = find(key);
    if (exact >= 0) return exact;
    for (size_t i = 0; i < n_public && i < fields.size(); ++i)
      if (under(fields[i].name, key)) return (int)i;
    return -1;
  }
};

struct ogb_sampler {
  std::atomic<int> refs{1};
  ogb_dataset* ds = nullptr;
  ogb_config cfg{};
  int kind = 0;
  uint64_t seed = 0;
  uint32_t stream_id = 0;
  uint64_t counter = 0;
  cudaStream_t stream = nullptr;
  bool owns_stream = true;
  bool debug = false;
  bool defer_index_check = false;        // host-output mode: given indices are range-checked by the kernel, the error
                                         // surfaces at ogb_batch_copy_to_host / ogb_batch_sync instead of at sample()
  bool static_tiles = false;             // debug bit 3: row gathers walk their tiles with a fixed stride (no tickets)
  bool canary = false;                   // debug: fill every batch block with 0xA5 first, so that tests can verify that
                                         // no kernel wrote outside the keys (ogb_batch_check_gaps)
  bool profile = false;                  // record timing events around the dominant kernel of every call
  int host_chunks = 1;                   // > 1: big launches are issued in row chunks so that the D2H copy of a finished
                                         // chunk overlaps the kernels of the next (output='numpy' of the Python wrapper)
  cudaStream_t copy_stream = nullptr;
  // trajectory tables
  std::vector<int32_t> term_host;
  int32_t* d_term = nullptr;
  int32_t* d_term_bucket = nullptr;
  int term_shift = 0;
  double* d_neg_lut = nullptr;
  double* d_pow_lut = nullptr;
  // one-probe segment table (valid_mode 3): valid row AND final state from the same lookup
  int4* d_seg_table = nullptr;
  int32_t* d_seg_bucket = nullptr;
  int seg_shift = -1;                    // < 0: not available for this dataset
  int n_seg_table = 0, n_seg_bucket = 0;
  int n_slots = 0;
  std::vector<KeyPlan> plan[2];  // [evaluation]
  std::map<std::pair<int, int>, CUtensorMap> tmaps;  // (field, band_rows) -> descriptor
  std::mutex mu;
  // Batch blocks are recycled through this small per-sampler cache instead of going back to the driver: a block
  // released by the consumer is handed to a later sample() on the same stream (stream order makes that safe).
  struct AtcTable {
    std::vector<int32_t> host;
    int32_t* dev = nullptr;
  };
  std::map<int64_t, AtcTable> atc_tables;      // ATC anchor rows per temporal offset k (datasets.py:417-436)
  AtcTable trl_rows;                           // TRL: valid_idxs override = every non-terminal row (datasets.py:198-204)
  cudaStream_t aux_stream = nullptr;           // index kernels of chunked launches
  // Ticket counters of the row gathers' dynamic tile scheduling (relabel_rows.cuh): kSchedSlots pairs, one 128-byte line
  // each, handed out round-robin per launch.  A launch leaves its pair at zero, and launches of one stream run one after
  // the other, so a pair is only ever shared by launches that are kSchedSlots launches apart.
  int32_t* h_flags = nullptr;                  // pinned ring for the deferred index flags of copies in flight
  uint32_t flag_seq = 0;
  static constexpr int kFlagSlots = 64;
  static constexpr int kSchedSlots = 64;
  uint32_t* d_sched = nullptr;
  uint32_t sched_seq = 0;
  uint32_t* next_sched() { return d_sched + 32 * (size_t)(sched_seq++ % kSchedSlots); }
  std::vector<cudaEvent_t> chunk_events;       // ring of join events (index kernel -> gathers)
  int next_event = 0;
  std::mutex cache_mu;
  struct CachedBlock {
    size_t bytes;
    uint8_t* ptr;
    std::vector<cudaEvent_t> free_after;   // the block may be rewritten once these have fired
  };
  std::vector<CachedBlock> block_cache;
  size_t cache_bytes = 0;
  // ogb_sampler_write_ring: the pinned stage of host rows (host[b] -> dev[b] on the stage's copy stream, `packed[b]` =
  // the scatter that read dev[b] has finished), and the calls whose device sources may still be read
  std::unique_ptr<WriteStage> ring_stage;
  uint64_t ring_ticket = 0, ring_retired = 0;
  std::deque<std::pair<uint64_t, cudaEvent_t>> ring_in_flight;
  std::vector<cudaEvent_t> ring_spare_events;
};

struct ogb_batch {
  std::atomic<int> refs{1};
  ogb_sampler* sampler = nullptr;
  uint8_t* block = nullptr;
  size_t block_bytes = 0;
  size_t keys_bytes = 0;
  int64_t batch = 0, n_batches = 1, total_rows = 0;
  std::vector<KeyPlan> keys;
  std::vector<size_t> offsets;
  std::vector<std::string> names;
  int32_t* vec_rows = nullptr;
  int32_t* vec_init = nullptr;
  int8_t* crop = nullptr;
  int n_slots = 0;
  int launches = 0;
  bool keep_axis = false;               // report the leading n_batches axis even when n_batches == 1 (sample_many)
  std::vector<int64_t> chunk_end;                          // host-output pipelining: rows [chunk_end[c-1], chunk_end[c]) ...
  std::vector<cudaEvent_t> chunk_done;                     // ... are complete once chunk_done[c] has fired
  int32_t* idx_error = nullptr;                            // device flag of the deferred index check (inside the block)
  cudaEvent_t prof_begin = nullptr, prof_end = nullptr;   // profile mode: brackets of the dominant kernel
  const char* dominant = "";                               // its name, with the template arguments ncu prints, e.g.
                                                           // "relabel_gather_kernel<0, 0, 2, 20>" (static storage)
  std::vector<const char*> kernel_names;                   // every launch's kernel, in issue order (static storage)
  cudaEvent_t ready = nullptr;
  cudaEvent_t copied = nullptr;                            // ogb_batch_copy_to_host_begin: the D2H copy of the block has finished
  volatile int32_t* h_idx_flag = nullptr;                  // ... and where the deferred index flag lands (pinned, sampler-owned)
  std::vector<cudaStream_t> consumers;
  bool main_stream_consumer = false;  // somebody took the batch on the sampler's own stream
  bool escaped = false;               // a raw pointer left through __cuda_array_interface__: consumers unknown
  std::mutex mu;
};

namespace {

constexpr size_t kMaxCachedBlocks = 6;
constexpr int kMaxChunks = 8;
constexpr int64_t kOverlapMinRows = 32768;   // below this a call is latency bound and stays on one stream

size_t block_size_class(size_t bytes) {  // round up to 1/8-octave steps so that similar requests share blocks
  size_t cls = 4096;
  while (cls < bytes) cls <<= 1;
  const size_t step = cls / 16;
  return step == 0 ? cls : (bytes + step - 1) / step * step;
}

int block_take(ogb_sampler* s, size_t bytes, uint8_t** out, size_t* out_bytes, std::vector<cudaEvent_t>* free_after) {
  const size_t want = block_size_class(bytes);
  free_after->clear();
  {
    std::lock_guard<std::mutex> lock(s->cache_mu);
    for (size_t i = 0; i < s->block_cache.size(); ++i)
      if (s->block_cache[i].bytes == want) {
        *out = s->block_cache[i].ptr;
        *out_bytes = want;
        free_after->swap(s->block_cache[i].free_after);
        s->cache_bytes -= want;
        s->block_cache.erase(s->block_cache.begin() + (long)i);
        return 0;
      }
  }
  cudaError_t e = cudaMalloc((void**)out, want);
  if (e != cudaSuccess) {  // drop the cache and retry once before giving up
    std::vector<ogb_sampler::CachedBlock> drop;
    {
      std::lock_guard<std::mutex> lock(s->cache_mu);
      drop.swap(s->block_cache);
      s->cache_bytes = 0;
    }
    cudaGetLastError();
    cudaDeviceSynchronize();
    for (auto& blk : drop) {
      for (cudaEvent_t ev : blk.free_after) cudaEventDestroy(ev);
      cudaFree(blk.ptr);
    }
    e = cudaMalloc((void**)out, want);
  }
  if (e != cudaSuccess) { *out = nullptr; return fail(OGB_ERR_CUDA, "cudaMalloc(%zu) for a batch block: %s", want, cudaGetErrorString(e)); }
  *out_bytes = want;
  return 0;
}

int ensure_aux(ogb_sampler* s) {
  if (s->aux_stream) return 0;
  OGB_CUDA(cudaStreamCreateWithFlags(&s->aux_stream, cudaStreamNonBlocking));
  s->chunk_events.resize(1 + kMaxChunks + 1);
  for (auto& ev : s->chunk_events) OGB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  return 0;
}

// Orders `to` behind the work issued so far on `from`, through the next event of the sampler's join ring.
int join_streams(ogb_sampler* s, cudaStream_t from, cudaStream_t to) {
  cudaEvent_t ev = s->chunk_events[s->next_event];
  s->next_event = (s->next_event + 1) % (int)s->chunk_events.size();
  OGB_CUDA(cudaEventRecord(ev, from));
  OGB_CUDA(cudaStreamWaitEvent(to, ev, 0));
  return 0;
}

// Rows a start index is drawn from: those of `table` (TRL rows, ATC anchors) when there is one, else the valid rows
// (every row that holds data when the dataset has no 'valids').
int64_t n_choices_for(const ogb_dataset* ds, const int32_t* table, int64_t table_rows) {
  return table ? table_rows : (ds->valid_mode == 0 ? ds->active_rows : ds->n_valid);
}

void block_give(ogb_sampler* s, uint8_t* block, size_t bytes, std::vector<cudaEvent_t>&& free_after) {
  ogb_sampler::CachedBlock evict{0, nullptr, {}};
  {
    std::lock_guard<std::mutex> lock(s->cache_mu);
    s->block_cache.push_back({bytes, block, std::move(free_after)});
    s->cache_bytes += bytes;
    if (s->block_cache.size() > kMaxCachedBlocks) {
      evict = std::move(s->block_cache.front());
      s->cache_bytes -= evict.bytes;
      s->block_cache.erase(s->block_cache.begin());
    }
  }
  if (evict.ptr) {
    for (cudaEvent_t ev : evict.free_after) { cudaEventSynchronize(ev); cudaEventDestroy(ev); }
    cudaFree(evict.ptr);
  }
}

void free_valid_tables(ogb_dataset* ds) {
  if (ds->d_valid_table) cudaFree(ds->d_valid_table);
  if (ds->d_gap_c) cudaFree(ds->d_gap_c);
  if (ds->d_gap_bucket) cudaFree(ds->d_gap_bucket);
  ds->d_valid_table = ds->d_gap_c = ds->d_gap_bucket = nullptr;
  ds->resident_bytes -= ds->table_bytes;
  ds->table_bytes = 0;
}

void dataset_unref(ogb_dataset* ds) {
  if (ds->refs.fetch_sub(1) != 1) return;
  {
    DeviceGuard device_guard(ds->device);
    ds->stage.reset();
    if (!ds->parent) {            // a view's memory belongs to its parent
      for (auto& f : ds->fields) if (f.dptr && !f.in_record) cudaFree(f.dptr);
      if (ds->record_base) cudaFree(ds->record_base);
    }
    free_valid_tables(ds);
  }
  ogb_dataset* parent = ds->parent;
  delete ds;
  if (parent) dataset_unref(parent);
}

// Dataset.__init__ (datasets.py:62-63): valid_idxs = nonzero(valids > 0), from the host flags valid_host, as a table of the
// valid rows or, when at most one row in eight is invalid, as the ranks of the gaps (c[m] = (m-th invalid row) - m).
int build_valid_tables(ogb_dataset* ds) {
  free_valid_tables(ds);
  ds->valid_mode = 0;
  ds->n_valid = -1;
  ds->gaps_host.clear();
  if (ds->valids_field < 0) return 0;
  const int64_t size = ds->size;
  const std::vector<uint8_t>& valid = ds->valid_host;
  std::vector<int32_t> table, gaps;
  for (int64_t r = 0; r < size; ++r) {
    if (valid[(size_t)r]) table.push_back((int32_t)r);
    else gaps.push_back((int32_t)(r - (int64_t)gaps.size()));
  }
  ds->n_valid = (int64_t)table.size();
  if (ds->n_valid == 0) return fail(OGB_ERR_INVALID, "dataset has no valid rows");
  int rc = 0;
  if ((int64_t)gaps.size() * 8 <= size) {
    ds->valid_mode = 2;
    ds->gap_shift = shift_for(ds->n_valid + 1, (int64_t)gaps.size());
    std::vector<int32_t> bucket = build_buckets(gaps, ds->n_valid + 1, ds->gap_shift);
    rc = upload_vector(gaps, &ds->d_gap_c);
    if (!rc) rc = upload_vector(bucket, &ds->d_gap_bucket);
    ds->gaps_host = gaps;
    ds->table_bytes = (gaps.size() + bucket.size()) * 4;
  } else {
    ds->valid_mode = 1;
    rc = upload_vector(table, &ds->d_valid_table);
    ds->table_bytes = table.size() * 4;
  }
  ds->resident_bytes += ds->table_bytes;
  return rc;
}

// Everything ogb_dataset_create derives from the uploaded rows [0, size): the shadow next observation, the host flags of
// `terminals` and `valids`, and the valid-row tables.  ogb_dataset_seal runs the same after the rows have been written.
int build_tables(ogb_dataset* ds) {
  const int64_t size = ds->size;
  if (ds->fields.size() > ds->n_public) {       // the hidden shadow field (the only one)
    const Field& obs = ds->fields[(size_t)ds->obs_field];
    const Field& sh = ds->fields[ds->n_public];
    ds->shadow_next_field = (int)ds->n_public;
    shadow_next_kernel<<<ds->sm_count * 8, 256>>>(ds->record_base, ds->record_stride, (uint32_t)obs.rec_off, (uint32_t)sh.rec_off,
                                                   (uint32_t)obs.row_bytes, size, 0, size);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return fail(OGB_ERR_CUDA, "shadow fill: %s", cudaGetErrorString(e));
  }
  auto host_copy_1d = [&](int fi, std::vector<uint8_t>* flags) -> int {
    const Field& f = ds->fields[fi];
    if (f.row_bytes != f.itemsize) return fail(OGB_ERR_UNSUPPORTED, "field '%s' must be one value per row", f.name.c_str());
    std::vector<uint8_t> raw((size_t)size * f.row_bytes);
    OGB_CUDA(cudaMemcpy2D(raw.data(), f.row_bytes, f.dptr, f.stride, f.row_bytes, (size_t)size, cudaMemcpyDeviceToHost));
    flags->resize((size_t)size);
    for (int64_t r = 0; r < size; ++r) (*flags)[(size_t)r] = positive_at(raw.data(), f.dtype, r) ? 1 : 0;
    return 0;
  };
  ds->terminals_host.clear();
  ds->valid_host.clear();
  if (ds->terminals_field >= 0) OGB_TRY(host_copy_1d(ds->terminals_field, &ds->terminals_host));
  if (ds->valids_field >= 0) OGB_TRY(host_copy_1d(ds->valids_field, &ds->valid_host));
  return build_valid_tables(ds);
}

void sampler_unref(ogb_sampler* s) {
  if (s->refs.fetch_sub(1) != 1) return;
  DeviceGuard device_guard(s->ds->device);
  if (s->stream) cudaStreamSynchronize(s->stream);
  if (s->aux_stream) { cudaStreamSynchronize(s->aux_stream); cudaStreamDestroy(s->aux_stream); }
  if (s->copy_stream) { cudaStreamSynchronize(s->copy_stream); cudaStreamDestroy(s->copy_stream); }
  for (auto& ev : s->chunk_events) cudaEventDestroy(ev);
  for (auto& blk : s->block_cache) {
    for (cudaEvent_t ev : blk.free_after) cudaEventDestroy(ev);
    cudaFree(blk.ptr);
  }
  if (s->owns_stream && s->stream) cudaStreamDestroy(s->stream);
  for (auto& kv : s->atc_tables) if (kv.second.dev) cudaFree(kv.second.dev);
  if (s->trl_rows.dev) cudaFree(s->trl_rows.dev);
  if (s->d_term) cudaFree(s->d_term);
  if (s->d_term_bucket) cudaFree(s->d_term_bucket);
  if (s->d_seg_table) cudaFree(s->d_seg_table);
  if (s->d_seg_bucket) cudaFree(s->d_seg_bucket);
  if (s->d_sched) cudaFree(s->d_sched);
  if (s->h_flags) cudaFreeHost(s->h_flags);
  if (s->d_neg_lut) cudaFree(s->d_neg_lut);
  if (s->d_pow_lut) cudaFree(s->d_pow_lut);
  s->ring_stage.reset();
  for (auto& t : s->ring_in_flight) cudaEventDestroy(t.second);
  for (cudaEvent_t ev : s->ring_spare_events) cudaEventDestroy(ev);
  dataset_unref(s->ds);
  delete s;
}

void batch_unref(ogb_batch* b) {
  if (b->refs.fetch_sub(1) != 1) return;
  ogb_sampler* s = b->sampler;
  DeviceGuard device_guard(s->ds->device);
  // The block goes back to the sampler's cache together with the events after which it may be rewritten: the
  // batch's own `ready` event, plus one event per consumer stream that took the batch through the DLPack protocol.
  std::vector<cudaEvent_t> free_after;
  if (b->ready) {
    free_after.push_back(b->ready);
  } else if (b->block) {  // sample() failed half-way: nothing is known about in-flight work on the block
    cudaStreamSynchronize(s->stream);
    if (s->aux_stream) cudaStreamSynchronize(s->aux_stream);
  }
  for (cudaEvent_t ev : b->chunk_done) cudaEventDestroy(ev);
  if (b->copied) free_after.push_back(b->copied);   // a copy begun and never ended still reads the block
  if (b->prof_begin) cudaEventDestroy(b->prof_begin);
  if (b->prof_end) cudaEventDestroy(b->prof_end);
  if (b->escaped) cudaDeviceSynchronize();
  if (b->main_stream_consumer) b->consumers.push_back(s->stream);
  for (cudaStream_t c : b->consumers) {
    cudaEvent_t ev;
    if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) == cudaSuccess) {
      cudaEventRecord(ev, c);
      free_after.push_back(ev);
    }
  }
  if (b->block) block_give(s, b->block, b->block_bytes, std::move(free_after));
  else for (cudaEvent_t ev : free_after) cudaEventDestroy(ev);
  delete b;
  sampler_unref(s);
}

// Segment table of valid_mode 3 (relabel_rows.cuh, valid_row_fast).  Segment m = the valid rows that have exactly m
// invalid rows before them.  Usable when (a) two boundaries c[m] are never closer than 16 positions, so that buckets
// of 2^shift <= min gap positions hold at most one of them, and (b) no trajectory ends inside a segment before its
// last valid row, so that final_state_idxs (datasets.py:306) is one value per segment.  Anything else keeps the
// general searches.
int build_segment_table(ogb_sampler* s) {
  const ogb_dataset* ds = s->ds;
  if (ds->valid_mode != 2 || ds->gaps_host.empty()) return 0;
  const std::vector<int32_t>& c = ds->gaps_host;
  const size_t n_gaps = c.size();
  int64_t min_gap = ds->n_valid;
  for (size_t m = 0; m + 1 < n_gaps; ++m) min_gap = std::min<int64_t>(min_gap, (int64_t)c[m + 1] - c[m]);
  if (min_gap < 16) return 0;
  int shift = 4;
  while (((int64_t)1 << (shift + 1)) <= min_gap) ++shift;
  if ((ds->n_valid >> shift) > ((int64_t)1 << 22)) return 0;
  std::vector<int32_t> fin(n_gaps + 2);
  for (size_t m = 0; m <= n_gaps; ++m) {
    const int64_t first_row = m == 0 ? 0 : (int64_t)c[m - 1] + (int64_t)(m - 1) + 1;          // invalid row m-1 is c[m-1] + (m-1)
    const int64_t last_valid = m < n_gaps ? (int64_t)c[m] + (int64_t)m - 1 : ds->size - 1;
    if (first_row > last_valid) { fin[m] = (int32_t)std::min<int64_t>(first_row, ds->size - 1); continue; }  // empty: never looked up
    auto it = std::lower_bound(s->term_host.begin(), s->term_host.end(), (int32_t)first_row);
    if (it == s->term_host.end() || (int64_t)*it < last_valid) return 0;                        // (b) fails
    fin[m] = *it;
  }
  fin[n_gaps + 1] = fin[n_gaps];
  // one entry per bucket: everything a position in that bucket can need (valid_row_fast)
  const std::vector<int32_t> bucket = build_buckets(c, ds->n_valid + 1, shift);
  std::vector<int4> table(bucket.size());
  for (size_t bi = 0; bi < bucket.size(); ++bi) {
    const size_t lo = (size_t)bucket[bi];
    table[bi] = make_int4(lo < n_gaps ? c[lo] : 0x7fffffff, fin[lo], fin[lo + 1], (int)lo);
  }
  OGB_TRY(upload_vector(table, &s->d_seg_table));
  s->seg_shift = shift;
  s->n_seg_table = (int)table.size();
  s->n_seg_bucket = 0;
  return 0;
}

// ------------------------------------------------ key plan ------------------------------------------------
struct PlanBuilder {
  const ogb_dataset* ds;
  const ogb_config* cfg;
  bool crop_possible;
  int slot_canon[ogb::kMaxSlots];
  std::vector<KeyPlan> keys;

  int canonical(int slot) const { return slot_canon[slot]; }

  void push(KeyPlan k) {
    if (k.route != ROUTE_SCALAR && cfg->dedup_keys) {
      for (size_t i = 0; i < keys.size(); ++i) {
        const KeyPlan& o = keys[i];
        if (o.route != ROUTE_SCALAR && o.alias_of < 0 && o.field == k.field && o.slot == k.slot && o.fs == k.fs &&
            o.crop == k.crop) {
          k.alias_of = (int)i;
          break;
        }
      }
    }
    keys.push_back(std::move(k));
  }

  void alias(const char* name, const char* target) {   // every leaf of `target` (the key itself, or "target/<path>")
    const size_t n_before = keys.size();
    for (size_t i = 0; i < n_before; ++i)
      if (ogb_dataset::under(keys[i].name, target)) {
        KeyPlan k = keys[i];
        k.name = std::string(name) + keys[i].name.substr(strlen(target));
        k.alias_of = keys[i].alias_of >= 0 ? keys[i].alias_of : (int)i;
        keys.push_back(std::move(k));
      }
  }

  void field_key(const char* name, int field, int slot, bool in_aug, int fs = 1) {
    const Field& f = ds->fields[field];
    KeyPlan k;
    k.name = name;
    k.field = field;
    k.slot = canonical(slot);
    k.fs = fs;
    k.dtype = f.dtype;
    k.ndim_tail = f.ndim - 1;
    for (int d = 1; d < f.ndim; ++d) k.tail[d - 1] = f.shape[d];
    if (fs > 1) {
      if (k.ndim_tail == 0) { k.ndim_tail = 1; k.tail[0] = 1; }  // never happens for real data
      k.tail[k.ndim_tail - 1] *= fs;                               // np.concatenate(axis=-1)  datasets.py:366
    }
    k.row_bytes = f.row_bytes * fs;
    k.crop = in_aug && crop_possible && (f.ndim == 4);             // len(arr.shape) == 4  datasets.py:337
    k.route = (fs > 1 || k.crop) ? ROUTE_FRAMES : ROUTE_ROW;
    push(std::move(k));
  }
  // key `name` for observation leaf `field`: "value_goals" for the plain "observations" field, "value_goals/<path>" for the
  // leaf "observations/<path>" of a pytree
  std::string leaf_name(const char* name, int field) const {
    const std::string& f = ds->fields[(size_t)field].name;
    return f.size() > 12 && f.compare(0, 13, "observations/") == 0 ? std::string(name) + f.substr(12) : std::string(name);
  }
  void obs_key(const char* name, int slot, bool in_aug) {
    const int fs = cfg->frame_stack > 0 ? cfg->frame_stack : 1;
    field_key(leaf_name(name, ds->obs_field).c_str(), ds->obs_field, slot, in_aug, fs);
    for (int leaf : ds->obs_extra) field_key(leaf_name(name, leaf).c_str(), leaf, slot, in_aug, fs);
  }
  void goal_key(const char* name, int slot, bool in_aug) {  // datasets.py:348-357
    if (ds->oracle_field >= 0) field_key(name, ds->oracle_field, slot, in_aug);
    else obs_key(name, slot, in_aug);
  }
  void scalar_key(const char* name, int sc, int dtype) {
    KeyPlan k;
    k.name = name;
    k.route = ROUTE_SCALAR;
    k.scalar = sc;
    k.dtype = cfg->jax_compat ? (dtype == OGB_F64 ? OGB_F32 : OGB_I32) : dtype;   // what jit narrows them to with x64 off
    k.ndim_tail = 0;
    k.row_bytes = cfg->jax_compat ? 4 : 8;
    push(std::move(k));
  }
  void base_keys() {  // datasets.py:78-83 (+ :229-231)
    for (size_t i = 0; i < ds->n_public; ++i) {
      const std::string& nm = ds->fields[i].name;
      if ((int)i == ds->obs_field) obs_key("observations", ogb::SLOT_IDX, true);        // every observation leaf
      else if (ogb_dataset::under(nm, "observations")) continue;                        // (emitted with the first leaf)
      else field_key(nm.c_str(), (int)i, ogb::SLOT_IDX, ogb_dataset::under(nm, "next_observations"));
    }
    if (ds->next_obs_field < 0) {
      // observations[min(idx + 1, size - 1)] (datasets.py:82): from the record's shadow copy when there is one
      // (never with frame stacking, whose next_observations is the un-clamped idx + 1 through the stacker, :231)
      if (ds->shadow_next_field >= 0 && cfg->frame_stack <= 0) field_key("next_observations", ds->shadow_next_field, ogb::SLOT_IDX, true);
      else obs_key("next_observations", ogb::SLOT_NEXT, true);
    }
  }
};

std::vector<KeyPlan> build_plan(const ogb_sampler* s, bool evaluation) {
  using namespace ogb;
  PlanBuilder pb;
  pb.ds = s->ds;
  pb.cfg = &s->cfg;
  pb.crop_possible = s->cfg.has_p_aug && !evaluation && s->cfg.p_aug > 0.0 && s->kind != OGB_KIND_PLAIN;
  for (int v = 0; v < kMaxSlots; ++v) pb.slot_canon[v] = v;
  if (s->kind == OGB_KIND_HGC && s->cfg.dedup_keys) {
    if (s->cfg.low_subgoal_steps == s->cfg.value_subgoal_steps) pb.slot_canon[HGC_LV_NEXT] = HGC_HV_NEXT;
    if (s->cfg.low_subgoal_steps == s->cfg.actor_subgoal_steps) pb.slot_canon[HGC_LA_NEXT] = HGC_HA_NEXT;
  }
  if (s->kind == OGB_KIND_ATC) {                    // datasets.py:406-413
    pb.obs_key("observations", SLOT_IDX, true);
    pb.obs_key("positive_observations", SLOT_NEXT, true);
    return pb.keys;
  }
  pb.base_keys();
  if (s->kind == OGB_KIND_GC) {                     // datasets.py:248-252, aug list :280
    pb.goal_key("value_goals", GC_VALUE_GOAL, true);
    pb.goal_key("actor_goals", GC_ACTOR_GOAL, true);
    pb.scalar_key("masks", SC_MASKS, OGB_F64);
    pb.scalar_key("rewards", SC_REWARDS, OGB_F64);
    if (s->cfg.trl) {                               // datasets.py:254-276, aug list :281-291
      const int actions = s->ds->find("actions");
      pb.obs_key("value_goal_observations", GC_VALUE_GOAL, true);
      pb.obs_key("actor_goal_observations", GC_VALUE_GOAL, true);   // the reference gathers value_goal_idxs here too (:262)
      pb.scalar_key("value_offsets", SC_TRL_OFFSETS, OGB_I64);
      pb.scalar_key("value_midpoint_offsets", SC_TRL_MID_OFFSETS, OGB_I64);
      pb.obs_key("value_midpoint_observations", GC_TRL_MID, true);
      if (actions >= 0) {
        pb.field_key("value_midpoint_actions", actions, GC_TRL_MID, false);
        pb.field_key("next_actions", actions, GC_TRL_PLUS1, false);
      }
      pb.goal_key("value_midpoint_goals", GC_TRL_MID, true);
      pb.goal_key("value_cur_goals", SLOT_IDX, true);
      pb.goal_key("value_next_goals", GC_TRL_PLUS1, true);
    }
  } else if (s->kind == OGB_KIND_HGC) {             // datasets.py:526-619, aug list :625-640
    pb.obs_key("high_value_reps", SLOT_IDX, false);
    pb.goal_key("high_value_goals", HGC_HV_GOAL, true);
    pb.goal_key("high_value_actions", HGC_HV_NEXT, true);
    pb.obs_key("high_value_next_observations", HGC_HV_NEXT, true);
    pb.scalar_key("high_value_offsets", SC_HV_OFFSETS, OGB_I64);
    pb.scalar_key("high_value_subgoal_steps", SC_HV_STEPS, OGB_I64);
    pb.scalar_key("high_value_masks", SC_HV_MASKS, OGB_F64);
    pb.scalar_key("high_value_rewards", SC_HV_REWARDS, OGB_F64);
    pb.obs_key("low_value_next_observations", HGC_LV_NEXT, true);
    pb.scalar_key("low_value_subgoal_steps", SC_LV_STEPS, OGB_I64);
    pb.scalar_key("low_value_masks", SC_LV_MASKS, OGB_F64);
    pb.scalar_key("low_value_rewards", SC_LV_REWARDS, OGB_F64);
    if (s->cfg.has_low_discount) pb.goal_key("low_value_goals", HGC_LV_GOAL, false);
    pb.alias("value_goals", "high_value_goals");
    pb.scalar_key("masks", SC_MASKS, OGB_F64);
    pb.scalar_key("rewards", SC_REWARDS, OGB_F64);
    pb.goal_key("high_actor_goals", HGC_HA_GOAL, true);
    pb.goal_key("high_actor_actions", HGC_HA_NEXT, true);
    pb.obs_key("high_actor_next_observations", HGC_HA_NEXT, true);
    pb.alias("high_actor_targets", "high_actor_actions");
    pb.goal_key("low_actor_goals", HGC_LA_GOAL, true);
    pb.obs_key("low_actor_goal_observations", HGC_LA_GOAL, true);
    pb.obs_key("low_actor_next_observations", HGC_LA_NEXT, true);
  }
  return pb.keys;
}

// ------------------------------------------------ TMA descriptors ------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int get_encode_fn(EncodeTiledFn* out) {
  static EncodeTiledFn cached = nullptr;
  if (!cached) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    OGB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || fn == nullptr) return fail(OGB_ERR_CUDA, "cuTensorMapEncodeTiled not available");
    cached = (EncodeTiledFn)fn;
  }
  *out = cached;
  return 0;
}

bool tma_eligible(const Field& f, const ogb_config& cfg, int fs) {
  if (f.dtype != OGB_U8 || f.ndim != 4 || f.shape[3] != 3) return false;
  const int64_t H = f.shape[1], W = f.shape[2];
  if (W % ogb::kGroupPx != 0 || W * 3 > 256 || H < 8) return false;
  if (fs < 1 || fs > 4 || cfg.crop_padding > 4) return false;
  if (f.stride != f.row_bytes || (f.row_bytes % 16) != 0) return false;
  return true;
}

int band_rows_for(int64_t H, int pad) {
  for (int rb = 32; rb > pad; --rb)
    if (H % rb == 0) return rb;
  return 0;
}

int get_tmap(ogb_sampler* s, int field, int band_rows, CUtensorMap* out) {
  auto it = s->tmaps.find({field, band_rows});
  if (it != s->tmaps.end()) { *out = it->second; return 0; }
  EncodeTiledFn encode;
  OGB_TRY(get_encode_fn(&encode));
  const Field& f = s->ds->fields[field];
  const cuuint64_t H = (cuuint64_t)f.shape[1], rowb = (cuuint64_t)f.shape[2] * 3;
  cuuint64_t gdim[3] = {rowb, H, (cuuint64_t)s->ds->size};
  cuuint64_t gstr[2] = {rowb, (cuuint64_t)f.stride};
  cuuint32_t box[3] = {(cuuint32_t)rowb, (cuuint32_t)band_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMap tm;
  CUresult r = encode(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, f.dptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OGB_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  s->tmaps[{field, band_rows}] = tm;
  *out = tm;
  return 0;
}

}  // namespace

// ================================================================================================================
extern "C" {

const char* ogb_last_error(void) { return g_error.c_str(); }
int ogb_abi_version(void) { return OGB_ABI_VERSION; }

int ogb_device_count(int* out) try {
  if (!out) return fail(OGB_ERR_INVALID, "null out");
  OGB_CUDA(cudaGetDeviceCount(out));
  return 0;
} OGB_CATCH_ALL

// ogb_dataset_create (empty = false) and ogb_dataset_create_empty (empty = true: zero-filled fields of the same layout,
// tables left to ogb_dataset_seal)
static int create_dataset(const ogb_field* fields, int32_t n_fields, int32_t device, bool empty, ogb_dataset** out) {
  if (!fields || n_fields <= 0 || !out) return fail(OGB_ERR_INVALID, "ogb_dataset_create: bad arguments");
  DeviceGuard device_guard(device);
  OGB_CUDA(device_guard.status);
  ogb_dataset* ds = new ogb_dataset();
  ds->device = device;
  cudaDeviceGetAttribute(&ds->sm_count, cudaDevAttrMultiProcessorCount, device);
  int rc = 0;
  auto bail = [&](int code) { dataset_unref(ds); return code; };
  int64_t size = 0;
  for (int i = 0; i < n_fields; ++i) {
    const ogb_field& in = fields[i];
    if (!in.name || (!in.data && in.on_device != 2 && !empty) || in.ndim < 1 || in.ndim > OGB_MAX_NDIM || dtype_size(in.dtype) == 0)
      return bail(fail(OGB_ERR_INVALID, "field %d: bad descriptor", i));
    if (empty && in.data) return bail(fail(OGB_ERR_INVALID, "field '%s': an empty dataset takes no data", in.name));
    size = std::max<int64_t>(size, in.shape[0]);  // get_size: the longest leaf (datasets.py:11-14)
  }
  for (int i = 0; i < n_fields; ++i)
    if (fields[i].shape[0] != size)
      return bail(fail(OGB_ERR_INVALID, "field '%s' has %lld rows, dataset size is %lld", fields[i].name,
                       (long long)fields[i].shape[0], (long long)size));
  if (size < 1 || size > (int64_t)2147483000) return bail(fail(OGB_ERR_UNSUPPORTED, "dataset size %lld out of range", (long long)size));
  ds->capacity = ds->size = size;
  ds->active_rows = size;

  // ---- resident layout ----
  // Every field whose row is at most kRecordMaxRow bytes lives in ONE packed record per dataset row:
  //   [observations | other fields ...], sub-fields of more than 16 bytes on 16-byte offsets (cp.async sources), smaller
  //   ones on their natural alignment, the record padded to 32, 64 or a multiple of 128 bytes.
  // DRAM moves 64-byte granules, so a transition's own fields (observation, action, terminal, valid: datasets.py:78-83
  // gathers them all at the same row) then cost one aligned span instead of one granule each, and a goal row costs
  // ceil(obs_bytes / 64) granules.  Larger rows (image frames) keep an array of their own.
  constexpr size_t kRecordMaxRow = 2048, kRecordMaxBytes = 4096;
  const bool no_records = ab().no_records;
  std::vector<int> order;
  for (int i = 0; i < n_fields; ++i) {
    const ogb_field& in = fields[i];
    Field f;
    f.name = in.name;
    f.dtype = in.dtype;
    f.ndim = in.ndim;
    f.itemsize = dtype_size(in.dtype);
    size_t row = f.itemsize;
    for (int d = 0; d < in.ndim; ++d) {
      f.shape[d] = in.shape[d];
      if (d > 0) row *= (size_t)in.shape[d];
    }
    f.row_bytes = row;
    if (row == 0) return bail(fail(OGB_ERR_INVALID, "field '%s' has empty rows", in.name));
    if (row > 0xFFFFFFF0ull) return bail(fail(OGB_ERR_UNSUPPORTED, "field '%s': row too large", in.name));
    // a field outside the record: rows <= 16 B stay dense, longer rows start on a 32-byte sector boundary
    f.stride = row <= 16 ? row : round_up(row, 32);
    ds->fields.push_back(f);
    if (!no_records && row <= kRecordMaxRow) order.push_back(i);
  }
  {
    auto align_of = [](const Field& f) -> size_t {
      if (f.row_bytes > 16) return 16;
      size_t a = 16;
      while (f.row_bytes % a != 0) a >>= 1;
      return a;
    };
    // observations first (goal gathers read a prefix of the record), then by decreasing alignment
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
      const bool oa = ds->fields[(size_t)a].name == "observations", ob = ds->fields[(size_t)b].name == "observations";
      if (oa != ob) return oa;
      return align_of(ds->fields[(size_t)a]) > align_of(ds->fields[(size_t)b]);
    });
    size_t cursor = 0;
    std::vector<int> packed;
    for (int i : order) {
      Field& f = ds->fields[(size_t)i];
      const size_t off = round_up(cursor, align_of(f));
      if (off + f.row_bytes > kRecordMaxBytes) continue;      // does not fit any more: keeps its own array
      f.rec_off = off;
      f.in_record = true;
      cursor = off + f.row_bytes;
      packed.push_back(i);
    }
    if (packed.size() < 2) {                                   // nothing to share a record with
      for (int i : packed) ds->fields[(size_t)i].in_record = false;
    } else {
      // 32- and 64-byte records stay sector / granule sized; longer ones are padded to whole 128-byte L2 lines, so that a
      // goal row (a prefix of the record) never straddles a line (measured on the 156-byte C2 record: stride 256 is
      // 8 % faster than 160 or 192 and 3 % faster than separate arrays)
      ds->record_used = cursor;
      ds->record_stride = cursor <= 32 ? 32 : cursor <= 64 ? 64 : round_up(cursor, 128);
      const size_t bytes = (size_t)size * ds->record_stride;
      cudaError_t e = cudaMalloc((void**)&ds->record_base, bytes);
      if (e == cudaSuccess) e = cudaMemset(ds->record_base, 0, bytes);
      if (e != cudaSuccess) return bail(fail(OGB_ERR_CUDA, "cudaMalloc(%zu) for the record table: %s", bytes, cudaGetErrorString(e)));
      ds->resident_bytes += bytes;
      for (int i : packed) {
        Field& f = ds->fields[(size_t)i];
        f.dptr = ds->record_base + f.rec_off;
        f.stride = ds->record_stride;
      }
    }
  }
  for (int i = 0; i < n_fields; ++i) {
    const ogb_field& in = fields[i];
    Field& f = ds->fields[(size_t)i];
    const size_t row = f.row_bytes;
    const size_t dense_bytes = (size_t)size * row, padded_bytes = (size_t)size * f.stride;
    cudaError_t e = cudaSuccess;
    if (!f.in_record) {
      e = cudaMalloc((void**)&f.dptr, padded_bytes);
      if (e != cudaSuccess) return bail(fail(OGB_ERR_CUDA, "cudaMalloc(%zu) for field '%s': %s", padded_bytes, in.name, cudaGetErrorString(e)));
      ds->resident_bytes += padded_bytes;
    }
    const cudaMemcpyKind kind = in.on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (in.on_device == 2 || empty) {  // zero-filled buffer (ReplayBuffer.create, datasets.py:101-103)
      if (!f.in_record) {     // (the record table is zero-filled as a whole)
        e = cudaMemset(f.dptr, 0, padded_bytes);
        if (e != cudaSuccess) return bail(fail(OGB_ERR_CUDA, "memset of field '%s': %s", in.name, cudaGetErrorString(e)));
      }
    } else if (f.stride == row) {
      e = cudaMemcpy(f.dptr, in.data, dense_bytes, kind);
      if (e != cudaSuccess) return bail(fail(OGB_ERR_CUDA, "upload of field '%s': %s", in.name, cudaGetErrorString(e)));
    } else {
      const uint8_t* dense = (const uint8_t*)in.data;
      uint8_t* staging = nullptr;
      if (!in.on_device) {
        e = cudaMalloc((void**)&staging, dense_bytes);
        if (e == cudaSuccess) e = cudaMemcpy(staging, in.data, dense_bytes, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { if (staging) cudaFree(staging); return bail(fail(OGB_ERR_CUDA, "staging of field '%s': %s", in.name, cudaGetErrorString(e))); }
        dense = staging;
      }
      if (!f.in_record) cudaMemset(f.dptr, 0, padded_bytes);
      const int v = std::min(2, largest_vec_log2(row, 16));
      repad_rows_kernel<<<ds->sm_count * 8, 256>>>(dense, f.dptr, size, (uint32_t)row, (uint32_t)f.stride, v);
      e = cudaDeviceSynchronize();
      if (staging) cudaFree(staging);
      if (e != cudaSuccess) return bail(fail(OGB_ERR_CUDA, "repad of field '%s': %s", in.name, cudaGetErrorString(e)));
    }
  }
  ds->n_public = ds->fields.size();
  ds->obs_field = ds->find_under("observations");
  for (size_t i = 0; i < ds->n_public; ++i)
    if ((int)i != ds->obs_field && ogb_dataset::under(ds->fields[i].name, "observations")) ds->obs_extra.push_back((int)i);
  if (ds->obs_field >= 0 && ds->obs_extra.empty() && ds->find_under("next_observations") < 0) {
    const Field obs = ds->fields[(size_t)ds->obs_field];
    size_t a = 16;
    while (obs.row_bytes % a != 0) a >>= 1;
    const size_t off = round_up(ds->record_used, a);
    if (obs.in_record && obs.row_bytes <= 16 && off + obs.row_bytes <= ds->record_stride) {
      Field sh = obs;
      sh.name = "\x01next_observations";      // not a name a caller can pass
      sh.rec_off = off;
      sh.dptr = ds->record_base + off;
      ds->fields.push_back(sh);                // (filled by build_tables)
    }
  }
  ds->terminals_field = ds->find("terminals");
  ds->valids_field = ds->find("valids");
  ds->next_obs_field = ds->find_under("next_observations");
  ds->oracle_field = ds->find("oracle_reps");
  if (ds->obs_field < 0) return bail(fail(OGB_ERR_ASSERT, "assert 'observations' in data (datasets.py:54)"));
  if (empty) {
    ds->sealed = false;
    ds->active_rows = 0;
    // the zero fill (legacy stream) must be done before ogb_dataset_write_rows writes on its non-blocking streams
    const cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return bail(fail(OGB_ERR_CUDA, "zero fill: %s", cudaGetErrorString(e)));
  } else {
    rc = build_tables(ds);
    if (rc) return bail(rc);
  }
  *out = ds;
  return 0;
}

int ogb_dataset_create(const ogb_field* fields, int32_t n_fields, int32_t device, ogb_dataset** out) try {
  return create_dataset(fields, n_fields, device, false, out);
} OGB_CATCH_ALL

int ogb_dataset_size(const ogb_dataset* ds, int64_t* out) try {
  if (!ds || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = ds->size;
  return 0;
} OGB_CATCH_ALL
int ogb_dataset_set_active_rows(ogb_dataset* ds, int64_t n) try {
  if (!ds) return fail(OGB_ERR_INVALID, "null dataset");
  if (ds->parent) return fail(OGB_ERR_INVALID, "a view has no active rows of its own");
  if (n < 0 || n > ds->size) return fail(OGB_ERR_INVALID, "active rows must be in [0, %lld]", (long long)ds->size);
  ds->active_rows = n;
  // a buffer that is still filling up clamps idx + 1 at its CURRENT last row (datasets.py:82 with ReplayBuffer.size), which
  // a shadow written against the allocated size cannot express: such datasets gather next_observations by row
  if (n != ds->size) ds->shadow_next_field = -1;
  return 0;
} OGB_CATCH_ALL
int ogb_dataset_num_valid(const ogb_dataset* ds, int64_t* out) try {
  if (!ds || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = ds->n_valid;
  return 0;
} OGB_CATCH_ALL
int ogb_dataset_resident_bytes(const ogb_dataset* ds, size_t* out) try {
  if (!ds || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = ds->resident_bytes;
  return 0;
} OGB_CATCH_ALL
int ogb_dataset_destroy(ogb_dataset* ds) try {
  if (!ds) return fail(OGB_ERR_INVALID, "null dataset");
  dataset_unref(ds);
  return 0;
} OGB_CATCH_ALL

int ogb_dataset_create_empty(const ogb_field* fields, int32_t n_fields, int32_t device, ogb_dataset** out) try {
  return create_dataset(fields, n_fields, device, true, out);
} OGB_CATCH_ALL

int ogb_dataset_write_rows(ogb_dataset* ds, int64_t row0, int64_t n_rows, const void* const* field_rows, int32_t n_fields) try {
  if (!ds || !field_rows) return fail(OGB_ERR_INVALID, "ogb_dataset_write_rows: null argument");
  if (ds->parent) return fail(OGB_ERR_INVALID, "rows cannot be written through a view");
  if (ds->refs.load() > 1) return fail(OGB_ERR_INVALID, "the dataset is held by a sampler or a view: its rows cannot change under it");
  if (n_fields != (int32_t)ds->n_public) return fail(OGB_ERR_INVALID, "expected %zu field pointers", ds->n_public);
  if (row0 < 0 || n_rows < 0 || row0 + n_rows > ds->capacity)
    return fail(OGB_ERR_INDEX, "rows [%lld, %lld) exceed the capacity of %lld rows", (long long)row0, (long long)(row0 + n_rows),
                (long long)ds->capacity);
  DeviceGuard device_guard(ds->device);
  OGB_CUDA(device_guard.status);
  ds->sealed = false;             // the shadow and the tables no longer describe the rows
  if (n_rows == 0) return 0;
  if (!ds->stage) {
    constexpr size_t kStageBytes = (size_t)8 << 20;
    size_t bytes = kStageBytes;
    for (size_t i = 0; i < ds->n_public; ++i) bytes = std::max(bytes, ds->fields[i].row_bytes);
    OGB_TRY(make_write_stage(bytes, true, &ds->stage));
  }
  WriteStage& st = *ds->stage;
  for (size_t i = 0; i < ds->n_public; ++i) {
    if (!field_rows[i]) continue;
    const Field& f = ds->fields[i];
    const size_t row = f.row_bytes;
    const int64_t block_rows = (int64_t)(st.bytes / row);
    const uint8_t* src = (const uint8_t*)field_rows[i];
    const int v = std::min(2, largest_vec_log2(row, 16));
    for (int64_t r = 0; r < n_rows; r += block_rows) {
      const int64_t n = std::min(block_rows, n_rows - r);
      const int b = (int)(st.block++ & 1);
      OGB_CUDA(cudaEventSynchronize(st.copied[b]));     // the pinned buffer is free once its previous copy has finished
      memcpy(st.host[b], src + (size_t)r * row, (size_t)n * row);
      uint8_t* dst = f.dptr + (size_t)(row0 + r) * f.stride;
      if (f.stride == row) {                             // dense rows: straight into place
        OGB_CUDA(cudaMemcpyAsync(dst, st.host[b], (size_t)n * row, cudaMemcpyHostToDevice, st.copy));
        OGB_CUDA(cudaEventRecord(st.copied[b], st.copy));
      } else {                                           // padded rows: the copy of the next block runs under this repad
        OGB_CUDA(cudaStreamWaitEvent(st.copy, st.packed[b], 0));
        OGB_CUDA(cudaMemcpyAsync(st.dev[b], st.host[b], (size_t)n * row, cudaMemcpyHostToDevice, st.copy));
        OGB_CUDA(cudaEventRecord(st.copied[b], st.copy));
        OGB_CUDA(cudaStreamWaitEvent(st.pack, st.copied[b], 0));
        repad_rows_kernel<<<ds->sm_count * 8, 256, 0, st.pack>>>(st.dev[b], dst, n, (uint32_t)row, (uint32_t)f.stride, v);
        OGB_CUDA(cudaGetLastError());
        OGB_CUDA(cudaEventRecord(st.packed[b], st.pack));
      }
    }
  }
  OGB_CUDA(cudaStreamSynchronize(st.copy));
  OGB_CUDA(cudaStreamSynchronize(st.pack));
  return 0;
} OGB_CATCH_ALL

int ogb_dataset_seal(ogb_dataset* ds, int64_t n_rows) try {
  if (!ds) return fail(OGB_ERR_INVALID, "null dataset");
  if (ds->parent) return fail(OGB_ERR_INVALID, "a view is not sealed: its parent is");
  if (ds->refs.load() > 1) return fail(OGB_ERR_INVALID, "the dataset is held by a sampler or a view: it cannot be sealed again");
  if (n_rows < 1 || n_rows > ds->capacity)
    return fail(OGB_ERR_INVALID, "%lld rows do not fit the capacity of %lld rows", (long long)n_rows, (long long)ds->capacity);
  DeviceGuard device_guard(ds->device);
  OGB_CUDA(device_guard.status);
  ds->stage.reset();
  ds->sealed = false;
  ds->size = ds->active_rows = n_rows;
  OGB_TRY(build_tables(ds));
  ds->sealed = true;
  return 0;
} OGB_CATCH_ALL

int ogb_dataset_view(ogb_dataset* parent, int64_t row0, int64_t n_rows, ogb_dataset** out) try {
  if (!parent || !out) return fail(OGB_ERR_INVALID, "ogb_dataset_view: null argument");
  if (!parent->sealed) return fail(OGB_ERR_INVALID, "a view needs a sealed dataset");
  if (parent->active_rows != parent->size) return fail(OGB_ERR_INVALID, "a view needs a dataset whose rows are all written");
  if (row0 < 0 || n_rows < 1 || row0 + n_rows > parent->size)
    return fail(OGB_ERR_INVALID, "view rows [%lld, %lld) are outside the dataset's %lld rows", (long long)row0, (long long)(row0 + n_rows),
                (long long)parent->size);
  // The kernels assume of a field's base pointer what cudaMalloc gives and the layout keeps at every row of the full
  // table: 16-byte span, group and cp.async sources in the records and in padded arrays (also the TMA global address),
  // 32 bytes for the single 256-bit load of a 32-byte record (point-maze kernel), and the row's own power-of-two
  // alignment for the whole-row loads of dense rows of at most 16 bytes.
  auto misaligned = [&](const uint8_t* base, size_t stride, size_t need) {
    return ((uintptr_t)(base + (size_t)row0 * stride) % need) != 0;
  };
  if (parent->record_base && misaligned(parent->record_base, parent->record_stride, parent->record_stride == 32 ? 32 : 16))
    return fail(OGB_ERR_UNSUPPORTED, "view at row %lld: the record table would lose its alignment", (long long)row0);
  for (size_t i = 0; i < parent->n_public; ++i) {
    const Field& f = parent->fields[i];
    if (f.in_record) continue;    // (offsets inside a record whose base is aligned)
    const size_t need = f.row_bytes > 16 ? 16 : ((size_t)1 << largest_vec_log2(f.row_bytes, f.row_bytes));
    if (misaligned(f.dptr, f.stride, need))
      return fail(OGB_ERR_UNSUPPORTED, "view at row %lld: field '%s' would lose its %zu-byte alignment", (long long)row0, f.name.c_str(), need);
  }
  DeviceGuard device_guard(parent->device);
  OGB_CUDA(device_guard.status);
  ogb_dataset* v = new ogb_dataset();
  v->device = parent->device;
  v->sm_count = parent->sm_count;
  v->capacity = v->size = v->active_rows = n_rows;
  v->fields = parent->fields;
  for (Field& f : v->fields) f.dptr += (size_t)row0 * f.stride;
  v->n_public = parent->n_public;
  v->record_used = parent->record_used;
  v->record_stride = parent->record_stride;
  if (parent->record_base) v->record_base = parent->record_base + (size_t)row0 * parent->record_stride;
  v->obs_field = parent->obs_field;
  v->obs_extra = parent->obs_extra;
  v->terminals_field = parent->terminals_field;
  v->valids_field = parent->valids_field;
  v->next_obs_field = parent->next_obs_field;
  v->oracle_field = parent->oracle_field;
  // The parent's shadow of row r is observations[r + 1]: at a view's last row that is the next view's first observation,
  // not the clamp min(r + 1, n_rows - 1) of the view.  Only the view that ends where the parent ends keeps the shadow; the
  // others gather next_observations by row.
  v->shadow_next_field = row0 + n_rows == parent->size ? parent->shadow_next_field : -1;
  if (!parent->terminals_host.empty())
    v->terminals_host.assign(parent->terminals_host.begin() + row0, parent->terminals_host.begin() + row0 + n_rows);
  if (!parent->valid_host.empty())
    v->valid_host.assign(parent->valid_host.begin() + row0, parent->valid_host.begin() + row0 + n_rows);
  v->parent = parent;
  parent->refs.fetch_add(1);
  const int rc = build_valid_tables(v);
  if (rc) { dataset_unref(v); return rc; }
  *out = v;
  return 0;
} OGB_CATCH_ALL

int ogb_sampler_create(ogb_dataset* ds, const ogb_config* cfg, int32_t kind, uint64_t seed, uint32_t stream_id, ogb_sampler** out) try {
  if (!ds || !cfg || !out) return fail(OGB_ERR_INVALID, "ogb_sampler_create: null argument");
  if (kind < OGB_KIND_GC || kind > OGB_KIND_ATC) return fail(OGB_ERR_INVALID, "unknown sampler kind %d", kind);
  if (stream_id >= (1u << 24)) return fail(OGB_ERR_INVALID, "stream_id must be < 2^24");
  // a row's crop shift is stored as int8 (dy, dx) with -128 meaning "not augmented"
  if (cfg->crop_padding < 0 || cfg->crop_padding > 127) return fail(OGB_ERR_INVALID, "crop padding %d out of [0, 127]", cfg->crop_padding);
  if (!ds->sealed) return fail(OGB_ERR_INVALID, "the dataset is not sealed: its rows are still being written (ogb_dataset_seal)");
  DeviceGuard device_guard(ds->device);
  OGB_CUDA(device_guard.status);
  if (kind == OGB_KIND_ATC) {
    if (ds->terminals_field < 0) return fail(OGB_ERR_INVALID, "KeyError: 'terminals'");
    if (cfg->frame_stack > 0 && ds->next_obs_field >= 0)
      return fail(OGB_ERR_ASSERT, "frame_stack needs a compact dataset: 'next_observations' present (datasets.py:396)");
  } else if (kind != OGB_KIND_PLAIN) {
    if (ds->terminals_field < 0) return fail(OGB_ERR_INVALID, "KeyError: 'terminals'");
    auto close1 = [](double x) { return std::fabs(x - 1.0) <= 1e-8 + 1e-5; };  // np.isclose(x, 1.0)
    if (!close1(cfg->value_p_curgoal + cfg->value_p_trajgoal + cfg->value_p_randomgoal))
      return fail(OGB_ERR_ASSERT, "value_p_* do not sum to 1 (datasets.py:191-193)");
    if (!close1(cfg->actor_p_curgoal + cfg->actor_p_trajgoal + cfg->actor_p_randomgoal))
      return fail(OGB_ERR_ASSERT, "actor_p_* do not sum to 1 (datasets.py:194-196)");
    if (cfg->frame_stack > 0 && ds->next_obs_field >= 0)
      return fail(OGB_ERR_ASSERT, "frame_stack needs a compact dataset: 'next_observations' present (datasets.py:208)");
    if (cfg->frame_stack < 0 || cfg->frame_stack > 64) return fail(OGB_ERR_INVALID, "frame_stack out of range");
    if (!(cfg->discount > 0.0 && cfg->discount < 1.0)) return fail(OGB_ERR_INVALID, "discount must be in (0, 1)");
    if (cfg->has_low_discount && !(cfg->low_discount > 0.0 && cfg->low_discount < 1.0))
      return fail(OGB_ERR_INVALID, "low_discount must be in (0, 1)");
    if (kind == OGB_KIND_HGC) {
      const int kmax = std::max({cfg->value_subgoal_steps, cfg->actor_subgoal_steps, cfg->low_subgoal_steps});
      if (cfg->value_subgoal_steps < 0 || cfg->actor_subgoal_steps < 0 || cfg->low_subgoal_steps < 0)
        return fail(OGB_ERR_INVALID, "subgoal steps must be >= 0");
      if (!cfg->neg_reward_lut || !cfg->pow_lut || cfg->lut_len < kmax + 1)
        return fail(OGB_ERR_INVALID, "reward tables must cover steps 0..%d", kmax);
    }
  }
  ogb_sampler* s = new ogb_sampler();
  s->ds = ds;
  ds->refs.fetch_add(1);
  s->cfg = *cfg;
  s->cfg.neg_reward_lut = nullptr;
  s->cfg.pow_lut = nullptr;
  s->kind = kind;
  s->seed = seed;
  s->stream_id = stream_id;
  auto bail = [&](int code) { sampler_unref(s); return code; };
  if (cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(fail(OGB_ERR_CUDA, "cudaStreamCreate failed"));

  if (kind != OGB_KIND_PLAIN) {
    // terminal_locs = nonzero(terminals > 0)  (datasets.py:186)
    for (int64_t r = 0; r < ds->size; ++r)
      if (ds->terminals_host[(size_t)r]) s->term_host.push_back((int32_t)r);
    if (s->term_host.empty() || s->term_host.back() != ds->size - 1)
      return bail(fail(OGB_ERR_ASSERT, "assert terminal_locs[-1] == size - 1 (datasets.py:188)"));
    s->term_shift = shift_for(ds->size, (int64_t)s->term_host.size());
    std::vector<int32_t> bucket = build_buckets(s->term_host, ds->size, s->term_shift);
    int rc = upload_vector(s->term_host, &s->d_term);
    if (!rc) rc = upload_vector(bucket, &s->d_term_bucket);
    if (rc) return bail(rc);
    {
      int rc2 = build_segment_table(s);
      if (rc2) return bail(rc2);
    }
    if (kind == OGB_KIND_GC && cfg->trl == 1) {  // datasets.py:198-204: arange(cur, terminal) for every terminal row
      for (int64_t r = 0; r < ds->size; ++r)
        if (!ds->terminals_host[(size_t)r]) s->trl_rows.host.push_back((int32_t)r);
      if (s->trl_rows.host.empty()) return bail(fail(OGB_ERR_INVALID, "TRL: the dataset has no non-terminal row"));
      rc = upload_vector(s->trl_rows.host, &s->trl_rows.dev);
      if (rc) return bail(rc);
    }
    if (kind == OGB_KIND_HGC) {
      std::vector<double> neg(cfg->neg_reward_lut, cfg->neg_reward_lut + cfg->lut_len), pw(cfg->pow_lut, cfg->pow_lut + cfg->lut_len);
      rc = upload_vector(neg, &s->d_neg_lut);
      if (!rc) rc = upload_vector(pw, &s->d_pow_lut);
      if (rc) return bail(rc);
    }
  }
  s->n_slots = kind == OGB_KIND_GC ? (cfg->trl ? ogb::GC_TRL_NUM_SLOTS : ogb::GC_NUM_SLOTS) : (kind == OGB_KIND_HGC ? ogb::HGC_NUM_SLOTS : 2);
  s->plan[0] = build_plan(s, false);
  s->plan[1] = build_plan(s, true);
  // ticket counters of the row gathers, zeroed once: every launch leaves its pair at zero
  if (cudaMalloc((void**)&s->d_sched, (size_t)ogb_sampler::kSchedSlots * 128) != cudaSuccess ||
      cudaMemset(s->d_sched, 0, (size_t)ogb_sampler::kSchedSlots * 128) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess)
    return bail(fail(OGB_ERR_CUDA, "ticket counters: %s", cudaGetErrorString(cudaGetLastError())));
  *out = s;
  return 0;
} OGB_CATCH_ALL

int ogb_sampler_set_stream(ogb_sampler* s, void* cuda_stream) try {
  if (!s) return fail(OGB_ERR_INVALID, "null sampler");
  DeviceGuard device_guard(s->ds->device);
  OGB_CUDA(device_guard.status);
  std::lock_guard<std::mutex> lock(s->mu);
  if (s->stream) cudaStreamSynchronize(s->stream);  // cached blocks may still be in flight on the old stream
  if (s->aux_stream) cudaStreamSynchronize(s->aux_stream);
  if (s->owns_stream && s->stream) cudaStreamDestroy(s->stream);
  s->stream = (cudaStream_t)cuda_stream;
  s->owns_stream = false;
  return 0;
} OGB_CATCH_ALL
int ogb_sampler_set_host_chunks(ogb_sampler* s, int32_t n_chunks) try {
  if (!s) return fail(OGB_ERR_INVALID, "null sampler");
  if (n_chunks < 1 || n_chunks > kMaxChunks) return fail(OGB_ERR_INVALID, "n_chunks must be in [1, %d]", kMaxChunks);
  s->host_chunks = n_chunks;
  return 0;
} OGB_CATCH_ALL
int ogb_sampler_set_deferred_index_check(ogb_sampler* s, int32_t on) try {
  if (!s) return fail(OGB_ERR_INVALID, "null sampler");
  s->defer_index_check = on != 0;
  return 0;
} OGB_CATCH_ALL
int ogb_sampler_set_profile(ogb_sampler* s, int32_t on) try {
  if (!s) return fail(OGB_ERR_INVALID, "null sampler");
  s->profile = on != 0;
  return 0;
} OGB_CATCH_ALL
int ogb_sampler_set_debug(ogb_sampler* s, int32_t keep) try {
  if (!s) return fail(OGB_ERR_INVALID, "null sampler");
  if (keep & ~11) return fail(OGB_ERR_INVALID, "debug flags 0x%x: only bits 0, 1 and 3 are defined", (unsigned)keep);
  s->debug = (keep & 1) != 0;
  s->canary = (keep & 2) != 0;
  s->static_tiles = (keep & 8) != 0;
  return 0;
} OGB_CATCH_ALL
int ogb_sampler_num_choices(const ogb_sampler* s, int64_t* out) try {
  if (!s || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = n_choices_for(s->ds, s->trl_rows.dev, (int64_t)s->trl_rows.host.size());
  return 0;
} OGB_CATCH_ALL

// ReplayBuffer.add_transition (datasets.py:134-142): overwrite row `row` of every field, ordered on the sampler's
// stream after the sample() calls already issued and before the ones that follow.
int ogb_sampler_write_row(ogb_sampler* s, int64_t row, const void* const* field_rows, int32_t n_fields) try {
  if (!s || !field_rows) return fail(OGB_ERR_INVALID, "null argument");
  ogb_dataset* ds = s->ds;
  if (ds->parent) return fail(OGB_ERR_INVALID, "rows cannot be written through a view");
  if (row < 0 || row >= ds->size) return fail(OGB_ERR_INDEX, "row %lld out of range", (long long)row);
  if (n_fields != (int32_t)ds->n_public) return fail(OGB_ERR_INVALID, "expected %zu field pointers", ds->n_public);
  DeviceGuard device_guard(ds->device);
  OGB_CUDA(device_guard.status);
  std::lock_guard<std::mutex> lock(s->mu);
  // index kernels of big launches read tiny fields on the auxiliary stream
  if (s->aux_stream) OGB_TRY(join_streams(s, s->aux_stream, s->stream));
  for (size_t i = 0; i < ds->n_public; ++i) {
    if (!field_rows[i]) continue;
    const Field& f = ds->fields[i];
    OGB_CUDA(cudaMemcpyAsync(f.dptr + (size_t)row * f.stride, field_rows[i], f.row_bytes, cudaMemcpyHostToDevice, s->stream));
  }
  if (ds->shadow_next_field >= 0 && field_rows[ds->obs_field]) {
    // keep the shadow coherent: row r-1 shadows row r, and the last row shadows itself (stream-ordered behind the copy)
    const Field& sh = ds->fields[(size_t)ds->shadow_next_field];
    const Field& obs = ds->fields[(size_t)ds->obs_field];
    const int64_t begin = row > 0 ? row - 1 : row, end = row == ds->size - 1 ? row + 1 : row;
    if (end > begin) {
      shadow_next_kernel<<<1, 32, 0, s->stream>>>(ds->record_base, ds->record_stride, (uint32_t)obs.rec_off, (uint32_t)sh.rec_off,
                                                  (uint32_t)obs.row_bytes, ds->size, begin, end);
      if (cudaGetLastError() != cudaSuccess) return fail(OGB_ERR_CUDA, "shadow update launch failed");
    }
  }
  return 0;
} OGB_CATCH_ALL

int ogb_sampler_get_stream(const ogb_sampler* s, void** out) try {
  if (!s || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = (void*)s->stream;
  return 0;
} OGB_CATCH_ALL

// ReplayBuffer.add_transition for n transitions at once (datasets.py:134-142): source row i -> row (row0 + i) mod size for
// i in [skip, n), every field in one ring_scatter_kernel launch per stage block, ordered on the sampler's stream like
// ogb_sampler_write_row.  Host rows are packed into the pinned stage (block k + 1 is packed and copied while block k is
// scattered); device rows are read in place.
int ogb_sampler_write_ring(ogb_sampler* s, int64_t row0, int64_t n, int64_t skip, const void* const* field_rows, int32_t n_fields,
                           const int32_t* on_device, void* producer_stream, uint64_t* out_ticket, uint64_t* out_retired) try {
  if (!s || !field_rows || !out_ticket || !out_retired) return fail(OGB_ERR_INVALID, "null argument");
  ogb_dataset* ds = s->ds;
  if (ds->parent) return fail(OGB_ERR_INVALID, "rows cannot be written through a view");
  const int64_t ring = ds->size;
  if (row0 < 0 || row0 >= ring) return fail(OGB_ERR_INDEX, "row0 %lld out of [0, %lld)", (long long)row0, (long long)ring);
  if (n < 0 || skip < 0 || skip > n) return fail(OGB_ERR_INVALID, "need 0 <= skip <= n (got n = %lld, skip = %lld)", (long long)n, (long long)skip);
  if (n - skip > ring)
    return fail(OGB_ERR_INVALID, "%lld rows exceed the %lld-row ring: only the last %lld can survive (skip = n - size)",
                (long long)(n - skip), (long long)ring, (long long)ring);
  if (n_fields != (int32_t)ds->n_public) return fail(OGB_ERR_INVALID, "expected %zu field pointers", ds->n_public);
  DeviceGuard device_guard(ds->device);
  OGB_CUDA(device_guard.status);
  const int64_t rows = n - skip;
  std::vector<int> write;                 // fields with a source
  size_t host_row_bytes = 0;              // bytes of one row of every host source
  bool any_device = false;
  for (size_t i = 0; i < ds->n_public; ++i) {
    if (!field_rows[i]) continue;
    write.push_back((int)i);
    if (!on_device || !on_device[i]) {
      host_row_bytes += ds->fields[i].row_bytes;
      continue;
    }
    cudaPointerAttributes attr{};
    if (cudaPointerGetAttributes(&attr, field_rows[i]) != cudaSuccess) {
      cudaGetLastError();
      attr.type = cudaMemoryTypeUnregistered;
    }
    if ((attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) || attr.device != ds->device)
      return fail(OGB_ERR_INVALID, "field '%s': the source is not device memory of device %d", ds->fields[i].name.c_str(), ds->device);
    any_device = true;
  }
  std::lock_guard<std::mutex> lock(s->mu);
  while (!s->ring_in_flight.empty()) {    // calls whose scatter has finished no longer read their device sources
    const cudaError_t q = cudaEventQuery(s->ring_in_flight.front().second);
    if (q == cudaErrorNotReady) break;
    if (q != cudaSuccess) return fail(OGB_ERR_CUDA, "ring write event: %s", cudaGetErrorString(q));
    s->ring_spare_events.push_back(s->ring_in_flight.front().second);
    s->ring_in_flight.pop_front();
  }
  auto take_event = [&](cudaEvent_t* ev) -> int {
    if (!s->ring_spare_events.empty()) {
      *ev = s->ring_spare_events.back();
      s->ring_spare_events.pop_back();
      return 0;
    }
    OGB_CUDA(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
    return 0;
  };
  const uint64_t ticket = ++s->ring_ticket;
  if (rows > 0) {
    // index kernels of big launches read tiny fields on the auxiliary stream
    if (s->aux_stream) OGB_TRY(join_streams(s, s->aux_stream, s->stream));
    if (any_device && producer_stream && producer_stream != (void*)s->stream) {
      cudaEvent_t ev;
      OGB_TRY(take_event(&ev));
      s->ring_spare_events.push_back(ev);   // (a wait takes the event's state when it is issued: free again right away)
      OGB_CUDA(cudaEventRecord(ev, (cudaStream_t)producer_stream));
      OGB_CUDA(cudaStreamWaitEvent(s->stream, ev, 0));
    }
    WriteStage* st = nullptr;
    int64_t block_rows = rows;
    if (host_row_bytes > 0) {
      if (!s->ring_stage) {
        size_t all = 0;
        for (size_t i = 0; i < ds->n_public; ++i) all += round_up(ds->fields[i].row_bytes, 16);
        OGB_TRY(make_write_stage(std::max<size_t>((size_t)8 << 20, all), false, &s->ring_stage));
      }
      st = s->ring_stage.get();
      block_rows = std::max<int64_t>(1, (int64_t)((st->bytes - 16 * write.size()) / host_row_bytes));
    }
    std::vector<size_t> stage_off(ds->n_public, 0);
    for (int64_t r = 0; r < rows; r += block_rows) {
      const int64_t k = std::min(block_rows, rows - r);
      int b = 0;
      if (st) {
        b = (int)(st->block++ & 1);
        OGB_CUDA(cudaEventSynchronize(st->copied[b]));     // host[b] is free once its previous copy has finished
        size_t off = 0;
        for (int i : write) {
          if (on_device && on_device[i]) continue;
          const size_t row = ds->fields[(size_t)i].row_bytes;
          memcpy(st->host[b] + off, (const uint8_t*)field_rows[i] + (size_t)(skip + r) * row, (size_t)k * row);
          stage_off[(size_t)i] = off;
          off = round_up(off + (size_t)k * row, 16);
        }
        OGB_CUDA(cudaStreamWaitEvent(st->copy, st->packed[b], 0));   // dev[b] is free once the scatter that read it has run
        OGB_CUDA(cudaMemcpyAsync(st->dev[b], st->host[b], off, cudaMemcpyHostToDevice, st->copy));
        OGB_CUDA(cudaEventRecord(st->copied[b], st->copy));
        OGB_CUDA(cudaStreamWaitEvent(s->stream, st->copied[b], 0));
      }
      for (size_t g = 0; g < write.size(); g += kRingMaxFields) {
        RingParams p{};
        p.n_fields = (int)std::min<size_t>(kRingMaxFields, write.size() - g);
        int64_t max_units = 1;
        for (int j = 0; j < p.n_fields; ++j) {
          const int i = write[g + (size_t)j];
          const Field& f = ds->fields[(size_t)i];
          const bool dev = on_device && on_device[i];
          const uint8_t* src = dev ? (const uint8_t*)field_rows[i] + (size_t)(skip + r) * f.row_bytes : st->dev[b] + stage_off[(size_t)i];
          int v = 4;     // the widest access that divides the row, both bases and the destination stride
          const uint64_t bits = (uint64_t)f.row_bytes | (uint64_t)f.stride | (uint64_t)(uintptr_t)f.dptr | (uint64_t)(uintptr_t)src;
          while (v > 0 && (bits & ((1ull << v) - 1)) != 0) --v;
          p.f[j] = RingField{src, f.dptr, (uint64_t)f.stride, (uint32_t)f.row_bytes, (uint32_t)v};
          max_units = std::max<int64_t>(max_units, k * (int64_t)(f.row_bytes >> v));
        }
        const int grid = (int)std::min<int64_t>((int64_t)ds->sm_count * 8, (max_units + 255) / 256);
        ring_scatter_kernel<<<grid, 256, 0, s->stream>>>(p, k, (row0 + skip + r) % ring, ring);
        OGB_CUDA(cudaGetLastError());
      }
      if (st) OGB_CUDA(cudaEventRecord(st->packed[b], s->stream));
    }
    if (any_device) {
      cudaEvent_t ev;
      OGB_TRY(take_event(&ev));
      OGB_CUDA(cudaEventRecord(ev, s->stream));
      s->ring_in_flight.emplace_back(ticket, ev);
    }
    if (ds->shadow_next_field >= 0 && field_rows[ds->obs_field]) {
      // row r shadows row r + 1, so the written rows' predecessors change, and the last row shadows itself.  Not fused into
      // the scatter: row r's shadow reads row r + 1, which another CTA may still be writing.
      const Field& sh = ds->fields[(size_t)ds->shadow_next_field];
      const Field& obs = ds->fields[(size_t)ds->obs_field];
      const int64_t dst0 = (row0 + skip) % ring, end = dst0 + rows;
      int64_t seg[2][2] = {{0, ring}, {0, 0}};
      if (rows < ring) {
        seg[0][0] = std::max<int64_t>(dst0 - 1, 0);
        seg[0][1] = std::min(end, ring);
        if (end > ring) seg[1][1] = end - ring;
      }
      for (auto& sg : seg) {
        if (sg[1] <= sg[0]) continue;
        const int grid = (int)std::min<int64_t>((int64_t)ds->sm_count * 8, ((sg[1] - sg[0]) * (int64_t)obs.row_bytes + 255) / 256);
        shadow_next_kernel<<<grid, 256, 0, s->stream>>>(ds->record_base, ds->record_stride, (uint32_t)obs.rec_off, (uint32_t)sh.rec_off,
                                                         (uint32_t)obs.row_bytes, ds->size, sg[0], sg[1]);
        OGB_CUDA(cudaGetLastError());
      }
    }
  }
  *out_ticket = ticket;
  *out_retired = s->ring_in_flight.empty() ? ticket : s->ring_in_flight.front().first - 1;
  return 0;
} OGB_CATCH_ALL

int ogb_sampler_num_terminals(const ogb_sampler* s, int64_t* out) try {
  if (!s || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = (int64_t)s->term_host.size();
  return 0;
} OGB_CATCH_ALL
int ogb_sampler_copy_bounds(const ogb_sampler* s, int64_t* terminal_locs, int64_t* initial_locs) try {
  if (!s) return fail(OGB_ERR_INVALID, "null sampler");
  for (size_t i = 0; i < s->term_host.size(); ++i) {
    if (terminal_locs) terminal_locs[i] = s->term_host[i];
    if (initial_locs) initial_locs[i] = i == 0 ? 0 : (int64_t)s->term_host[i - 1] + 1;  // datasets.py:187
  }
  return 0;
} OGB_CATCH_ALL
int ogb_sampler_get_counter(const ogb_sampler* s, uint64_t* out) try {
  if (!s || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = s->counter;
  return 0;
} OGB_CATCH_ALL
int ogb_sampler_set_counter(ogb_sampler* s, uint64_t counter) try {
  if (!s) return fail(OGB_ERR_INVALID, "null sampler");
  s->counter = counter;
  return 0;
} OGB_CATCH_ALL
int ogb_sampler_destroy(ogb_sampler* s) try {
  if (!s) return fail(OGB_ERR_INVALID, "null sampler");
  sampler_unref(s);
  return 0;
} OGB_CATCH_ALL

}  // extern "C"

namespace {

// What one launch sequence computes: the sampler's own plan (sample) or a derived one (gather, ATC).
struct RunSpec {
  int kind;                              // index-kernel behaviour: OGB_KIND_*
  const std::vector<KeyPlan>* plan;
  int n_slots;
  int64_t next_offset = 1;               // SLOT_NEXT = idx + next_offset (ATC: the temporal offset k)
  const int32_t* choice_table = nullptr; // ATC: anchor rows for this k (replaces the valid-row table)
  int64_t n_choices = -1;
  bool trl = false;
  int crop_padding = -1;                 // >= 0: crop every image key with the injected shifts and this padding (augment())
};

std::string kernel_name(const char* base, std::initializer_list<int> args) {
  std::string out = std::string(base) + "<";
  bool first = true;
  for (int a : args) { out += (first ? "" : ", ") + std::to_string(a); first = false; }
  return out + ">";
}

// A kernel and the name ogb_batch_dominant_kernel reports for it (the one ncu prints, which bench.py looks up in
// profiles/traffic.json), both taken from the same template arguments.
struct KernelChoice {
  const void* fn;
  const char* name;
  int resident = 0;   // index kernels: CTAs resident per SM without dynamic shared memory (4 if the query fails)
};

template <bool kInject, int kFlavour, bool kSmemTables, bool kPoint = false, int kMinBlocks = 4>
KernelChoice index_instance() {
  static const std::string name = kernel_name("relabel_index_kernel", {kInject, kFlavour, kSmemTables, kPoint, kMinBlocks});
  const void* fn = (const void*)ogb::relabel_index_kernel<kInject, kFlavour, kSmemTables, kPoint, kMinBlocks>;
  static const int resident = [fn] {
    int n = 0;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, fn, ogb::kRelabelThreads, 0) == cudaSuccess && n >= 1 ? n : 4;
  }();
  return {fn, name.c_str(), resident};
}
template <int kFlavour>
KernelChoice index_flavour(bool inject, bool smem_tables) {
  return inject ? (smem_tables ? index_instance<true, kFlavour, true>() : index_instance<true, kFlavour, false>())
                : (smem_tables ? index_instance<false, kFlavour, true>() : index_instance<false, kFlavour, false>());
}
// relabel_index_kernel for injected or Philox draws, the flavour, the segment table in shared memory or not, and the
// point-maze record (always a GCDataset launch)
KernelChoice choose_index_kernel(bool inject, int flavour, bool smem_tables, bool point_record) {
  using namespace ogb;
  // 48 registers, five CTAs per SM: 0.556 vs 0.541 of peak with four (six spill: 0.541), profiles/r2_ab_shapes.txt
  if (point_record && !inject)
    return smem_tables ? index_instance<false, FLAVOUR_GC, true, true, 5>() : index_instance<false, FLAVOUR_GC, false, true, 5>();
  if (point_record && !smem_tables) return index_instance<true, FLAVOUR_GC, false, true>();
  return flavour == FLAVOUR_GC ? index_flavour<FLAVOUR_GC>(inject, smem_tables)
       : flavour == FLAVOUR_HGC ? index_flavour<FLAVOUR_HGC>(inject, smem_tables) : index_flavour<FLAVOUR_PLAIN>(inject, smem_tables);
}

template <bool kInject, int kFlavour, int kStages = ogb::kAsyncStages, int kWarps = ogb::kAsyncWarps>
KernelChoice fused_instance() {
  static const std::string name = kernel_name("relabel_gather_kernel", {kInject, kFlavour, kStages, kWarps});
  return {(const void*)ogb::relabel_gather_kernel<kInject, kFlavour, kStages, kWarps>, name.c_str()};
}
// relabel_gather_kernel in a shape of split_span_jobs (2 x 20 and 2 x 16 are compiled for the fused GCDataset launch with
// Philox draws only)
KernelChoice choose_fused_kernel(bool inject, int flavour, int shape) {
  using namespace ogb;
  if (shape == 220 || shape == 216) return shape == 220 ? fused_instance<false, FLAVOUR_GC, 2, 20>() : fused_instance<false, FLAVOUR_GC, 2, 16>();
  if (flavour == FLAVOUR_GC) return inject ? fused_instance<true, FLAVOUR_GC>() : fused_instance<false, FLAVOUR_GC>();
  if (flavour == FLAVOUR_HGC) return inject ? fused_instance<true, FLAVOUR_HGC>() : fused_instance<false, FLAVOUR_HGC>();
  return inject ? fused_instance<true, FLAVOUR_PLAIN>() : fused_instance<false, FLAVOUR_PLAIN>();
}

template <int kStages, int kWarps>
KernelChoice async_instance() {
  static const std::string name = kernel_name("gather_rows_async_kernel", {kStages, kWarps});
  return {(const void*)ogb::gather_rows_async_kernel<kStages, kWarps>, name.c_str()};
}

template <int FS>
KernelChoice frames_instance() {
  static const std::string name = kernel_name("gather_frames_tma_kernel", {FS});
  return {(const void*)ogb::gather_frames_tma_kernel<FS>, name.c_str()};
}

// OGB_HOST_PHASES=1 (measurement switch): host time of run_sample by phase, summed over all calls, printed at exit.
struct HostPhases {
  static constexpr int kN = 7;
  double ns[kN] = {0};
  long calls = 0;
  bool on = getenv("OGB_HOST_PHASES") != nullptr;
  ~HostPhases() {
    if (!on || calls == 0) return;
    static const char* names[kN] = {"checks", "batch+layout", "block", "params", "classify", "prepare", "launch+event"};
    fprintf(stderr, "[ogb host phases] %ld calls:", calls);
    for (int i = 0; i < kN; ++i) fprintf(stderr, " %s %.2f us", names[i], ns[i] / calls * 1e-3);
    fprintf(stderr, "\n");
  }
};
HostPhases g_phases;
struct PhaseClock {
  std::chrono::steady_clock::time_point t;
  int next = 0;
  PhaseClock() { if (g_phases.on) t = std::chrono::steady_clock::now(); }
  void mark() {
    if (!g_phases.on) return;
    const auto now = std::chrono::steady_clock::now();
    if (next < HostPhases::kN) g_phases.ns[next++] += std::chrono::duration<double, std::nano>(now - t).count();
    t = now;
  }
};

// The start-row tables of `p`: `table` (TRL rows, ATC anchors) when there is one, else the dataset's valid rows --
// through the sampler's one-probe segment table when it has one --, and the trajectory tables.
void set_row_tables(const ogb_sampler* s, const int32_t* table, int64_t n_choices, ogb::RelabelParams* p) {
  const ogb_dataset* ds = s->ds;
  p->term = s->d_term;
  p->term_bucket = s->d_term_bucket;
  p->term_shift = s->term_shift;
  p->valid_table = table ? table : ds->d_valid_table;
  p->gap_c = ds->d_gap_c;
  p->gap_bucket = ds->d_gap_bucket;
  p->gap_shift = ds->gap_shift;
  p->valid_mode = table ? 1 : ds->valid_mode;
  if (!table && s->seg_shift >= 0) {
    p->valid_mode = 3;
    p->seg_table = s->d_seg_table;
    p->seg_bucket = s->d_seg_bucket;
    p->seg_shift = s->seg_shift;
    p->n_seg_table = s->n_seg_table;
    p->n_seg_bucket = s->n_seg_bucket;
  }
  p->n_choices = n_choices;
}

// How one goal set draws its goals (datasets.py:296-327).
ogb::GoalSpec goal_spec(double p_cur, double p_traj, bool geom, double discount) {
  auto word_threshold = [](double prob, uint32_t* thr, uint8_t* always) {
    // (w * 2^-32 < prob) <=> (w < ceil(prob * 2^32)) for 32-bit words w; the scaling by 2^32 is exact in float64
    const double t = std::ceil(prob * 4294967296.0);
    *always = t >= 4294967296.0 ? 1 : 0;
    *thr = t <= 0.0 ? 0u : (t >= 4294967296.0 ? 0xFFFFFFFFu : (uint32_t)t);
  };
  ogb::GoalSpec g{};
  g.geom = geom;
  g.cur_only = p_cur == 1.0;
  g.p_cur = p_cur;
  g.thr_traj = g.cur_only ? 0.0 : p_traj / (1.0 - p_cur);
  g.log_1mp = std::log(1.0 - (1.0 - discount));
  g.geo_abs_margin = (float)(1.5e-8 / std::fabs(g.log_1mp));
  word_threshold(g.thr_traj, &g.thr_traj32, &g.traj_always);
  word_threshold(g.p_cur, &g.thr_cur32, &g.cur_always);
  return g;
}

// Can the cp.async row gather read field f: rows at most kAsyncMaxStride apart, the whole field below 64 GiB, and the
// register-staged gather not forced (OGB_GATHER=lsu)?
bool async_reachable(const ogb_dataset* ds, const Field& f) {
  return f.stride <= (size_t)ogb::kAsyncMaxStride && (size_t)ds->size * f.stride < ((size_t)1 << 36) && !ab().gather_lsu;
}

// A span job loads one contiguous piece of the source rows named by one index vector and feeds one output per key.
struct SpanJob {
  int slot;
  const uint8_t* src;            // 16-byte aligned start of the span in row 0
  size_t stride, bytes;          // source row stride, span length (multiple of 16)
  std::vector<std::pair<size_t, size_t>> outs;   // (plan index, offset of the field inside the span)
};

// Sorts the row keys of a call by path: tiny rows ride along in the index kernel (the tiny jobs, groups and fields of
// `p`), the rest go to a gather launch -- the returned span jobs of the cp.async row gather, or register-staged (LSU) keys.
std::vector<SpanJob> classify_rows(const ogb_dataset* ds, const std::vector<KeyPlan>& plan, uint8_t* base,
                                   const std::vector<size_t>& offsets, ogb::RelabelParams* p, std::vector<size_t>* lsu_keys) {
  using namespace ogb;
  // Fields of the packed record table that are gathered through the same index vector and lie next to each other
  // (observations, actions, terminals, valids of the sampled transition) share ONE span.
  std::vector<SpanJob> span_jobs;
  p->n_tiny = 0;
  auto add_tiny = [&](size_t i) -> bool {
    const Field& f = ds->fields[(size_t)plan[i].field];
    if (f.row_bytes > 16 || p->n_tiny >= kMaxTinyJobs) return false;
    TinyJob& t = p->tiny[p->n_tiny++];
    const int v = largest_vec_log2(f.row_bytes, f.row_bytes);
    t.src = f.dptr;
    t.dst = base + offsets[i];
    t.slot = (uint8_t)plan[i].slot;
    t.size_log2 = (uint8_t)v;
    t.n_elem = (uint8_t)(f.row_bytes >> v);
    t.row_bytes = (uint8_t)f.row_bytes;
    t.stride = (uint16_t)f.stride;
    return true;
  };
  std::map<int, std::vector<size_t>> record_keys;   // slot -> keys whose field lives in the record table
  for (size_t i = 0; i < plan.size(); ++i) {
    if (plan[i].route != ROUTE_ROW || plan[i].alias_of >= 0) continue;
    const Field& f = ds->fields[(size_t)plan[i].field];
    if (f.in_record && async_reachable(ds, f)) {
      record_keys[plan[i].slot].push_back(i);
    } else if (add_tiny(i)) {
    } else if (f.row_bytes > 16 && async_reachable(ds, f)) {
      span_jobs.push_back({plan[i].slot, f.dptr, f.stride, round_up(f.row_bytes, 16), {{i, 0}}});
    } else {
      lsu_keys->push_back(i);
    }
  }
  for (auto& kv : record_keys) {
    std::vector<size_t>& keys = kv.second;
    std::sort(keys.begin(), keys.end(), [&](size_t a, size_t c) {
      return ds->fields[(size_t)plan[a].field].rec_off < ds->fields[(size_t)plan[c].field].rec_off;
    });
    for (size_t k0 = 0; k0 < keys.size();) {
      // extend the span while the next field starts within 32 bytes of the end of the current one, and while one
      // gather launch still holds the span's outputs (items x fields, at the span's own stage budget: a launch's
      // budget is never smaller, so it never has more items per span); an over-full span becomes two at a field boundary
      const Field& f0 = ds->fields[(size_t)plan[keys[k0]].field];
      size_t lo = f0.rec_off & ~(size_t)15, hi = f0.rec_off + f0.row_bytes, k1 = k0 + 1;
      bool has_long = f0.row_bytes > 16;
      while (k1 < keys.size()) {
        const Field& fn = ds->fields[(size_t)plan[keys[k1]].field];
        if (fn.rec_off > hi + 32) break;
        const size_t pitch = round_up(std::max(hi, fn.rec_off + fn.row_bytes) - lo, 16);
        if ((32 / rows_per_item(pitch, stage_budget(pitch))) * (k1 - k0 + 1) > (size_t)kMaxItemOuts) break;
        hi = std::max(hi, fn.rec_off + fn.row_bytes);
        has_long |= fn.row_bytes > 16;
        ++k1;
      }
      if (has_long) {
        SpanJob job{kv.first, ds->record_base + lo, ds->record_stride, round_up(hi - lo, 16), {}};
        for (size_t k = k0; k < k1; ++k) job.outs.push_back({keys[k], ds->fields[(size_t)plan[keys[k]].field].rec_off - lo});
        span_jobs.push_back(std::move(job));
      } else {
        // all tiny.  Fields of whole 4-byte words whose span fits two 16-byte loads become one group of the index
        // kernel (one record load for all of them); whatever does not fit is copied field by field.
        size_t k = k0;
        const bool no_groups = ab().no_tiny_groups;
        while (!no_groups && k < k1 && p->n_tiny_groups < kMaxTinyGroups) {
          const Field& fa = ds->fields[(size_t)plan[keys[k]].field];
          const size_t glo = fa.rec_off & ~(size_t)15;
          size_t kk = k, n_f = 0;
          int n_fields_total = 0;
          for (int gi = 0; gi < p->n_tiny_groups; ++gi) n_fields_total += p->tiny_groups[gi].n_fields;
          while (kk < k1) {
            const Field& fk = ds->fields[(size_t)plan[keys[kk]].field];
            if (fk.row_bytes % 4 != 0 || fk.rec_off % 4 != 0 || fk.rec_off + fk.row_bytes > glo + 32 ||
                (fk.row_bytes == 16 && (fk.rec_off - glo) % 16 != 0) || n_fields_total + (int)n_f >= kMaxTinyFields) break;
            ++kk; ++n_f;
          }
          if (n_f < 2) break;                    // a single field gains nothing over a plain tiny copy
          TinyGroup& grp = p->tiny_groups[p->n_tiny_groups++];
          grp.src = ds->record_base + glo;
          grp.stride = (uint16_t)ds->record_stride;
          grp.slot = (uint8_t)kv.first;
          grp.first_field = (uint8_t)n_fields_total;
          grp.n_fields = (uint8_t)n_f;
          size_t ghi = glo;
          for (size_t t = k; t < kk; ++t) {
            const Field& fk = ds->fields[(size_t)plan[keys[t]].field];
            TinyField& tf = p->tiny_fields[n_fields_total++];
            tf.dst = base + offsets[keys[t]];
            tf.word = (uint8_t)((fk.rec_off - glo) / 4);
            tf.n_words = (uint8_t)(fk.row_bytes / 4);
            tf.group = (uint8_t)(p->n_tiny_groups - 1);
            ghi = std::max(ghi, fk.rec_off + fk.row_bytes);
          }
          grp.n_vec = (uint8_t)(ghi - glo > 16 ? 2 : 1);
          p->n_tiny_fields = n_fields_total;
          k = kk;
        }
        for (; k < k1; ++k)
          if (!add_tiny(keys[k])) {   // more tiny rows than the index kernel takes: a span of their own
            const Field& fk = ds->fields[(size_t)plan[keys[k]].field];
            const size_t l2 = fk.rec_off & ~(size_t)15;
            span_jobs.push_back({kv.first, ds->record_base + l2, ds->record_stride, round_up(fk.rec_off + fk.row_bytes - l2, 16),
                                 {{keys[k], fk.rec_off - l2}}});
          }
      }
      k0 = k1;
    }
  }
  // rows of 4, 8 or 16 bytes first: the index kernel copies those four at a time
  auto fast = [](const TinyJob& t) { return t.row_bytes == 4 || t.row_bytes == 8 || t.row_bytes == 16; };
  std::stable_partition(p->tiny, p->tiny + p->n_tiny, fast);
  p->n_tiny_fast = (int32_t)std::count_if(p->tiny, p->tiny + p->n_tiny, fast);
  return span_jobs;
}

// The point-maze record (relabel_row<..., kPoint>): one group of the transition's own 32-byte record holding
// observations f32[2] | actions f32[2] | terminals | valids | shadow next observation, and the two 8-byte goal rows;
// nothing else to gather.  The index kernel then runs with these copies compiled in.
// (the kernel also compiles out what such a launch cannot need: index vectors in memory -- no later kernel, debug off --,
// frame-stack rows, the SLOT_NEXT row, the TRL branch, and every valid-row form but the segment table)
bool is_point_record(const ogb_sampler* s, const RunSpec& spec, const ogb::RelabelParams& p, bool any_gather) {
  using namespace ogb;
  if (!(spec.kind == OGB_KIND_GC && !spec.trl && !any_gather &&
        !s->debug && p.valid_mode == 3 && p.vec_init == nullptr &&
        p.n_tiny_groups == 1 && p.n_tiny_fields == 5 && p.n_tiny == 2 && p.n_tiny_fast == 2 &&
        p.tiny_groups[0].slot == SLOT_IDX && p.tiny_groups[0].n_vec == 2 &&
        p.tiny[0].slot == GC_VALUE_GOAL && p.tiny[0].row_bytes == 8 && p.tiny[1].slot == GC_ACTOR_GOAL && p.tiny[1].row_bytes == 8))
    return false;
  static const int kWord[5] = {0, 2, 4, 5, 6}, kCount[5] = {2, 2, 1, 1, 2};
  for (int f = 0; f < 5; ++f)
    if (p.tiny_fields[f].word != kWord[f] || p.tiny_fields[f].n_words != kCount[f]) return false;
  return true;
}

// One launch of the cp.async row gather: span jobs [first, end), its stage budget and stage bytes, and its shape
// (100 * stages + warps per CTA).
struct RowLaunch {
  size_t first, end, budget;
  int stage_bytes, shape;
};

// Splits the span jobs over launches (all element widths in one launch; a job list that needs more items or outputs
// than a launch holds goes to several).  The first launch is the fused one when `fuse`; `gc_philox`: the call is a
// GCDataset one with Philox draws.
int split_span_jobs(const std::vector<SpanJob>& span_jobs, bool fuse, bool gc_philox, std::vector<RowLaunch>* out) {
  using namespace ogb;
  for (size_t q0 = 0; q0 < span_jobs.size();) {
    size_t q1 = std::min(span_jobs.size(), q0 + (size_t)kMaxRowJobs), budget = 0;
    for (;; --q1) {   // the largest prefix of the remaining jobs whose items and outputs fit one launch
      size_t max_pitch = 0, n_items = 0, n_outs = 0;
      for (size_t t = q0; t < q1; ++t) max_pitch = std::max(max_pitch, span_jobs[t].bytes);
      budget = stage_budget(max_pitch);
      for (size_t t = q0; t < q1; ++t) {
        const size_t r = rows_per_item(span_jobs[t].bytes, budget);
        n_items += 32 / r;
        n_outs += (32 / r) * span_jobs[t].outs.size();
      }
      if ((n_items <= (size_t)kMaxItems && n_outs <= (size_t)kMaxItemOuts) || q1 == q0 + 1) {
        if (n_items > (size_t)kMaxItems || n_outs > (size_t)kMaxItemOuts)
          return fail(OGB_ERR_UNSUPPORTED, "a %zu-byte row span with %zu keys does not fit one gather launch", span_jobs[q0].bytes, span_jobs[q0].outs.size());
        break;
      }
    }
    size_t stage = 0;
    for (size_t t = q0; t < q1; ++t) stage = std::max(stage, rows_per_item(span_jobs[t].bytes, budget) * span_jobs[t].bytes);
    const int stage_bytes = (int)round_up(stage, 128);
    // (stages, warps per CTA): 3 x 8 (two CTAs per SM), except for the fused GCDataset launch (2 x 20, or 2 x 16 when
    // 20 warps' rings do not fit) and the un-fused gather with stages over 4 KB (3 x 10).
    // Measured on B200 (profiles/r2_ab_shapes.txt).  Fused GCDataset launch: ONE CTA of 20 warps with two stages per warp
    // (160 KB of shared memory with 4 KB stages) -- 2 x 16 had beaten 3 x 8 x 2 CTAs by 4 % (C2) / 2 % (C5) with static
    // tiles; with ticket-scheduled tiles and ~1 ms launches 2 x 20 is another 4 % ahead on C2 (0.945-0.961 vs 0.908-0.927
    // of peak; five warps per scheduler instead of four) and level on C5 (0.950 vs 0.943-0.951); 18, 22 or 24 warps lose
    // 4-13 % (uneven warps per scheduler, and a register cap that makes the index algebra spill; 24 warps with the index
    // algebra out of line, to keep the loops under the 80-register cap, lost 25 %).  Un-fused gather: three
    // stages; with 6 KB stages (rows > 256 B: C3) ten warps in one CTA, 0.979 vs 0.964 for eight (twelve: 0.968).
    const bool fused_here = fuse && q0 == 0;
    int shape = 308;
    if (fused_here && gc_philox) shape = (size_t)20 * 2 * stage_bytes <= (size_t)200 * 1024 ? 220 : 216;
    else if (!fused_here && stage_bytes > 4096 && (size_t)10 * 3 * stage_bytes <= (size_t)200 * 1024) shape = 310;
    out->push_back({q0, q1, budget, stage_bytes, shape});
    q0 = q1;
  }
  return 0;
}

// The item and output tables of one row-gather launch (relabel_rows.cuh, ItemDesc / OutDesc: the jobs unrolled into the
// items of one 32-row tile), with the drain kind of every output, the index-vector prefetch links and the item at which
// a warp claims its next tile.  Returns the number of (tile, index vector) pairs.
size_t fill_row_tables(const ogb_dataset* ds, const std::vector<KeyPlan>& plan, uint8_t* base, const std::vector<size_t>& offsets,
                       const std::vector<SpanJob>& span_jobs, const RowLaunch& rl, bool fused, ogb::AsyncGatherParams* ap) {
  using namespace ogb;
  auto magic = [](uint32_t d) -> uint32_t { return d <= 1 ? 0u : (uint32_t)((((uint64_t)1 << 32) + d - 1) / d); };
  for (size_t q = rl.first; q < rl.end; ++q) {
    const SpanJob& sj = span_jobs[q];
    const uint32_t cpr = (uint32_t)(sj.bytes / 16), pitch = cpr * 16u;
    const uint32_t rpi = (uint32_t)rows_per_item(pitch, rl.budget);
    for (uint32_t sub = 0; sub < 32; sub += rpi) {
      ItemDesc& it = ap->items[ap->n_items++];
      it.src16 = reinterpret_cast<const uint4*>(sj.src);
      it.stride16 = (uint32_t)(sj.stride / 16);
      it.cpr = cpr;
      it.cpr_magic = magic(cpr);
      it.dr = 32 / cpr;
      it.dch = 32 % cpr;
      it.slot = (uint32_t)sj.slot;
      it.sub = sub;
      it.rows = rpi;
      it.flags = sub == 0 ? 1u : 0u;
      it.out_begin_n = (uint32_t)ap->n_outs | ((uint32_t)sj.outs.size() << 16);
      for (const auto& po : sj.outs) {
        const Field& f = ds->fields[(size_t)plan[po.first].field];
        OutDesc& out = ap->outs[ap->n_outs++];
        out.dst = base + offsets[po.first] + (size_t)sub * f.row_bytes;
        out.tile_bytes = (uint32_t)(32 * f.row_bytes);
        out.soff = (uint32_t)po.second;
        out.gap = pitch - (uint32_t)f.row_bytes;
        uint32_t kind, vec_log2 = 0;
        if (f.row_bytes % 16 == 0 && out.gap == 0) {
          kind = DRAIN_DENSE16;
          out.epr = (uint32_t)f.row_bytes;
        } else if (f.row_bytes % 4 == 0 && po.second % 4 == 0) {
          // items start on 16-byte boundaries of the dense output unless an item holds fewer than four odd-sized rows
          kind = ((size_t)sub * f.row_bytes) % 16 == 0 ? DRAIN_WORDS : DRAIN_WORDS_UNALIGNED;
          out.epr = (uint32_t)(f.row_bytes / 4);
        } else {
          kind = DRAIN_ELEMS;
          vec_log2 = (f.row_bytes % 2 == 0 && po.second % 2 == 0) ? 1 : 0;
          out.epr = (uint32_t)(f.row_bytes >> vec_log2);
        }
        out.epr_magic = magic(out.epr);
        out.kind = kind | (vec_log2 << 8) | (pitch << 16);
      }
    }
  }
  // index-vector prefetch of the un-fused kernel: every pair's first item names the slot (and tile) of the pair after it
  for (int k = 0; k < ap->n_items; ++k) {
    if (!(ap->items[k].flags & 1u)) continue;
    int nk = k + 1;
    while (nk < ap->n_items && !(ap->items[nk].flags & 1u)) ++nk;
    const bool wraps = nk == ap->n_items;
    ap->items[k].flags |= (ap->items[wraps ? 0 : nk].slot << 8) | (wraps ? 0x10000u : 0u);
  }
  // Dynamic tile scheduling: the ticket of the next tile is taken ahead of the item where the head needs the tile -- the
  // fused kernel needs it when it leaves the tile, the un-fused one already at the first item of the last pair, where it
  // prefetches the next tile's index vector.  How far ahead, measured (profiles/r2_ab_shapes.txt, batch r2k): the fused
  // launches (16 warps per SM) are best with one pair -- a ticket taken earlier keeps a tile away from a faster warp
  // (C2 0.890 / 0.888 / 0.876 of peak for 1 / 2 / all pairs ahead); the un-fused gather with 8 warps per SM does not cover
  // a late ticket's round trip through the busy memory system (C3 0.952 / 0.956 / 0.960 / 0.963 for 1 / 2 / 3 / all),
  // while C5b's shape prefers <= 3 (1.021 vs 1.011) -> three.
  std::vector<int> pair_first;
  for (int k = 0; k < ap->n_items; ++k) if (ap->items[k].flags & 1u) pair_first.push_back(k);
  // index (into pair_first) of the pair at whose first item the tile is needed; the fused kernel needs it one pair "later"
  const int need = (int)pair_first.size() - (fused ? 0 : 1);
  const int ahead = fused ? 1 : 3;
  ap->claim_item = pair_first[(size_t)std::max(0, need - ahead)];
  return pair_first.size();
}

typedef std::function<int(int64_t, int64_t, cudaStream_t)> LaunchFn;

// relabel_index_kernel over rows [begin, end); `dominant`: it is the call's dominant kernel, and names itself as it launches
LaunchFn index_launch(ogb_sampler* s, ogb_batch* b, const ogb::RelabelParams& params, bool inject, int flavour, bool point_record,
                      bool dominant) {
  using namespace ogb;
  return [=, p = params](int64_t begin, int64_t end, cudaStream_t st) mutable -> int {
    p.row_begin = begin;
    p.row_end = end;
    const int64_t blocks_needed = (end - begin + kRelabelThreads - 1) / kRelabelThreads;
    // Shared memory (0: the plain grid).  Big launches over a dataset whose segment table is small keep the table in shared
    // memory (persistent CTAs) when they run on the auxiliary stream under another call's gather: the persistent form
    // with few CTAs disturbs the gather less (C3 0.716 vs 0.730 ms); alone on its stream the plain grid is faster (C1
    // 0.047 vs 0.049).
    const size_t table_bytes = (size_t)p.n_seg_table * 16 + (size_t)p.n_seg_bucket * 4;
    const size_t smem = st != s->stream && p.valid_mode == 3 && table_bytes > 0 && table_bytes <= 48 * 1024 &&
                        end - begin >= 65536 ? table_bytes : 0;
    const KernelChoice k = choose_index_kernel(inject, flavour, smem > 0, point_record);
    // Grid cap: a whole number of waves of resident CTAs (a 16-per-SM grid of the five-per-SM point-maze kernel is 3.2
    // waves, and the last, fifth-full wave cost C1 5 %: 0.731 vs 0.771-0.775 of peak for 5, 10 or 32 per SM, batch r2l).
    int64_t grid_cap = (int64_t)s->ds->sm_count * 2 * k.resident;
    if (smem > 0) {
      int per_sm = 0;
      if (cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
          cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k.fn, kRelabelThreads, smem) != cudaSuccess || per_sm < 1)
        return fail(OGB_ERR_CUDA, "relabel_index_kernel (shared tables): occupancy query failed");
      grid_cap = (int64_t)s->ds->sm_count * per_sm;
    }
    const unsigned grid = (unsigned)std::min<int64_t>(blocks_needed, grid_cap);
    void* args[] = {(void*)&p};
    if (cudaLaunchKernel(k.fn, dim3(grid), dim3(kRelabelThreads), args, smem, st) != cudaSuccess)
      return fail(OGB_ERR_CUDA, "relabel_index_kernel launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (cudaGetLastError() != cudaSuccess) return fail(OGB_ERR_CUDA, "relabel_index_kernel launch failed");
    if (dominant) b->dominant = k.name;
    b->kernel_names.push_back(k.name);
    b->launches++;
    return 0;
  };
}

// One run_sample call: its arguments, what they imply under the sampler's config, its batch and its launches.  The steps
// run in this order: check, new_batch, fill_params, the prepare_* steps, issue.
struct Run {
  ogb_sampler* s;
  const ogb_dataset* ds;
  const ogb_config& cfg;
  const RunSpec& spec;
  const std::vector<KeyPlan>& plan;
  int64_t batch, total;
  int32_t n_batches;
  const int64_t* idxs;
  const ogb_draws* draws;
  bool stacked_next = false;
  int64_t idx_last = 0;             // the largest index a given row may have
  bool defer_check = false;         // given indices are range-checked by the kernel (the flag is read later)
  int64_t n_choices = 0;
  bool aug_mode = false;
  double p_aug = 0.0;
  int crop_pad = 0;
  bool goal_used[3] = {false, false, false};   // goal sets drawn: value, low-value, actor
  ogb_batch* b = nullptr;
  cudaStream_t first = nullptr;     // stream of the uploads and of the index kernel or fused launch
  // where the scratch arrays of the batch block start (the keys come first, at ogb_batch::offsets)
  size_t off_rows = 0, off_init = 0, off_crop = 0, off_idxs = 0, off_idx_error = 0, off_trl_mid = 0;
  size_t off_draw_i64[1 + 3 * 2 + 1] = {0}, off_draw_f64[3 * 3] = {0};
  // the launches, prepared once and issued per row chunk: the index kernel -- or the fused launch, which does its work
  // too -- and the gathers behind it
  LaunchFn index, fused;
  std::vector<LaunchFn> gathers;
  ogb::RelabelParams p;             // of the index algebra (index kernel or fused launch)

  int check(bool evaluation) {
    if (batch < 0 || n_batches < 1) return fail(OGB_ERR_INVALID, "batch_size must be >= 0 and n_batches >= 1");
    if (draws && n_batches != 1) return fail(OGB_ERR_INVALID, "validation draws need n_batches == 1");
    if (total > (int64_t)1 << 31) return fail(OGB_ERR_UNSUPPORTED, "more than 2^31 rows in one launch");
    stacked_next = (cfg.frame_stack > 0 && spec.kind != OGB_KIND_PLAIN) || spec.kind == OGB_KIND_ATC;
    idx_last = (stacked_next ? ds->size - spec.next_offset : ds->size) - 1;
    defer_check = idxs && s->defer_index_check;
    if (idxs && !defer_check) {  // numpy fancy indexing would raise IndexError (negative wrap-around is not supported here)
      // branch-free scan (vectorises): idx < 0 or idx > last sets the sign bit of idx | (last - idx)
      int64_t bad = 0;
      for (int64_t r = 0; r < total; ++r) bad |= idxs[r] | (idx_last - idxs[r]);
      if (bad < 0)
        for (int64_t r = 0; r < total; ++r)
          if (idxs[r] < 0 || idxs[r] > idx_last)
            return fail(OGB_ERR_INDEX, "index %lld is out of bounds for axis 0 with size %lld", (long long)idxs[r], (long long)ds->size);
    }
    if (idxs && spec.trl) {
      // datasets.py:255-256: `assert (idxs != final_state_idxs).all()` -- a given index that is a trajectory's final state
      // (a terminal row) has no midpoint span, and its idx + 1 belongs to the next trajectory (or lies past the table)
      for (int64_t r = 0; r < total; ++r)
        if (idxs[r] >= 0 && idxs[r] < ds->size && !ds->terminals_host.empty() && ds->terminals_host[(size_t)idxs[r]])
          return fail(OGB_ERR_ASSERT, "assert (idxs != final_state_idxs).all() (datasets.py:256): index %lld is a final state", (long long)idxs[r]);
    }
    n_choices = n_choices_for(ds, spec.choice_table, spec.n_choices);
    if (n_choices < 1) return fail(OGB_ERR_INVALID, "nothing to sample from: the dataset holds no rows yet");
    const bool forced_crop = spec.crop_padding >= 0;
    aug_mode = forced_crop || (cfg.has_p_aug && !evaluation && spec.kind != OGB_KIND_PLAIN);
    p_aug = forced_crop ? 1.0 : cfg.p_aug;
    crop_pad = forced_crop ? spec.crop_padding : cfg.crop_padding;
    goal_used[0] = goal_used[2] = spec.kind == OGB_KIND_GC || spec.kind == OGB_KIND_HGC;
    goal_used[1] = spec.kind == OGB_KIND_HGC && cfg.has_low_discount;
    if (draws) {
      const bool geom[3] = {cfg.value_geom_sample != 0, true, cfg.actor_geom_sample != 0};
      const bool cur_only[3] = {cfg.value_p_curgoal == 1.0, cfg.value_p_curgoal == 1.0, cfg.actor_p_curgoal == 1.0};
      if (!idxs && !draws->idx_pos) return fail(OGB_ERR_INVALID, "validation mode needs idx_pos or idxs");
      for (int gs = 0; gs < 3; ++gs) {
        if (!goal_used[gs]) continue;
        const ogb_goal_draws& d = draws->goals[gs];
        if (!d.rand_pos || (geom[gs] ? !d.offset : !d.dist) || (!cur_only[gs] && (!d.u_traj || !d.u_cur)))
          return fail(OGB_ERR_INVALID, "validation mode: goal set %d is missing draws", gs);
        for (int64_t r = 0; r < batch; ++r)
          if (d.rand_pos[r] < 0 || d.rand_pos[r] >= n_choices) return fail(OGB_ERR_INDEX, "rand_pos out of range");
      }
      if (draws->idx_pos && !idxs)
        for (int64_t r = 0; r < batch; ++r)
          if (draws->idx_pos[r] < 0 || draws->idx_pos[r] >= n_choices) return fail(OGB_ERR_INDEX, "idx_pos out of range");
      if (aug_mode && !draws->has_aug_coin) return fail(OGB_ERR_INVALID, "validation mode: the augmentation coin is missing");
      if (aug_mode && draws->aug_coin < p_aug && !draws->crop) return fail(OGB_ERR_INVALID, "validation mode: crop draws are missing");
    }
    return 0;
  }
  // A batch of the call's keys and the layout of its device block: keys first (so that one D2H copy takes the whole
  // batch), then the index vectors and the uploaded arguments.
  void new_batch(bool want_init, bool want_crop) {
    b = new ogb_batch();
    b->sampler = s;
    s->refs.fetch_add(1);
    b->batch = batch;
    b->n_batches = n_batches;
    b->total_rows = total;
    b->keys = plan;
    b->offsets.assign(plan.size(), 0);
    b->n_slots = spec.n_slots;
    size_t cursor = 0;
    for (size_t i = 0; i < plan.size(); ++i) {
      if (plan[i].alias_of >= 0) continue;
      b->offsets[i] = cursor;
      cursor = round_up(cursor + (size_t)total * plan[i].row_bytes, 256);
    }
    for (size_t i = 0; i < plan.size(); ++i)
      if (plan[i].alias_of >= 0) b->offsets[i] = b->offsets[(size_t)plan[i].alias_of];
    b->keys_bytes = cursor;
    auto carve = [&](size_t bytes) { size_t off = cursor; cursor = round_up(cursor + bytes, 256); return off; };
    off_rows = carve((size_t)spec.n_slots * total * 4);
    if (want_init) off_init = carve((size_t)spec.n_slots * total * 4);
    if (want_crop) off_crop = carve((size_t)total * 2);
    if (idxs) off_idxs = carve((size_t)total * 8);
    if (defer_check) off_idx_error = carve(4);
    if (draws) {
      off_draw_i64[0] = carve((size_t)batch * 8);
      for (int gs = 0; gs < 3; ++gs) {
        off_draw_i64[1 + 2 * gs] = carve((size_t)batch * 8);
        off_draw_i64[2 + 2 * gs] = carve((size_t)batch * 8);
        for (int q = 0; q < 3; ++q) off_draw_f64[3 * gs + q] = carve((size_t)batch * 8);
      }
      off_draw_i64[7] = carve((size_t)batch * 16);
      if (spec.trl) off_trl_mid = carve((size_t)batch * 8);
    }
    b->block_bytes = std::max<size_t>(cursor, 256);
  }
  // The parameters of the index algebra (index kernel or fused launch) except the row keys; uploads the given indices and
  // validation draws on `first`.
  int fill_params() {
    using namespace ogb;
    uint8_t* base = b->block;
    memset(&p, 0, sizeof(p));
    set_row_tables(s, spec.choice_table, n_choices, &p);
    p.next_offset = (int32_t)spec.next_offset;
    p.trl = spec.trl ? 1 : 0;
    // (a ReplayBuffer that is still filling up clamps idx + 1 at its current size, datasets.py:82 with self.size = fill)
    p.n_rows_ds = (int32_t)(spec.kind == OGB_KIND_PLAIN && ds->active_rows > 0 ? ds->active_rows : ds->size);
    p.goal[0] = goal_spec(cfg.value_p_curgoal, cfg.value_p_trajgoal, cfg.value_geom_sample != 0, cfg.discount);
    p.goal[1] = goal_spec(cfg.value_p_curgoal, cfg.value_p_trajgoal, true, cfg.has_low_discount ? cfg.low_discount : cfg.discount);
    p.goal[2] = goal_spec(cfg.actor_p_curgoal, cfg.actor_p_trajgoal, cfg.actor_geom_sample != 0, cfg.discount);
    {  // the actor coins are only drawn when they can change the outcome
      const GoalSpec& a = p.goal[2];
      const bool cur_fixed = a.cur_only || a.cur_always || a.thr_cur32 == 0;
      const bool traj_fixed = a.traj_always || a.thr_traj32 == 0;
      p.actor_mix = (a.cur_only || (cur_fixed && traj_fixed)) ? 0 : 1;
    }
    p.neg_lut = s->d_neg_lut;
    p.pow_lut = s->d_pow_lut;
    p.kind = spec.kind;
    p.has_low_goal = goal_used[1];
    p.k_val = cfg.value_subgoal_steps;
    p.k_act = cfg.actor_subgoal_steps;
    p.k_lo = cfg.low_subgoal_steps;
    p.gc_negative = cfg.gc_negative;
    p.stacked_next = stacked_next;
    p.aug_mode = aug_mode;
    p.crop_pad = crop_pad;
    p.p_aug = p_aug;
    p.key = make_rng_key(s->seed, s->stream_id);
    p.batch0 = s->counter;
    p.batch = batch;
    p.batch_magic = batch > 1 && batch < ((int64_t)1 << 32) ? (uint64_t)(~(uint64_t)0 / (uint64_t)batch) + 1 : 0;
    p.total_rows = total;
    p.n_slots = spec.n_slots;
    p.narrow = cfg.jax_compat ? 1 : 0;
    p.vec_rows = b->vec_rows;
    p.vec_init = b->vec_init;
    p.crop_out = b->crop;

    cudaError_t e = cudaSuccess;
    // copies `src` (when there is one) to the block at `off` unless an earlier copy failed; returns where it went
    auto up = [&](size_t off, const void* src, size_t bytes) -> uint8_t* {
      if (!src || e != cudaSuccess) return nullptr;
      e = cudaMemcpyAsync(base + off, src, bytes, cudaMemcpyHostToDevice, first);
      return base + off;
    };
    if (idxs) {
      p.given_idxs = (const int64_t*)up(off_idxs, idxs, (size_t)total * 8);
      if (e != cudaSuccess) return fail(OGB_ERR_CUDA, "H2D of idxs failed");
      if (defer_check) {
        b->idx_error = (int32_t*)(base + off_idx_error);
        if (cudaMemsetAsync(b->idx_error, 0, 4, first) != cudaSuccess) return fail(OGB_ERR_CUDA, "memset of the index flag failed");
        p.idx_error = b->idx_error;
        p.idx_last = idx_last;
      }
    }
    if (draws) {
      const size_t n = (size_t)batch;
      if (!idxs) p.in_idx_pos = (const int64_t*)up(off_draw_i64[0], draws->idx_pos, n * 8);
      for (int gs = 0; gs < 3; ++gs) {
        if (!goal_used[gs]) continue;
        const ogb_goal_draws& d = draws->goals[gs];
        GoalInject& g = p.in_goal[gs];
        g.rand_pos = (const int64_t*)up(off_draw_i64[1 + 2 * gs], d.rand_pos, n * 8);
        g.offset = (const int64_t*)up(off_draw_i64[2 + 2 * gs], d.offset, n * 8);
        g.dist = (const double*)up(off_draw_f64[3 * gs], d.dist, n * 8);
        g.u_traj = (const double*)up(off_draw_f64[3 * gs + 1], d.u_traj, n * 8);
        g.u_cur = (const double*)up(off_draw_f64[3 * gs + 2], d.u_cur, n * 8);
      }
      p.in_crop = (const int64_t*)up(off_draw_i64[7], draws->crop, n * 16);
      if (spec.trl && e == cudaSuccess && !draws->trl_midpoints)
        return fail(OGB_ERR_INVALID, "validation mode: TRL midpoint draws are missing");
      if (spec.trl) p.in_trl_mid = (const int64_t*)up(off_trl_mid, draws->trl_midpoints, n * 8);
      p.in_coin = draws->has_aug_coin ? draws->aug_coin : 2.0;
      if (p.aug_mode && !(p.in_coin < p.p_aug)) p.in_crop = nullptr;
      if (e != cudaSuccess) return fail(OGB_ERR_CUDA, "H2D of validation draws failed: %s", cudaGetErrorString(e));
    }
    for (size_t i = 0; i < plan.size(); ++i) {
      if (plan[i].route != ROUTE_SCALAR) continue;
      void* ptr = base + b->offsets[i];
      switch (plan[i].scalar) {
        case SC_MASKS: p.masks = (double*)ptr; break;
        case SC_REWARDS: p.rewards = (double*)ptr; break;
        case SC_HV_OFFSETS: p.hv_offsets = (int64_t*)ptr; break;
        case SC_HV_STEPS: p.hv_steps = (int64_t*)ptr; break;
        case SC_HV_MASKS: p.hv_masks = (double*)ptr; break;
        case SC_HV_REWARDS: p.hv_rewards = (double*)ptr; break;
        case SC_LV_STEPS: p.lv_steps = (int64_t*)ptr; break;
        case SC_LV_MASKS: p.lv_masks = (double*)ptr; break;
        case SC_LV_REWARDS: p.lv_rewards = (double*)ptr; break;
        case SC_TRL_OFFSETS: p.trl_offsets = (int64_t*)ptr; break;
        case SC_TRL_MID_OFFSETS: p.trl_mid_offsets = (int64_t*)ptr; break;
        default: break;
      }
    }
    return 0;
  }
  // The cp.async row gathers of the span jobs; with `fuse`, the first launch is the fused one, which also does the index
  // algebra of `p` (and stores the index vectors when later launches read them).
  int prepare_row_gathers(const std::vector<SpanJob>& span_jobs, bool fuse, bool inject, int flavour) {
    using namespace ogb;
    std::vector<RowLaunch> split;
    OGB_TRY(split_span_jobs(span_jobs, fuse, p.kind == OGB_KIND_GC && !inject, &split));
    for (const RowLaunch& rl : split) {
      const bool fused_here = fuse && rl.first == 0;
      const int n_stages = rl.shape / 100, n_warps = rl.shape % 100;
      AsyncGatherParams ap;
      memset(&ap, 0, sizeof(ap));
      ap.vec_rows = b->vec_rows;
      ap.total_rows = total;
      ap.stage_bytes = rl.stage_bytes;
      ap.ring_bytes = n_stages * ap.stage_bytes;
      const size_t n_pairs = fill_row_tables(ds, plan, b->block, b->offsets, span_jobs, rl, fused_here, &ap);
      // (a single-pair un-fused launch keeps static tiles)
      const bool dyn_tiles = !s->static_tiles && (fused_here || n_pairs >= 2);
      // shared memory: item table, output table, one 16-byte tile FIFO per warp, then the rings
      ap.ring_offset = (int)round_up((size_t)ap.n_items * sizeof(ItemDesc) + (size_t)ap.n_outs * sizeof(OutDesc) + (size_t)n_warps * 16, 128);
      const size_t smem = (size_t)ap.ring_offset + (size_t)n_warps * ap.ring_bytes;
      if (smem > (size_t)225 * 1024)
        return fail(OGB_ERR_UNSUPPORTED, "internal: gather shape %d needs %zu bytes of shared memory", rl.shape, smem);
      // persistent grid: exactly the CTAs that are resident at once.  Fused: shared memory bounds them (the fused kernels
      // are compiled for gather_min_blocks(warps) CTAs per SM, so registers allow at least that many); un-fused: what the
      // occupancy query finds for registers and shared memory together.
      const KernelChoice k = fused_here ? choose_fused_kernel(inject, flavour, rl.shape)
                           : rl.shape == 310 ? async_instance<3, 10>() : async_instance<kAsyncStages, kAsyncWarps>();
      int per_sm = (int)std::max<size_t>(1, std::min<size_t>(n_warps <= 8 ? 2 : 1, (size_t)(220 * 1024) / smem));
      if (!fused_here) {
        OGB_CUDA(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k.fn, n_warps * 32, smem) != cudaSuccess || per_sm < 1)
          return fail(OGB_ERR_CUDA, "gather_rows_async_kernel: occupancy query failed (%zu bytes of shared memory)", smem);
      }
      if (rl.first == 0) b->dominant = k.name;
      // index algebra + the first (normally the only) group of row jobs in ONE launch; the launches that take the
      // remaining jobs read the index vectors this one computes
      if (fused_here && rl.end < span_jobs.size()) p.write_vecs = 1;
      std::shared_ptr<FusedParams> keep(new FusedParams);   // (the un-fused kernel takes .gather alone)
      if (fused_here) keep->relabel = p;
      keep->gather = ap;
      const char* what = fused_here ? "relabel_gather_kernel" : "gather_rows_async_kernel";
      LaunchFn launch = [=](int64_t begin, int64_t end, cudaStream_t st) -> int {
        FusedParams& f = *keep;
        f.relabel.row_begin = f.gather.row_begin = begin;
        f.relabel.row_end = f.gather.row_end = end;
        const int64_t n_warp_tiles = (end - begin + 31) / 32;
        const unsigned grid = (unsigned)std::min<int64_t>((n_warp_tiles + n_warps - 1) / n_warps, (int64_t)ds->sm_count * per_sm);
        // (tickets only when there are more tiles than warps: a small launch gives every warp at most its first tile)
        f.gather.sched = dyn_tiles && n_warp_tiles > (int64_t)grid * n_warps ? s->next_sched() : nullptr;
        if (fused_here && cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
          return fail(OGB_ERR_CUDA, "cudaFuncSetAttribute(relabel_gather_kernel) failed");
        void* args[] = {fused_here ? (void*)&f : (void*)&f.gather};
        if (cudaLaunchKernel(k.fn, dim3(grid), dim3((unsigned)n_warps * 32), args, smem, st) != cudaSuccess)
          return fail(OGB_ERR_CUDA, "%s launch failed: %s", what, cudaGetErrorString(cudaGetLastError()));
        if (!fused_here && cudaGetLastError() != cudaSuccess) return fail(OGB_ERR_CUDA, "%s launch failed", what);
        b->kernel_names.push_back(k.name);
        b->launches++;
        return 0;
      };
      if (fused_here) fused = launch;
      else gathers.push_back(launch);
    }
    return 0;
  }
  // register-staged gather for what the asynchronous kernel does not take (very long rows): one launch per element width
  // and kMaxRowJobs keys
  int prepare_lsu_gathers(const std::vector<size_t>& row_keys) {
    using namespace ogb;
    std::vector<int> vec_of(row_keys.size());
    for (size_t q = 0; q < row_keys.size(); ++q) {
      const Field& f = ds->fields[(size_t)plan[row_keys[q]].field];
      vec_of[q] = largest_vec_log2(f.row_bytes, f.stride);
    }
    for (int v = 4; v >= 0; --v) {
      size_t q = 0;
      while (q < row_keys.size()) {
        GatherParams gp;
        memset(&gp, 0, sizeof(gp));
        gp.vec_rows = b->vec_rows;
        gp.total_rows = total;
        for (; q < row_keys.size() && gp.n_jobs < kMaxRowJobs; ++q) {
          if (vec_of[q] != v) continue;
          const KeyPlan& k = plan[row_keys[q]];
          const Field& f = ds->fields[(size_t)k.field];
          if ((f.row_bytes >> v) > 65535) return fail(OGB_ERR_UNSUPPORTED, "row of field '%s' too long for the row path", f.name.c_str());
          RowJob& job = gp.jobs[gp.n_jobs++];
          job.src = f.dptr;
          job.dst = b->block + b->offsets[row_keys[q]];
          job.src_stride = (uint32_t)f.stride;
          job.row_bytes = (uint32_t)f.row_bytes;
          job.vec_log2 = (uint8_t)v;
          job.epr = (uint16_t)(f.row_bytes >> v);
          int lpr = 0;
          while ((1 << lpr) < job.epr && lpr < 5) ++lpr;
          job.lpr_log2 = (uint8_t)lpr;
          job.n_coliter = (uint16_t)((job.epr + (1 << lpr) - 1) >> lpr);
          job.slot = (uint8_t)k.slot;
        }
        if (gp.n_jobs == 0) break;
        gathers.push_back([=](int64_t begin, int64_t end, cudaStream_t st) mutable -> int {
          gp.row_begin = begin;
          gp.row_end = end;
          const int64_t n_warp_tiles = (end - begin + 31) / 32;
          const unsigned grid = (unsigned)std::min<int64_t>((n_warp_tiles + 7) / 8, (int64_t)ds->sm_count * 32);
          static const void* const kWidth[5] = {(const void*)gather_rows_kernel<uint8_t>, (const void*)gather_rows_kernel<uint16_t>,
              (const void*)gather_rows_kernel<uint32_t>, (const void*)gather_rows_kernel<uint2>, (const void*)gather_rows_kernel<uint4>};
          void* args[] = {(void*)&gp};
          (void)cudaLaunchKernel(kWidth[v], dim3(grid), dim3(kRelabelThreads), args, 0, st);   // reported below
          if (cudaGetLastError() != cudaSuccess) return fail(OGB_ERR_CUDA, "gather_rows_kernel launch failed");
          b->kernel_names.push_back("gather_rows_kernel");
          b->launches++;
          return 0;
        });
      }
    }
    if (!*b->dominant) b->dominant = "gather_rows_kernel";   // no row gather outranks it
    return 0;
  }
  // image keys: frame stacking + crop fused into the gather; one launch per field and stack depth
  int prepare_frame_gathers() {
    using namespace ogb;
    std::vector<size_t> frame_keys;
    for (size_t i = 0; i < plan.size(); ++i)
      if (plan[i].route == ROUTE_FRAMES && plan[i].alias_of < 0) frame_keys.push_back(i);
    std::vector<bool> taken(frame_keys.size(), false);
    const char* tma_name = nullptr;   // the first TMA launch's kernel
    for (size_t a = 0; a < frame_keys.size(); ++a) {
      if (taken[a]) continue;
      const KeyPlan& ka = plan[frame_keys[a]];
      const Field& f = ds->fields[(size_t)ka.field];
      FramesParams fp;
      memset(&fp, 0, sizeof(fp));
      fp.vec_rows = b->vec_rows;
      fp.vec_init = b->vec_init;
      fp.crop = b->crop;
      fp.total_rows = total;
      if (f.ndim == 4) { fp.H = (int)f.shape[1]; fp.W = (int)f.shape[2]; fp.inner_bytes = (int)(f.shape[3] * f.itemsize); }
      else {  // stacking of non-image rows: concatenate on the last axis, everything before it is "pixels"
        int64_t outer = 1;
        for (int d = 1; d < f.ndim - 1; ++d) outer *= f.shape[d];
        fp.H = 1; fp.W = (int)outer; fp.inner_bytes = (int)((f.ndim > 1 ? f.shape[f.ndim - 1] : 1) * f.itemsize);
      }
      // rb == 0: not a TMA shape, or no band height in (padding, 32] divides H; the generic kernel serves those
      const int rb = tma_eligible(f, cfg, ka.fs) && crop_pad <= 4 ? band_rows_for(fp.H, crop_pad) : 0;
      for (size_t c = a; c < frame_keys.size() && fp.n_jobs < kMaxFrameJobs; ++c) {
        const KeyPlan& kc = plan[frame_keys[c]];
        if (taken[c] || kc.field != ka.field || kc.fs != ka.fs) continue;
        taken[c] = true;
        FrameJob& job = fp.jobs[fp.n_jobs++];
        job.src = f.dptr;
        job.dst = b->block + b->offsets[frame_keys[c]];
        job.src_row_stride = (int64_t)f.stride;
        job.slot = kc.slot;
        job.crop = kc.crop;
        job.fs = kc.fs;
      }
      if (rb > 0) {
        fp.band_rows = rb;
        fp.n_bands = fp.H / rb;
        CUtensorMap tm;
        OGB_TRY(get_tmap(s, ka.field, rb, &tm));
        const int band_bytes = rb * fp.W * 3;
        const size_t smem = (size_t)ka.fs * (ogb::frame_stride_bytes(band_bytes) + band_bytes);
        // (the last instance serves every stack deeper than three)
        const KernelChoice k = ka.fs == 1 ? frames_instance<1>() : ka.fs == 2 ? frames_instance<2>() : ka.fs == 3 ? frames_instance<3>() : frames_instance<4>();
        if (!tma_name) tma_name = k.name;
        gathers.push_back([=](int64_t begin, int64_t end, cudaStream_t st) mutable -> int {
          fp.row_begin = begin;
          fp.row_end = end;
          const int64_t n_items = (end - begin) * fp.n_jobs * fp.n_bands;
          if (n_items > 0x7fffffff) return fail(OGB_ERR_UNSUPPORTED, "too many frame tiles in one launch");
          OGB_CUDA(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
          void* args[] = {(void*)&tm, (void*)&fp};
          (void)cudaLaunchKernel(k.fn, dim3((unsigned)n_items), dim3(kFramesThreads), args, smem, st);   // reported below
          OGB_CUDA(cudaGetLastError());
          b->kernel_names.push_back(k.name);
          b->launches++;
          return 0;
        });
      } else {
        const int v = largest_vec_log2((size_t)fp.inner_bytes, f.stride);
        gathers.push_back([=](int64_t begin, int64_t end, cudaStream_t st) mutable -> int {
          fp.row_begin = begin;
          fp.row_end = end;
          for (int jj = 0; jj < fp.n_jobs; ++jj) {
            gather_frames_generic_kernel<<<ds->sm_count * 8, 256, 0, st>>>(fp, jj, v);
            if (cudaGetLastError() != cudaSuccess) return fail(OGB_ERR_CUDA, "gather_frames_generic_kernel launch failed");
            b->kernel_names.push_back("gather_frames_generic_kernel");
            b->launches++;
          }
          return 0;
        });
      }
    }
    b->dominant = tma_name ? tma_name : "gather_frames_generic_kernel";
    return 0;
  }
  // Issues the launches row chunk by row chunk: the index kernel (or the fused launch) on `first`, the gathers on the
  // sampler's stream behind it.
  int issue() {
    const bool timeline = ab().timeline;   // debug: when did each phase run on the device
    auto stamp = [&](cudaStream_t st) {
      if (!timeline) return;
      cudaEvent_t ev;
      cudaEventCreate(&ev);
      cudaEventRecord(ev, st);
      g_timeline.push_back(ev);
    };
    // profile mode: events around the launches `launch` makes on `st` (those of the dominant kernel)
    auto profiled = [&](bool on, cudaStream_t st, auto&& launch) -> int {
      if (on) {
        cudaEventCreate(&b->prof_begin);
        cudaEventCreate(&b->prof_end);
        cudaEventRecord(b->prof_begin, st);
      }
      const int rc = launch();
      if (!rc && on) cudaEventRecord(b->prof_end, st);
      return rc;
    };
    // row chunks (multiples of 32 rows, each at least kChunkMinRows): one unless the batch is headed for host memory
    constexpr int64_t kChunkMinRows = 16384;
    int n_chunks = 1;
    if (s->host_chunks > 1 && !draws && total >= 2 * kChunkMinRows) n_chunks = (int)std::min<int64_t>(std::min(s->host_chunks, kMaxChunks), total / kChunkMinRows);
    const int64_t chunk_rows = ((total + n_chunks - 1) / n_chunks + 31) / 32 * 32;
    const bool gathers_dominate = !gathers.empty() && !fused;
    for (int c = 0; c < n_chunks; ++c) {
      const int64_t begin = (int64_t)c * chunk_rows, end = std::min<int64_t>(total, begin + chunk_rows);
      if (begin >= end) break;
      const bool prof = s->profile && c == 0 && n_chunks == 1;
      stamp(first);
      int rc = profiled(prof && !gathers_dominate, first, [&] { return fused ? fused(begin, end, first) : index(begin, end, first); });
      if (rc) return rc;
      stamp(first);
      if (first != s->stream && join_streams(s, first, s->stream)) return fail(OGB_ERR_CUDA, "stream join failed");
      stamp(s->stream);
      rc = profiled(prof && gathers_dominate, s->stream, [&] {
        int r = 0;
        for (size_t q = 0; q < gathers.size() && !r; ++q) r = gathers[q](begin, end, s->stream);
        return r;
      });
      if (rc) return rc;
      stamp(s->stream);
      if (n_chunks > 1) {
        cudaEvent_t done;
        if (cudaEventCreateWithFlags(&done, cudaEventDisableTiming) != cudaSuccess || cudaEventRecord(done, s->stream) != cudaSuccess)
          return fail(OGB_ERR_CUDA, "chunk event failed");
        b->chunk_done.push_back(done);
        b->chunk_end.push_back(end);
      }
    }
    return 0;
  }
};

int run_sample(ogb_sampler* s, const RunSpec& spec, int64_t batch_size, int32_t n_batches, const int64_t* idxs, int32_t evaluation,
               const ogb_draws* draws, ogb_batch** out) {
  PhaseClock phase;
  if (!s || !out) return fail(OGB_ERR_INVALID, "ogb_sampler_sample: null argument");
  const ogb_dataset* ds = s->ds;
  Run r{s, ds, s->cfg, spec, *spec.plan, batch_size, batch_size * (int64_t)n_batches, n_batches, idxs, draws};
  OGB_TRY(r.check(evaluation != 0));
  DeviceGuard device_guard(ds->device);
  OGB_CUDA(device_guard.status);
  std::lock_guard<std::mutex> lock(s->mu);
  phase.mark();   // checks

  bool any_frames = false, any_long = false, any_async = false;   // image keys; row keys over 16 bytes, and on the cp.async path
  for (const KeyPlan& k : r.plan) {
    if (k.alias_of >= 0) continue;
    any_frames |= k.route == ROUTE_FRAMES;
    if (k.route != ROUTE_ROW || ds->fields[(size_t)k.field].row_bytes <= 16) continue;
    any_long = true;
    any_async |= async_reachable(ds, ds->fields[(size_t)k.field]);
  }
  const bool want_init = any_frames && s->cfg.frame_stack > 1;
  r.new_batch(want_init, any_frames);
  ogb_batch* b = r.b;
  auto bail = [&](int code) { batch_unref(b); return code; };
  // When some key goes through the cp.async row gather, the index algebra is fused into that launch (one kernel per
  // sample() for vector observations); otherwise the index kernel runs on its own.
  // Measured on B200 with ~1M-row launches: fused wins for GCDataset shapes (C2 0.201 vs 0.216 ms, C5 0.356 vs 0.372)
  // and loses for the heavier HGC algebra with its 16-row items (C3 0.757 vs 0.730 ms), so big HGC launches stay split;
  // small launches always fuse (one kernel launch less).  Image batches keep the index kernel apart (it overlaps the
  // previous call's frame gathers).  OGB_FUSE=0/1 forces either.
  const int fuse_env = ab().fuse;
  bool fuse = any_async && (fuse_env >= 0 ? fuse_env != 0 : (!any_frames && (r.total < kOverlapMinRows || spec.kind != OGB_KIND_HGC)));
  // Phase-one work (uploads of validation draws, the index kernel) goes to `first`: for big launches that is the
  // auxiliary stream, so that the index kernel of this call overlaps the gathers of the previous call, which are
  // still running on the main stream.  The recycled block only has to wait for its own previous owner.
  // Image batches are few rows with long gathers: their (latency-bound) index kernel always goes to the auxiliary
  // stream, where it runs under the frame gathers of the previous call.
  // (any_frames || any_long: is there a gather launch for the index kernel to hide under?)
  const bool use_aux = !fuse && (any_frames || any_long) && (r.total >= kOverlapMinRows || any_frames);
  if (use_aux) {
    int rc = ensure_aux(s);
    if (rc) return bail(rc);
  }
  cudaStream_t first = r.first = use_aux ? s->aux_stream : s->stream;
  phase.mark();   // batch + layout
  {
    std::vector<cudaEvent_t> free_after;
    int rc = block_take(s, b->block_bytes, &b->block, &b->block_bytes, &free_after);
    for (cudaEvent_t ev : free_after) {
      cudaStreamWaitEvent(first, ev, 0);
      if (first != s->stream) cudaStreamWaitEvent(s->stream, ev, 0);
      cudaEventDestroy(ev);
    }
    if (rc) return bail(rc);
  }
  uint8_t* base = b->block;
  phase.mark();   // block
  if (s->canary) {
    cudaMemsetAsync(base, 0xA5, b->block_bytes, first);
    // the gathers on the main stream must not start before the fill has finished
    if (first != s->stream) join_streams(s, first, s->stream);
  }
  b->vec_rows = (int32_t*)(base + r.off_rows);
  if (any_frames) b->crop = (int8_t*)(base + r.off_crop);
  if (want_init) b->vec_init = (int32_t*)(base + r.off_init);
  if (r.total > 0) {   // an empty batch is legal (np.random.randint(n, size=0) in the reference): every key with zero rows, no launch
    ogb::RelabelParams& p = r.p;
    int rc = r.fill_params();
    if (rc) return bail(rc);
    phase.mark();   // params
    std::vector<size_t> lsu_keys;
    const std::vector<SpanJob> spans = classify_rows(ds, r.plan, base, b->offsets, &p, &lsu_keys);
    fuse = fuse && !spans.empty();
    const bool any_gather = !spans.empty() || !lsu_keys.empty() || any_frames;   // a launch after the index kernel
    const bool point_record = is_point_record(s, spec, p, any_gather);
    // the index vectors only go to memory when a later launch (or the debug interface) reads them; a fused launch that
    // leaves span jobs to a second row-gather launch sets it in prepare_row_gathers, where the launch split is known
    p.write_vecs = ((!fuse && !spans.empty()) || !lsu_keys.empty() || any_frames || s->debug) ? 1 : 0;
    phase.mark();   // classify
    // Every launch.  Each family names the dominant kernel -- the one that moves the batch's bytes -- as it is prepared, in
    // rising precedence: the row gather (fused or not), the register-staged one, the frame gather; when there is none of
    // them, the index kernel names itself as it launches (datasets whose rows are all <= 16 bytes).  (The index launch
    // takes the parameters as they are: they change only for a fused launch, which replaces it.)
    const int flavour = spec.kind == OGB_KIND_GC ? ogb::FLAVOUR_GC : (spec.kind == OGB_KIND_HGC ? ogb::FLAVOUR_HGC : ogb::FLAVOUR_PLAIN);
    r.index = index_launch(s, b, p, draws != nullptr, flavour, point_record, !any_gather);
    rc = r.prepare_row_gathers(spans, fuse, draws != nullptr, flavour);
    if (!rc && !lsu_keys.empty()) rc = r.prepare_lsu_gathers(lsu_keys);
    if (!rc && any_frames) rc = r.prepare_frame_gathers();
    // every launch after a fused one reads the index vectors from memory: the fused launch must have stored them
    if (!rc && r.fused && !r.gathers.empty() && !p.write_vecs)
      rc = fail(OGB_ERR_UNSUPPORTED, "internal: a fused launch followed by %zu gather launches does not store the index vectors",
                r.gathers.size());
    if (rc) return bail(rc);
    phase.mark();   // prepare
    rc = r.issue();
    if (rc) return bail(rc);
  }
  if (cudaEventCreateWithFlags(&b->ready, cudaEventDisableTiming) != cudaSuccess || cudaEventRecord(b->ready, s->stream) != cudaSuccess)
    return bail(fail(OGB_ERR_CUDA, "ready event failed"));
  if (!draws) s->counter += (uint64_t)n_batches;
  *out = b;
  if (r.total == 0) return 0;
  phase.mark();   // launch + event
  if (g_phases.on) ++g_phases.calls;
  return 0;
}

// One key of rows `idxs`: the observations -- cropped with the injected shifts and `crop_padding` when that is >= 0 -- or
// the goal observations (get_observations, get_goal_observations, augment).
int run_rows(ogb_sampler* s, bool goal, int crop_padding, const int64_t* idxs, int64_t n, const ogb_draws* draws, ogb_batch** out) {
  PlanBuilder pb;
  pb.ds = s->ds;
  pb.cfg = &s->cfg;
  pb.crop_possible = crop_padding >= 0;
  for (int v = 0; v < ogb::kMaxSlots; ++v) pb.slot_canon[v] = v;
  if (goal) pb.goal_key("goal_observations", ogb::SLOT_IDX, false);
  else pb.obs_key("observations", ogb::SLOT_IDX, crop_padding >= 0);
  RunSpec spec;
  spec.kind = OGB_KIND_PLAIN;
  spec.plan = &pb.keys;
  spec.n_slots = 2;
  spec.crop_padding = crop_padding;
  return run_sample(s, spec, n, 1, idxs, draws ? 0 : 1, draws, out);
}

}  // namespace

extern "C" {

int ogb_sampler_sample(ogb_sampler* s, int64_t batch_size, int32_t n_batches, const int64_t* idxs, int32_t evaluation,
                       const ogb_draws* draws, ogb_batch** out) try {
  if (!s || !out) return fail(OGB_ERR_INVALID, "ogb_sampler_sample: null argument");
  if (s->kind == OGB_KIND_ATC) return fail(OGB_ERR_INVALID, "an ATC sampler is sampled with ogb_sampler_sample_atc");
  RunSpec spec;
  spec.kind = s->kind;
  spec.plan = &s->plan[evaluation ? 1 : 0];
  spec.n_slots = s->n_slots;
  spec.trl = s->cfg.trl != 0 && s->kind == OGB_KIND_GC;
  if (s->trl_rows.dev) {
    spec.choice_table = s->trl_rows.dev;
    spec.n_choices = (int64_t)s->trl_rows.host.size();
  }
  return run_sample(s, spec, batch_size, n_batches, idxs, evaluation, draws, out);
} OGB_CATCH_ALL

// get_observations / get_goal_observations (datasets.py:341-357): rows `idxs` of the observations (frame-stacked as
// the sampler's config says) or of the goal representation.
int ogb_sampler_gather(ogb_sampler* s, int32_t which, const int64_t* idxs, int64_t n, ogb_batch** out) try {
  if (!s || (!idxs && n > 0) || !out || n < 0) return fail(OGB_ERR_INVALID, "ogb_sampler_gather: bad argument");
  static const int64_t no_rows = 0;
  if (n == 0) idxs = &no_rows;   // an empty gather is legal (observations[np.zeros(0, int)]); run_sample wants a non-null pointer
  if (which < 0 || which > 1) return fail(OGB_ERR_INVALID, "which must be 0 (observations) or 1 (goal observations)");
  if (s->cfg.frame_stack > 0 && s->term_host.empty()) return fail(OGB_ERR_INVALID, "frame stacking needs trajectory boundaries");
  return run_rows(s, which == 1, -1, idxs, n, nullptr, out);
} OGB_CATCH_ALL

// GCDataset.augment (datasets.py:329-339) for one image array: rows `idxs` of the observations, each cropped with its
// own (cy, cx) shift after edge padding by `padding` (datasets.py:17-33).  `crop` is [n, 2] int64 (host), the
// reference's randint(0, 2 * padding + 1, (n, 2)).
int ogb_sampler_gather_cropped(ogb_sampler* s, const int64_t* idxs, int64_t n, const int64_t* crop, int32_t padding, ogb_batch** out) try {
  if (!s || !idxs || !crop || !out || n < 1 || padding < 0) return fail(OGB_ERR_INVALID, "ogb_sampler_gather_cropped: bad argument");
  if (padding > 127) return fail(OGB_ERR_INVALID, "crop padding %d out of [0, 127]", padding);   // int8 shifts, as in ogb_sampler_create
  for (int64_t r = 0; r < 2 * n; ++r)
    if (crop[r] < 0 || crop[r] > 2 * (int64_t)padding) return fail(OGB_ERR_INVALID, "crop shift out of [0, 2 * padding]");
  ogb_draws d;
  memset(&d, 0, sizeof(d));
  d.has_aug_coin = 1;
  d.aug_coin = 0.0;
  d.crop = crop;
  return run_rows(s, false, padding, idxs, n, &d, out);
} OGB_CATCH_ALL

}  // extern "C"

namespace {
struct GoalsParams {
  ogb::RelabelParams r;
  const int64_t* idxs;
  int64_t* out;
  int64_t n;
};

// GCDataset.sample_goals (datasets.py:296-327) for explicit rows
template <bool kInject>
__global__ void __launch_bounds__(256) sample_goals_kernel(const __grid_constant__ GoalsParams q) {
  using namespace ogb;
  const RelabelParams& p = q.r;
  const SegView seg{p.seg_bucket, p.seg_table};
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < q.n; g += (int64_t)gridDim.x * blockDim.x) {
    const int32_t i = (int32_t)q.idxs[g];
    const int tl = lower_bound_bucketed(p.term, p.term_bucket, p.term_shift, i);
    const int32_t fin = __ldg(p.term + tl);
    int32_t goal;
    if (kInject) {
      goal = pick_goal_injected<false>(p, seg, 0, i, fin, g);
    } else {
      const uint4 w0 = draw4(p.key, p.batch0, (uint32_t)g, PURPOSE_IDX);
      const uint4 gb = draw4(p.key, p.batch0, (uint32_t)g, PURPOSE_GOAL);
      goal = pick_goal_philox<false>(p, seg, 0, i, fin, make_uint2(w0.z, w0.w), make_uint2(gb.x, gb.y));
    }
    q.out[g] = goal;
  }
}

// HGCDataset.compute_high_next_idxs (datasets.py:478-491)
__global__ void high_next_kernel(const int64_t* __restrict__ idxs, const int64_t* __restrict__ fin, const int64_t* __restrict__ goal,
                                 int64_t k, int64_t n, int64_t* __restrict__ next, int64_t* __restrict__ steps) {
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x) {
    int64_t st = fin[g] - idxs[g] < k ? fin[g] - idxs[g] : k;
    const int64_t d = goal[g] - idxs[g];
    if (0 <= d && d < st) st = d;
    next[g] = idxs[g] + st;
    steps[g] = st;
  }
}

struct DeviceScratch {   // a few temporary device arrays of a helper call
  std::vector<void*> ptrs;
  ~DeviceScratch() { for (void* q : ptrs) cudaFree(q); }
  template <typename T>
  int upload(const T* host, int64_t n, T** out) {
    OGB_CUDA(cudaMalloc((void**)out, (size_t)std::max<int64_t>(n, 1) * sizeof(T)));
    ptrs.push_back(*out);
    if (host) OGB_CUDA(cudaMemcpy(*out, host, (size_t)n * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
  }
};
}  // namespace

extern "C" {

int ogb_sampler_table_info(const ogb_sampler* s, ogb_table_info* info) try {
  if (!s || !info) return fail(OGB_ERR_INVALID, "ogb_sampler_table_info: null argument");
  const int64_t n_choices = n_choices_for(s->ds, s->trl_rows.dev, (int64_t)s->trl_rows.host.size());
  ogb::RelabelParams p;
  memset(&p, 0, sizeof(p));
  set_row_tables(s, s->trl_rows.dev, n_choices, &p);
  memset(info, 0, sizeof(*info));
  info->valid_mode = p.valid_mode;
  info->seg_shift = s->seg_shift;
  info->n_seg_table = s->n_seg_table;
  info->gap_shift = s->ds->gap_shift;
  info->term_shift = s->term_shift;
  info->n_choices = n_choices;
  return 0;
} OGB_CATCH_ALL

int ogb_sampler_sample_goals(ogb_sampler* s, const int64_t* idxs, int64_t n, double p_curgoal, double p_trajgoal, int32_t geom_sample,
                             double discount, const ogb_goal_draws* draws, int64_t* out_goal_idxs) try {
  using namespace ogb;
  if (!s || !idxs || !out_goal_idxs || n < 1) return fail(OGB_ERR_INVALID, "ogb_sampler_sample_goals: bad argument");
  if (s->term_host.empty()) return fail(OGB_ERR_INVALID, "this sampler has no trajectory boundaries");
  if (!(discount > 0.0 && discount < 1.0)) return fail(OGB_ERR_INVALID, "discount must be in (0, 1)");
  const ogb_dataset* ds = s->ds;
  for (int64_t r = 0; r < n; ++r)
    if (idxs[r] < 0 || idxs[r] >= ds->size) return fail(OGB_ERR_INDEX, "index %lld is out of bounds for axis 0 with size %lld", (long long)idxs[r], (long long)ds->size);
  const bool cur_only = p_curgoal == 1.0;
  const int64_t n_choices = n_choices_for(ds, s->trl_rows.dev, (int64_t)s->trl_rows.host.size());
  if (draws) {
    if (!draws->rand_pos || (geom_sample ? !draws->offset : !draws->dist) || (!cur_only && (!draws->u_traj || !draws->u_cur)))
      return fail(OGB_ERR_INVALID, "sample_goals: missing draws");
    for (int64_t r = 0; r < n; ++r)
      if (draws->rand_pos[r] < 0 || draws->rand_pos[r] >= n_choices) return fail(OGB_ERR_INDEX, "rand_pos out of range");
  }
  DeviceGuard device_guard(ds->device);
  OGB_CUDA(device_guard.status);
  std::lock_guard<std::mutex> lock(s->mu);
  GoalsParams q;
  memset(&q, 0, sizeof(q));
  RelabelParams& p = q.r;
  set_row_tables(s, s->trl_rows.dev, n_choices, &p);
  p.n_rows_ds = (int32_t)ds->size;
  p.goal[0] = goal_spec(p_curgoal, p_trajgoal, geom_sample != 0, discount);
  p.key = make_rng_key(s->seed, s->stream_id);
  p.batch0 = s->counter;
  DeviceScratch tmp;
  int64_t *d_idxs = nullptr, *d_out = nullptr;
  OGB_TRY(tmp.upload(idxs, n, &d_idxs));
  OGB_TRY(tmp.upload<int64_t>(nullptr, n, &d_out));
  q.idxs = d_idxs;
  q.out = d_out;
  q.n = n;
  if (draws) {
    int64_t *d_pos = nullptr, *d_off = nullptr;
    double *d_dist = nullptr, *d_ut = nullptr, *d_uc = nullptr;
    OGB_TRY(tmp.upload(draws->rand_pos, n, &d_pos));
    p.in_goal[0].rand_pos = d_pos;
    if (draws->offset) { OGB_TRY(tmp.upload(draws->offset, n, &d_off)); p.in_goal[0].offset = d_off; }
    if (draws->dist) { OGB_TRY(tmp.upload(draws->dist, n, &d_dist)); p.in_goal[0].dist = d_dist; }
    if (draws->u_traj) { OGB_TRY(tmp.upload(draws->u_traj, n, &d_ut)); p.in_goal[0].u_traj = d_ut; }
    if (draws->u_cur) { OGB_TRY(tmp.upload(draws->u_cur, n, &d_uc)); p.in_goal[0].u_cur = d_uc; }
  }
  const unsigned grid = (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)ds->sm_count * 8);
  if (draws) sample_goals_kernel<true><<<grid, 256, 0, s->stream>>>(q);
  else sample_goals_kernel<false><<<grid, 256, 0, s->stream>>>(q);
  OGB_CUDA(cudaGetLastError());
  OGB_CUDA(cudaMemcpyAsync(out_goal_idxs, d_out, (size_t)n * 8, cudaMemcpyDeviceToHost, s->stream));
  OGB_CUDA(cudaStreamSynchronize(s->stream));
  if (!draws) s->counter += 1;
  return 0;
} OGB_CATCH_ALL

int ogb_sampler_compute_high_next_idxs(ogb_sampler* s, const int64_t* idxs, const int64_t* final_state_idxs, const int64_t* goal_idxs,
                                       int64_t n, int64_t subgoal_steps, int64_t* out_next, int64_t* out_steps) try {
  if (!s || !idxs || !final_state_idxs || !goal_idxs || !out_next || !out_steps || n < 1)
    return fail(OGB_ERR_INVALID, "ogb_sampler_compute_high_next_idxs: bad argument");
  DeviceGuard device_guard(s->ds->device);
  OGB_CUDA(device_guard.status);
  std::lock_guard<std::mutex> lock(s->mu);
  DeviceScratch tmp;
  int64_t *d_i = nullptr, *d_f = nullptr, *d_g = nullptr, *d_n = nullptr, *d_s = nullptr;
  OGB_TRY(tmp.upload(idxs, n, &d_i));
  OGB_TRY(tmp.upload(final_state_idxs, n, &d_f));
  OGB_TRY(tmp.upload(goal_idxs, n, &d_g));
  OGB_TRY(tmp.upload<int64_t>(nullptr, n, &d_n));
  OGB_TRY(tmp.upload<int64_t>(nullptr, n, &d_s));
  high_next_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)s->ds->sm_count * 8), 256, 0, s->stream>>>(d_i, d_f, d_g, subgoal_steps, n, d_n, d_s);
  OGB_CUDA(cudaGetLastError());
  OGB_CUDA(cudaMemcpyAsync(out_next, d_n, (size_t)n * 8, cudaMemcpyDeviceToHost, s->stream));
  OGB_CUDA(cudaMemcpyAsync(out_steps, d_s, (size_t)n * 8, cudaMemcpyDeviceToHost, s->stream));
  OGB_CUDA(cudaStreamSynchronize(s->stream));
  return 0;
} OGB_CATCH_ALL

namespace {
// get_valid_atc_idxs (datasets.py:417-436): anchors i with i + k < size and i + k <= final_state(i), valid rows only
int atc_anchors(ogb_sampler* s, int64_t k, const std::vector<int32_t>** host, const int32_t** dev) {
  auto it = s->atc_tables.find(k);
  if (it == s->atc_tables.end()) {
    const ogb_dataset* ds = s->ds;
    ogb_sampler::AtcTable t;
    size_t ti = 0;
    for (int64_t i = 0; i < ds->size; ++i) {
      while (ti < s->term_host.size() && s->term_host[ti] < i) ++ti;   // final_state(i) = first terminal >= i
      if (!ds->valid_host.empty() && !ds->valid_host[(size_t)i]) continue;
      if (i + k >= ds->size || ti >= s->term_host.size()) continue;
      if (i + k <= (int64_t)s->term_host[ti]) t.host.push_back((int32_t)i);
    }
    if (t.host.empty()) return fail(OGB_ERR_INVALID, "No valid ATC indices found for k=%lld.", (long long)k);
    int rc = upload_vector(t.host, &t.dev);
    if (rc) return rc;
    it = s->atc_tables.emplace(k, std::move(t)).first;
  }
  if (host) *host = &it->second.host;
  if (dev) *dev = it->second.dev;
  return 0;
}
}  // namespace

int ogb_sampler_num_atc_anchors(ogb_sampler* s, int64_t k, int64_t* out) try {
  if (!s || !out) return fail(OGB_ERR_INVALID, "null argument");
  if (k < 0) return fail(OGB_ERR_INVALID, "k must be >= 0");
  DeviceGuard device_guard(s->ds->device);           // a new offset uploads its anchor table
  OGB_CUDA(device_guard.status);
  std::lock_guard<std::mutex> lock(s->mu);
  const std::vector<int32_t>* host;
  OGB_TRY(atc_anchors(s, k, &host, nullptr));
  *out = (int64_t)host->size();
  return 0;
} OGB_CATCH_ALL
int ogb_sampler_copy_atc_anchors(ogb_sampler* s, int64_t k, int64_t* out) try {
  if (!s || !out) return fail(OGB_ERR_INVALID, "null argument");
  DeviceGuard device_guard(s->ds->device);
  OGB_CUDA(device_guard.status);
  std::lock_guard<std::mutex> lock(s->mu);
  const std::vector<int32_t>* host;
  OGB_TRY(atc_anchors(s, k, &host, nullptr));
  for (size_t i = 0; i < host->size(); ++i) out[i] = (*host)[i];
  return 0;
} OGB_CATCH_ALL

// ATCDataset.sample (datasets.py:401-415): anchor rows for the temporal offset k, observations at idx and idx + k
int ogb_sampler_sample_atc(ogb_sampler* s, int64_t batch_size, int32_t n_batches, int64_t k, int32_t evaluation,
                           const ogb_draws* draws, ogb_batch** out) try {
  if (!s || !out) return fail(OGB_ERR_INVALID, "null argument");
  if (s->kind != OGB_KIND_ATC) return fail(OGB_ERR_INVALID, "not an ATC sampler");
  if (k < 0) return fail(OGB_ERR_INVALID, "k must be >= 0");
  const std::vector<int32_t>* host;
  const int32_t* dev;
  DeviceGuard device_guard(s->ds->device);
  OGB_CUDA(device_guard.status);
  {
    std::lock_guard<std::mutex> lock(s->mu);
    OGB_TRY(atc_anchors(s, k, &host, &dev));
  }
  RunSpec spec;
  spec.kind = OGB_KIND_ATC;
  spec.plan = &s->plan[evaluation ? 1 : 0];
  spec.n_slots = 2;
  spec.next_offset = k;
  spec.choice_table = dev;
  spec.n_choices = (int64_t)host->size();
  return run_sample(s, spec, batch_size, n_batches, nullptr, evaluation, draws, out);
} OGB_CATCH_ALL

int ogb_batch_num_keys(const ogb_batch* b, int32_t* out) try {
  if (!b || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = (int32_t)b->keys.size();
  return 0;
} OGB_CATCH_ALL

int ogb_batch_key_info(const ogb_batch* b, int32_t i, ogb_key_info* out) try {
  if (!b || !out || i < 0 || i >= (int32_t)b->keys.size()) return fail(OGB_ERR_INVALID, "bad key index");
  const KeyPlan& k = b->keys[(size_t)i];
  memset(out, 0, sizeof(*out));
  out->name = k.name.c_str();
  out->dtype = k.dtype;
  int nd = 0;
  if (b->n_batches > 1 || b->keep_axis) out->shape[nd++] = b->n_batches;
  out->shape[nd++] = b->batch;
  for (int d = 0; d < k.ndim_tail; ++d) out->shape[nd++] = k.tail[d];
  out->ndim = nd;
  out->offset = b->offsets[(size_t)i];
  out->device_ptr = b->block + out->offset;
  out->nbytes = (size_t)b->total_rows * k.row_bytes;
  out->alias_of = k.alias_of;
  return 0;
} OGB_CATCH_ALL

int ogb_batch_keep_leading_axis(ogb_batch* b, int32_t on) try {
  if (!b) return fail(OGB_ERR_INVALID, "null batch");
  b->keep_axis = on != 0;
  return 0;
} OGB_CATCH_ALL
int ogb_batch_nbytes(const ogb_batch* b, size_t* out) try {
  if (!b || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = b->keys_bytes;
  return 0;
} OGB_CATCH_ALL
int ogb_batch_device_block(const ogb_batch* b, void** out) try {
  if (!b || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = b->block;
  return 0;
} OGB_CATCH_ALL
int ogb_batch_launches(const ogb_batch* b, int32_t* out) try {
  if (!b || !out) return fail(OGB_ERR_INVALID, "null argument");
  *out = b->launches;
  return 0;
} OGB_CATCH_ALL
int ogb_batch_kernel_names(const ogb_batch* b, const char** buf, int32_t cap, int32_t* n_out) try {
  if (!b || !n_out || cap < 0 || (!buf && cap > 0)) return fail(OGB_ERR_INVALID, "ogb_batch_kernel_names: bad argument");
  *n_out = (int32_t)b->kernel_names.size();
  for (int32_t i = 0; i < cap && i < *n_out; ++i) buf[i] = b->kernel_names[(size_t)i];
  return 0;
} OGB_CATCH_ALL
int ogb_batch_dominant_kernel(ogb_batch* b, const char** name, float* ms) try {
  if (!b || !name || !ms) return fail(OGB_ERR_INVALID, "null argument");
  *name = b->dominant;
  *ms = -1.0f;
  if (b->prof_begin && b->prof_end) {
    OGB_CUDA(cudaEventSynchronize(b->prof_end));
    OGB_CUDA(cudaEventElapsedTime(ms, b->prof_begin, b->prof_end));
  }
  return 0;
} OGB_CATCH_ALL
int ogb_batch_sync(ogb_batch* b) try {
  if (!b) return fail(OGB_ERR_INVALID, "null batch");
  OGB_CUDA(cudaEventSynchronize(b->ready));
  if (b->idx_error) {
    int32_t flag = 0;
    OGB_CUDA(cudaMemcpy(&flag, b->idx_error, 4, cudaMemcpyDeviceToHost));
    if (flag) return fail(OGB_ERR_INDEX, "an index is out of bounds for axis 0 with size %lld", (long long)b->sampler->ds->size);
  }
  return 0;
} OGB_CATCH_ALL
int ogb_batch_wait_on_stream(ogb_batch* b, void* consumer_stream) try {
  if (!b) return fail(OGB_ERR_INVALID, "null batch");
  cudaStream_t c = (cudaStream_t)consumer_stream;
  if (c == b->sampler->stream) { b->main_stream_consumer = true; return 0; }
  DeviceGuard device_guard(b->sampler->ds->device);
  OGB_CUDA(device_guard.status);
  OGB_CUDA(cudaStreamWaitEvent(c, b->ready, 0));
  std::lock_guard<std::mutex> lock(b->mu);
  if (std::find(b->consumers.begin(), b->consumers.end(), c) == b->consumers.end()) b->consumers.push_back(c);
  return 0;
} OGB_CATCH_ALL
// D2H of the whole block in two calls.  `begin` only enqueues: the copy runs on a stream of its own behind the batch's
// `ready` event, not on the sampler's stream, so a caller that has already launched the NEXT batch gets that launch's
// upload and kernels under this copy instead of behind it -- and copies begun one after the other queue back to back on
// the copy engine (Prefetcher: launch k+1 and begin its copy, then end copy k).  `end` host-waits and reports the
// deferred index check.
int ogb_batch_copy_to_host_begin(ogb_batch* b, void* dst, size_t nbytes) try {
  if (!b || !dst) return fail(OGB_ERR_INVALID, "null argument");
  if (nbytes < b->keys_bytes) return fail(OGB_ERR_INVALID, "host buffer too small: %zu < %zu", nbytes, b->keys_bytes);
  if (b->copied) return fail(OGB_ERR_INVALID, "a copy of this batch has already been begun");
  ogb_sampler* s = b->sampler;
  DeviceGuard device_guard(s->ds->device);
  OGB_CUDA(device_guard.status);
  std::lock_guard<std::mutex> lock(s->mu);
  if (!s->copy_stream) OGB_CUDA(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
  if (b->idx_error) {
    if (!s->h_flags) {
      OGB_CUDA(cudaHostAlloc((void**)&s->h_flags, sizeof(int32_t) * ogb_sampler::kFlagSlots, cudaHostAllocDefault));
      memset(s->h_flags, 0, sizeof(int32_t) * ogb_sampler::kFlagSlots);
    }
    b->h_idx_flag = s->h_flags + (s->flag_seq++ % ogb_sampler::kFlagSlots);
    *b->h_idx_flag = 0;
  }
  if (b->chunk_done.size() > 1) {
    // pipelined: chunk c's rows of every key travel as soon as chunk c's kernels are done, while the kernels of chunk
    // c+1 are still running
    int64_t begin = 0;
    for (size_t c = 0; c < b->chunk_done.size(); ++c) {
      const int64_t end = b->chunk_end[c];
      OGB_CUDA(cudaStreamWaitEvent(s->copy_stream, b->chunk_done[c], 0));
      for (size_t i = 0; i < b->keys.size(); ++i) {
        if (b->keys[i].alias_of >= 0) continue;
        const size_t rb = b->keys[i].row_bytes, off = b->offsets[i] + (size_t)begin * rb;
        OGB_CUDA(cudaMemcpyAsync((uint8_t*)dst + off, b->block + off, (size_t)(end - begin) * rb, cudaMemcpyDeviceToHost, s->copy_stream));
      }
      begin = end;
    }
  } else {
    OGB_CUDA(cudaStreamWaitEvent(s->copy_stream, b->ready, 0));
    OGB_CUDA(cudaMemcpyAsync(dst, b->block, b->keys_bytes, cudaMemcpyDeviceToHost, s->copy_stream));
  }
  // (the deferred index check covers chunked launches too: every chunk's kernels are done by the time this copy runs)
  if (b->idx_error) OGB_CUDA(cudaMemcpyAsync((void*)b->h_idx_flag, b->idx_error, 4, cudaMemcpyDeviceToHost, s->copy_stream));
  OGB_CUDA(cudaEventCreateWithFlags(&b->copied, cudaEventDisableTiming));
  OGB_CUDA(cudaEventRecord(b->copied, s->copy_stream));
  return 0;
} OGB_CATCH_ALL
int ogb_batch_copy_to_host_end(ogb_batch* b) try {
  if (!b) return fail(OGB_ERR_INVALID, "null argument");
  if (!b->copied) return fail(OGB_ERR_INVALID, "no copy of this batch has been begun");
  ogb_sampler* s = b->sampler;
  DeviceGuard device_guard(s->ds->device);
  OGB_CUDA(device_guard.status);
  OGB_CUDA(cudaEventSynchronize(b->copied));
  cudaEventDestroy(b->copied);
  b->copied = nullptr;
  const bool bad = b->h_idx_flag != nullptr && *b->h_idx_flag != 0;
  b->h_idx_flag = nullptr;
  if (bad) return fail(OGB_ERR_INDEX, "an index is out of bounds for axis 0 with size %lld", (long long)s->ds->size);
  return 0;
} OGB_CATCH_ALL
int ogb_batch_copy_to_host(ogb_batch* b, void* dst, size_t nbytes) try {
  const int rc = ogb_batch_copy_to_host_begin(b, dst, nbytes);
  return rc ? rc : ogb_batch_copy_to_host_end(b);
} OGB_CATCH_ALL
int ogb_batch_copy_key_to_host(ogb_batch* b, int32_t i, void* dst, size_t nbytes) try {
  if (!b || !dst || i < 0 || i >= (int32_t)b->keys.size()) return fail(OGB_ERR_INVALID, "bad argument");
  const size_t need = (size_t)b->total_rows * b->keys[(size_t)i].row_bytes;
  if (nbytes < need) return fail(OGB_ERR_INVALID, "host buffer too small: %zu < %zu", nbytes, need);
  DeviceGuard device_guard(b->sampler->ds->device);
  OGB_CUDA(device_guard.status);
  OGB_CUDA(cudaMemcpyAsync(dst, b->block + b->offsets[(size_t)i], need, cudaMemcpyDeviceToHost, b->sampler->stream));
  OGB_CUDA(cudaStreamSynchronize(b->sampler->stream));
  return 0;
} OGB_CATCH_ALL
// one batch of a multi-batch launch (see ogb_batch_dlpack_slice), D2H, synchronous
int ogb_batch_copy_slice_to_host(ogb_batch* b, int32_t i, int64_t batch_index, void* dst, size_t nbytes) try {
  if (!b || !dst || i < 0 || i >= (int32_t)b->keys.size()) return fail(OGB_ERR_INVALID, "bad argument");
  if (batch_index < 0 || batch_index >= b->n_batches) return fail(OGB_ERR_INDEX, "batch %lld of %d", (long long)batch_index, b->n_batches);
  const size_t need = (size_t)b->batch * b->keys[(size_t)i].row_bytes;
  if (nbytes < need) return fail(OGB_ERR_INVALID, "host buffer too small: %zu < %zu", nbytes, need);
  DeviceGuard device_guard(b->sampler->ds->device);
  OGB_CUDA(device_guard.status);
  OGB_CUDA(cudaMemcpyAsync(dst, b->block + b->offsets[(size_t)i] + (size_t)batch_index * need, need, cudaMemcpyDeviceToHost, b->sampler->stream));
  OGB_CUDA(cudaStreamSynchronize(b->sampler->stream));
  return 0;
} OGB_CATCH_ALL
// debug (ogb_sampler_set_debug(s, 2)): bytes of the key area that belong to no key must still hold the 0xA5 fill
int ogb_batch_check_gaps(ogb_batch* b, int64_t* n_bad) try {
  if (!b || !n_bad) return fail(OGB_ERR_INVALID, "null argument");
  if (!b->sampler->canary) return fail(OGB_ERR_INVALID, "the sampler was not put into canary mode before this batch was drawn");
  std::vector<uint8_t> host(b->keys_bytes);
  DeviceGuard device_guard(b->sampler->ds->device);
  OGB_CUDA(device_guard.status);
  OGB_CUDA(cudaMemcpyAsync(host.data(), b->block, host.size(), cudaMemcpyDeviceToHost, b->sampler->stream));
  OGB_CUDA(cudaStreamSynchronize(b->sampler->stream));
  std::vector<uint8_t> owned(host.size(), 0);
  for (size_t i = 0; i < b->keys.size(); ++i) {
    if (b->keys[i].alias_of >= 0) continue;
    const size_t n = (size_t)b->total_rows * b->keys[i].row_bytes;
    std::fill(owned.begin() + (long)b->offsets[i], owned.begin() + (long)(b->offsets[i] + n), 1);
  }
  int64_t bad = 0;
  for (size_t k = 0; k < host.size(); ++k) bad += (!owned[k] && host[k] != 0xA5) ? 1 : 0;
  *n_bad = bad;
  return 0;
} OGB_CATCH_ALL
int ogb_batch_index_vector(ogb_batch* b, int32_t slot, int64_t* dst_host) try {
  if (!b || !dst_host) return fail(OGB_ERR_INVALID, "null argument");
  if (slot < 0 || slot >= b->n_slots) return fail(OGB_ERR_INVALID, "bad slot");
  std::vector<int32_t> tmp((size_t)b->total_rows);
  DeviceGuard device_guard(b->sampler->ds->device);
  OGB_CUDA(device_guard.status);
  OGB_CUDA(cudaMemcpyAsync(tmp.data(), b->vec_rows + (size_t)slot * b->total_rows, tmp.size() * 4, cudaMemcpyDeviceToHost, b->sampler->stream));
  OGB_CUDA(cudaStreamSynchronize(b->sampler->stream));
  for (size_t i = 0; i < tmp.size(); ++i) dst_host[i] = tmp[i];
  return 0;
} OGB_CATCH_ALL
int ogb_batch_crop_shifts(ogb_batch* b, int64_t* dst_host) try {
  if (!b || !dst_host) return fail(OGB_ERR_INVALID, "null argument");
  if (!b->crop) return fail(OGB_ERR_INVALID, "this batch has no image keys, hence no crop shifts");
  std::vector<int8_t> tmp((size_t)b->total_rows * 2);
  DeviceGuard device_guard(b->sampler->ds->device);
  OGB_CUDA(device_guard.status);
  OGB_CUDA(cudaMemcpyAsync(tmp.data(), b->crop, tmp.size(), cudaMemcpyDeviceToHost, b->sampler->stream));
  OGB_CUDA(cudaStreamSynchronize(b->sampler->stream));
  const int pad = b->sampler->cfg.crop_padding;
  for (size_t i = 0; i < tmp.size(); ++i) dst_host[i] = tmp[i] == -128 ? -1 : tmp[i] + pad;
  return 0;
} OGB_CATCH_ALL

static void dl_deleter(DLManagedTensor_* t) {
  if (!t) return;
  ogb_batch* b = (ogb_batch*)t->manager_ctx;
  delete[] t->dl_tensor.shape;
  delete t;
  batch_unref(b);
}

int ogb_batch_dlpack(ogb_batch* b, int32_t i, void** out) try {
  if (!b || !out || i < 0 || i >= (int32_t)b->keys.size()) return fail(OGB_ERR_INVALID, "bad key index");
  ogb_key_info info;
  OGB_TRY(ogb_batch_key_info(b, i, &info));
  DLManagedTensor_* t = new DLManagedTensor_();
  t->dl_tensor.data = info.device_ptr;
  t->dl_tensor.device.device_type = 2;  // kDLCUDA
  t->dl_tensor.device.device_id = b->sampler->ds->device;
  t->dl_tensor.ndim = info.ndim;
  uint8_t code = 0;
  switch (info.dtype) {
    case OGB_U8: case OGB_U16: case OGB_U32: case OGB_U64: code = 1; break;
    case OGB_F16: case OGB_F32: case OGB_F64: code = 2; break;
    case OGB_BOOL: code = 6; break;
    default: code = 0; break;
  }
  t->dl_tensor.dtype.code = code;
  t->dl_tensor.dtype.bits = (uint8_t)(dtype_size(info.dtype) * 8);
  t->dl_tensor.dtype.lanes = 1;
  t->dl_tensor.shape = new int64_t[(size_t)std::max(info.ndim, 1)];
  for (int d = 0; d < info.ndim; ++d) t->dl_tensor.shape[d] = info.shape[d];
  t->dl_tensor.strides = nullptr;  // compact row-major
  t->dl_tensor.byte_offset = 0;
  t->manager_ctx = b;
  t->deleter = dl_deleter;
  b->refs.fetch_add(1);
  *out = t;
  return 0;
} OGB_CATCH_ALL
// One batch of a multi-batch launch as a tensor of its own ([batch, ...], the leading axis dropped): what a look-ahead
// sampler hands out for the i-th of K batches it drew in one launch.  Same ownership as ogb_batch_dlpack.
int ogb_batch_dlpack_slice(ogb_batch* b, int32_t i, int64_t batch_index, void** out) try {
  if (!b || !out || i < 0 || i >= (int32_t)b->keys.size()) return fail(OGB_ERR_INVALID, "bad key index");
  if (batch_index < 0 || batch_index >= b->n_batches) return fail(OGB_ERR_INDEX, "batch %lld of %d", (long long)batch_index, b->n_batches);
  void* whole = nullptr;
  OGB_TRY(ogb_batch_dlpack(b, i, &whole));
  DLManagedTensor_* t = (DLManagedTensor_*)whole;
  const KeyPlan& k = b->keys[(size_t)i];
  const bool has_axis = b->n_batches > 1 || b->keep_axis;
  if (has_axis) {
    for (int d = 1; d < t->dl_tensor.ndim; ++d) t->dl_tensor.shape[d - 1] = t->dl_tensor.shape[d];
    t->dl_tensor.ndim -= 1;
  }
  t->dl_tensor.data = (uint8_t*)t->dl_tensor.data + (size_t)batch_index * (size_t)b->batch * k.row_bytes;
  *out = t;
  return 0;
} OGB_CATCH_ALL
int ogb_batch_mark_escaped(ogb_batch* b) try {
  if (!b) return fail(OGB_ERR_INVALID, "null batch");
  b->escaped = true;
  return 0;
} OGB_CATCH_ALL
int ogb_batch_retain(ogb_batch* b) try {
  if (!b) return fail(OGB_ERR_INVALID, "null batch");
  b->refs.fetch_add(1);
  return 0;
} OGB_CATCH_ALL
int ogb_batch_release(ogb_batch* b) try {
  if (!b) return fail(OGB_ERR_INVALID, "null batch");
  batch_unref(b);
  return 0;
} OGB_CATCH_ALL

int ogb_host_alloc(size_t nbytes, void** out) try {
  if (!out) return fail(OGB_ERR_INVALID, "null out");
  OGB_CUDA(cudaHostAlloc(out, std::max<size_t>(nbytes, 1), cudaHostAllocDefault));
  return 0;
} OGB_CATCH_ALL
int ogb_host_free(void* p) try {
  if (p) OGB_CUDA(cudaFreeHost(p));
  return 0;
} OGB_CATCH_ALL

int ogb_searchsorted_warp(const int64_t* sorted_host, int64_t n, const int64_t* keys_host, int64_t m, int32_t side_right,
                          int32_t device, int64_t* out_host) try {
  if (!sorted_host || !keys_host || !out_host || n < 0 || m < 0) return fail(OGB_ERR_INVALID, "bad arguments");
  DeviceGuard device_guard(device);
  OGB_CUDA(device_guard.status);
  int64_t *d_t = nullptr, *d_k = nullptr, *d_o = nullptr;
  OGB_CUDA(cudaMalloc((void**)&d_t, std::max<int64_t>(n, 1) * 8));
  OGB_CUDA(cudaMalloc((void**)&d_k, std::max<int64_t>(m, 1) * 8));
  OGB_CUDA(cudaMalloc((void**)&d_o, std::max<int64_t>(m, 1) * 8));
  OGB_CUDA(cudaMemcpy(d_t, sorted_host, (size_t)n * 8, cudaMemcpyHostToDevice));
  OGB_CUDA(cudaMemcpy(d_k, keys_host, (size_t)m * 8, cudaMemcpyHostToDevice));
  if (m > 0) searchsorted_warp_kernel<<<(unsigned)std::min<int64_t>((m + 7) / 8, 148 * 8), 256>>>(d_t, n, d_k, m, side_right, d_o);
  OGB_CUDA(cudaGetLastError());
  OGB_CUDA(cudaMemcpy(out_host, d_o, (size_t)m * 8, cudaMemcpyDeviceToHost));
  cudaFree(d_t); cudaFree(d_k); cudaFree(d_o);
  return 0;
} OGB_CATCH_ALL

int ogb_debug_timeline(double* out_ms, int32_t capacity, int32_t* n_out) try {
  if (!out_ms || !n_out) return fail(OGB_ERR_INVALID, "null argument");
  OGB_CUDA(cudaDeviceSynchronize());
  const int n = (int)std::min<size_t>(g_timeline.size(), (size_t)std::max(capacity, 0));
  for (int i = 0; i < n; ++i) {
    float ms = 0.0f;
    OGB_CUDA(cudaEventElapsedTime(&ms, g_timeline[0], g_timeline[(size_t)i]));
    out_ms[i] = ms;
  }
  for (cudaEvent_t ev : g_timeline) cudaEventDestroy(ev);
  g_timeline.clear();
  *n_out = n;
  return 0;
} OGB_CATCH_ALL

int ogb_geometric_check(double discount, uint64_t seed, int64_t n, int32_t device, int64_t* mismatches) try {
  if (!mismatches || n < 0 || !(discount > 0.0 && discount < 1.0)) return fail(OGB_ERR_INVALID, "bad arguments");
  DeviceGuard device_guard(device);
  OGB_CUDA(device_guard.status);
  unsigned long long* d = nullptr;
  OGB_CUDA(cudaMalloc((void**)&d, 8));
  OGB_CUDA(cudaMemset(d, 0, 8));
  const double log_1mp = std::log(1.0 - (1.0 - discount));
  const ogb::RngKey key = ogb::make_rng_key(seed, 0);
  if (n > 0) geometric_check_kernel<<<148 * 8, 256>>>(key, log_1mp, (float)(1.5e-8 / std::fabs(log_1mp)), n, d);
  OGB_CUDA(cudaGetLastError());
  unsigned long long host = 0;
  OGB_CUDA(cudaMemcpy(&host, d, 8, cudaMemcpyDeviceToHost));
  cudaFree(d);
  *mismatches = (int64_t)host;
  return 0;
} OGB_CATCH_ALL

int ogb_philox_fill(uint64_t seed, uint32_t stream_id, uint64_t batch, uint32_t purpose, int64_t n, int32_t device, uint32_t* out_host) try {
  if (!out_host || n < 0) return fail(OGB_ERR_INVALID, "bad arguments");
  DeviceGuard device_guard(device);
  OGB_CUDA(device_guard.status);
  uint4* d = nullptr;
  OGB_CUDA(cudaMalloc((void**)&d, std::max<int64_t>(n, 1) * 16));
  const ogb::RngKey key = ogb::make_rng_key(seed, stream_id);
  if (n > 0) philox_fill_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 148 * 8), 256>>>(key, batch, purpose, n, d);
  OGB_CUDA(cudaGetLastError());
  OGB_CUDA(cudaMemcpy(out_host, d, (size_t)n * 16, cudaMemcpyDeviceToHost));
  cudaFree(d);
  return 0;
} OGB_CATCH_ALL

}  // extern "C"
