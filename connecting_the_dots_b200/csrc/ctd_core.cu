// Library-wide state of libctd_b200: error messages, launch accounting, options.
#include <atomic>
#include <mutex>
#include <stdarg.h>
#include <string.h>

#include "ctd_common.cuh"

namespace ctd {

int g_force_generic = 0;  // tests: route every op through its generic kernel
int g_xcorr_direct = 0;   // tests / A-B runs: XCorrVol through the direct (centred two-pass) tile kernel
int g_xcorr_hitcap = -1;  // tests: size of XCorrVol's fix-up hit list (0 forces the overflow path), -1 = automatic
int g_xcorr_nofix = 0;    // experiments: skip XCorrVol's fix-up pass (fast-path error measurements)
int g_host_graphs = 0;        // host-buffer API: 1 = capture repeated batches into CUDA graphs and replay them (measured: same step time -- the bus bounds it -- and 0.09 -> 0.01 ms of host time in the calls)
int g_host_chunks_graph = 2;  // image chunks per call in a batch that is captured (measured: finer chunks lose on the bus even with no host cost)
int g_host_chunks_batch = 2;  // ... inside ctd_host_begin_batch / end_batch, where neighbouring calls already overlap
int g_host_chunks = 4;     // host-buffer API: image chunks per call (copies below ~2 MB lose PCIe efficiency)
int g_disable_tma = 0;    // tests / A-B runs: use the shared-memory tile kernels instead of the TMA ones
static std::atomic<uint64_t> g_launches{0};

char* err_buf() {
  static thread_local char buf[512] = {0};
  return buf;
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}

void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

struct RelaxedCaptureMode {
  cudaStreamCaptureMode mode = cudaStreamCaptureModeRelaxed;
  RelaxedCaptureMode() { cudaThreadExchangeStreamCaptureMode(&mode); }
  ~RelaxedCaptureMode() { cudaThreadExchangeStreamCaptureMode(&mode); }
};

static cudaMemPool_t scratch_pool() {
  static std::mutex mtx;
  static cudaMemPool_t pools[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lk(mtx);
  if (!pools[dev]) {
    // the first use may come from inside a stream capture (global capture mode forbids allocation-like calls there):
    // create the pool in relaxed mode, the capture is not affected
    RelaxedCaptureMode relaxed;
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t p = nullptr;
    if (cudaMemPoolCreate(&p, &props) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    uint64_t keep = UINT64_MAX;
    cudaMemPoolSetAttribute(p, cudaMemPoolAttrReleaseThreshold, &keep);
    pools[dev] = p;
  }
  return pools[dev];
}

// Workspace of finish_masked_sums (ticket + block partials): static device memory, so the masked loss calls need no
// allocation, memset or free around the kernel (each of those is a graph node and ~1.5 us on a 30 us kernel).  A
// slot's ticket is zero at load time and is reset by the block that finishes the sums.  Ownership rules (a slot is
// never shared by two launches that may run concurrently):
//   * eager launches: one slot per (device, stream), found in a small table -- launches on one stream are ordered, so
//     the kernel that reuses the slot starts after its predecessor reset the ticket;
//   * launches being captured into a CUDA graph: the slot address is baked into the graph, so every captured call gets
//     a slot of its own from a separate pool that is never handed out twice (graphs may replay on any stream,
//     concurrently with each other and with eager calls);
//   * when a pool is exhausted (more than MS_EAGER streams, more than MS_GRAPH captured calls in the process), or the
//     grid has more than MS_MAXBLK blocks, the workspace comes from the stream-ordered scratch pool with a memset node
//     in front of the kernel: slower by ~1.5 us, never shared.
// A kernel that dies (trap, illegal address) leaves the context unusable anyway (sticky CUDA error), so a ticket stuck
// at a non-zero value cannot be observed by a later successful launch of the same process.
__device__ __align__(16) unsigned char g_ms_slots[MS_EAGER + MS_GRAPH][16 + MS_MAXBLK * 16];

static unsigned char* ms_base(int dev) {
  static std::mutex mtx;
  static unsigned char* bases[64] = {};
  if (dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lk(mtx);
  if (!bases[dev]) {
    RelaxedCaptureMode relaxed;  // may load the module: not a capturable operation
    void* p = nullptr;
    if (cudaGetSymbolAddress(&p, g_ms_slots) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    bases[dev] = static_cast<unsigned char*>(p);
  }
  return bases[dev];
}

int g_ms_force_scratch = 0;  // tests: always take the scratch-memory path (as if the static slots were exhausted)

bool ms_acquire(size_t nblocks, cudaStream_t st, MsSlot* s) {
  s->ticket = nullptr;
  s->partials = nullptr;
  s->scratch = nullptr;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return false;
  int slot = -1;
  if (nblocks <= MS_MAXBLK && dev < 64 && !g_ms_force_scratch) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    static std::mutex mtx;
    std::lock_guard<std::mutex> lk(mtx);
    if (cap == cudaStreamCaptureStatusActive) {
      static int next_graph[64] = {};
      if (next_graph[dev] < MS_GRAPH) slot = MS_EAGER + next_graph[dev]++;
    } else {
      static cudaStream_t owner[64][MS_EAGER];
      static int n_owner[64] = {};
      for (int i = 0; i < n_owner[dev] && slot < 0; ++i)
        if (owner[dev][i] == st) slot = i;
      if (slot < 0 && n_owner[dev] < MS_EAGER) {
        owner[dev][n_owner[dev]] = st;
        slot = n_owner[dev]++;
      }
    }
  }
  unsigned char* base = slot >= 0 ? ms_base(dev) : nullptr;
  if (base) {
    unsigned char* p = base + (size_t)slot * (16 + MS_MAXBLK * 16);
    s->ticket = reinterpret_cast<unsigned*>(p);
    s->partials = reinterpret_cast<double*>(p + 16);
    return true;
  }
  char* sc = static_cast<char*>(scratch_alloc(16 + nblocks * 16, st));
  cudaError_t e = sc ? cudaMemsetAsync(sc, 0, 16, st) : cudaErrorMemoryAllocation;
  if (e != cudaSuccess) {
    fail(CTD_ERR_NOMEM, "reduction workspace from the scratch pool: %s", cudaGetErrorString(e));
    cudaGetLastError();
    scratch_free(sc, st);
    return false;
  }
  s->scratch = sc;
  s->ticket = reinterpret_cast<unsigned*>(sc);
  s->partials = reinterpret_cast<double*>(sc + 16);
  return true;
}

void ms_release(MsSlot* s, cudaStream_t st) {
  scratch_free(s->scratch, st);  // stream-ordered: after the kernel that was just enqueued
  s->scratch = nullptr;
}

void* scratch_alloc(size_t bytes, cudaStream_t st) {
  cudaMemPool_t pool = scratch_pool();
  void* p = nullptr;
  if (!pool || cudaMallocFromPoolAsync(&p, bytes, pool, st) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}

void scratch_free(void* p, cudaStream_t st) {
  if (p) cudaFreeAsync(p, st);
}

int check_launch(const char* what) {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    cudaGetLastError();  // clear the sticky launch error so the next call starts clean
    return fail(CTD_ERR_CUDA, "%s: launch failed: %s", what, cudaGetErrorString(e));
  }
  return CTD_OK;
}

extern int g_census_sym;          // census_sym.cu
extern int g_census_sym_dbg;      // census_sym.cu
extern int g_census_sym_noguard;  // census_sym.cu
extern int g_xcorr_serial;        // xcorrvol.cu

// The names ctd_set_option accepts and the variable each one sets (meanings and defaults where they are defined).
static const struct {
  const char* name;
  int* value;
} k_options[] = {
    {"force_generic", &g_force_generic},
    {"disable_tma", &g_disable_tma},
    {"census_sym", &g_census_sym},
    {"census_sym_dbg", &g_census_sym_dbg},
    {"census_sym_noguard", &g_census_sym_noguard},
    {"xcorr_direct", &g_xcorr_direct},
    {"xcorr_serial", &g_xcorr_serial},
    {"xcorr_hitcap", &g_xcorr_hitcap},
    {"xcorr_nofix", &g_xcorr_nofix},
    {"host_graphs", &g_host_graphs},
    {"host_chunks", &g_host_chunks},
    {"host_chunks_batch", &g_host_chunks_batch},
    {"host_chunks_graph", &g_host_chunks_graph},
    {"ms_force_scratch", &g_ms_force_scratch},
};

}  // namespace ctd

CTD_API const char* ctd_last_error(void) { return ctd::err_buf(); }
CTD_API const char* ctd_version(void) { return "ctd_b200 0.1 (sm_100a)"; }
CTD_API uint64_t ctd_launch_count(void) { return ctd::g_launches.load(std::memory_order_relaxed); }

CTD_API int ctd_set_option(const char* name, int value) {
  for (const auto& o : ctd::k_options) {
    if (name && !strcmp(name, o.name)) {
      *o.value = value;
      return CTD_OK;
    }
  }
  return ctd::fail(CTD_ERR_INVALID, "ctd_set_option: unknown option '%s'", name ? name : "(null)");
}

// ---- TMA tensor-map encoder (driver entry point fetched through the runtime, no -lcuda needed)
#include "ctd_tma.cuh"
namespace ctd {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

bool make_plane_tensor_map(CUtensorMap* map, const float* base, int64_t planes, int64_t H, int64_t W, int box_w, int box_h) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn || (reinterpret_cast<uintptr_t>(base) & 15) || W % 4 || planes < 1 || H < 1 || W < 4) return false;
  if (box_w > 256 || box_h > 256 || (box_w * 4) % 16) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)planes};
  const cuuint64_t strides[2] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4};
  const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
}  // namespace ctd
