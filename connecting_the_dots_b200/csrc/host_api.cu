// Host-buffer entry points of libctd_b200 (ctd_host_*): what a CPU-side caller -- the reference's
// ext_cpu.cpp entry points (torchext/ext/ext_cpu.cpp:14-184) -- binds to.  Inputs and outputs are
// host memory (pinned memory makes the copies asynchronous DMA); each call stages through a
// per-thread, grow-only device workspace on the current device, runs the same kernels as the
// device-pointer API, copies the results back and returns once they are in host memory.  The image-wise
// ops (photometric, LCN, XCorrVol) are cut into chunks of whole images and software-pipelined over three
// private streams -- upload of chunk i+1, kernels of chunk i and download of chunk i-1 run concurrently, so
// with pinned buffers both PCIe directions stay busy and the kernels hide behind the copies.
// Between ctd_host_begin_batch() and ctd_host_end_batch() the calls only enqueue: consecutive ops then overlap as well
// (the upload of the next call runs under the download of the previous one), results are in host memory when
// ctd_host_end_batch() returns.  ctd_host_end_batch_async() leaves the batch in flight and ctd_host_wait_batch() waits for the
// oldest one: with two batches outstanding the uploads of step k + 1 run under the downloads of step k (bench step: 1.20 ->
// 0.94 ms, bus floor 0.90 ms).
// Opt-in (ctd_set_option("host_graphs", 1)): a batch that repeats -- the same calls with the same arguments and host
// buffers, which is what a training loop over fixed pinned buffers issues every step -- is captured into a CUDA graph the
// second time it is seen and replayed from the third on: its ~60 copy / launch / event calls become one cudaGraphLaunch
// (0.09 -> 0.01 ms of host time per bench step; the step itself is bound by the bus and takes the same 1.2 ms against
// a floor of 0.90 ms for its 79 MB with both directions busy: profiles/r02_e2e_chunks.json, r02_pcie_floor.json).  See submit().
// There is no CPU compute path: without a CUDA device these calls fail with CTD_ERR_CUDA.
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <atomic>
#include <functional>
#include <string>
#include <vector>

#include "ctd_common.cuh"

namespace ctd {

constexpr int CTD_RETRY_EAGER = -1000;  // internal: the call cannot be captured, issue the batch the ordinary way

static std::atomic<bool> g_process_exiting{false};
static void mark_exiting() { g_process_exiting.store(true, std::memory_order_relaxed); }
static void register_exit_hook() {
  static const int once = atexit(mark_exiting);
  (void)once;
}

struct Workspace {
  int device = -1;
  char* base = nullptr;
  size_t cap = 0;
  cudaStream_t stream = nullptr;                 // compute (and, for the unpipelined ops, copies)
  cudaStream_t s_in = nullptr, s_out = nullptr;  // upload / download streams of the chunk pipeline
  static constexpr int MAX_CHUNKS = 16;
  cudaEvent_t ev_in[MAX_CHUNKS] = {}, ev_run[MAX_CHUNKS] = {};
  bool deferred = false;  // inside ctd_host_begin_batch / ctd_host_end_batch
  size_t used = 0;        // bytes of the workspace owned by calls still in flight (deferred mode: no reuse)
  // Two batches in flight (ctd_host_end_batch_async / ctd_host_wait_batch): the uploads of step k + 1 then run under the
  // downloads of step k -- the same three streams, in issue order, nothing else is needed for the overlap.  Once a thread
  // has used the asynchronous end, its batches alternate between the two halves of the workspace.
  bool async_mode = false;
  int slot = 0;                       // half of the open (or last) batch
  size_t slot_off = 0;                // its first byte
  bool busy[2] = {false, false};      // enqueued, not waited for
  size_t lo[2] = {0, 0}, hi[2] = {0, 0};  // workspace bytes [lo, hi) a busy batch occupies
  int last_ended = 0;
  cudaEvent_t done_out[2] = {}, done_main[2] = {}, done_in[2] = {};

  int wait_slot(int s) {
    if (!busy[s]) return CTD_OK;
    busy[s] = false;
    cudaError_t e1 = cudaEventSynchronize(done_out[s]), e2 = cudaEventSynchronize(done_main[s]), e3 = cudaEventSynchronize(done_in[s]);
    const cudaError_t e = e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3);
    if (e != cudaSuccess) return fail(CTD_ERR_CUDA, "host api: waiting for a batch: %s", cudaGetErrorString(e));
    return CTD_OK;
  }
  int wait_batches() {  // both, oldest first
    const int first = last_ended ^ 1;
    const int r1 = wait_slot(first), r2 = wait_slot(first ^ 1);
    return r1 ? r1 : r2;
  }
  // Uploads of the open batch: an input (same host address, same size) that several calls of a batch read -- the
  // image pair of the sad and the census loss, the gradient weights -- crosses the bus once.  Later calls find the
  // device copy of the earlier one; their kernels are enqueued on the same compute stream after the kernel that
  // waited for that upload, so no extra dependency is needed.  Host inputs must not change while a batch is open.
  struct Upload {
    const void* host;
    size_t bytes;
    char* dev;
  };
  std::vector<Upload> uploads;
  // Downloads of the open batch that have been enqueued but not waited for: host ranges whose contents are not there
  // yet.  A later call of the batch that reads such a range (LCN's std as the mask of the loss, ProjNN's indices as
  // CrossCheck's input) must not upload it -- the host still holds the old bytes.  The newest download that overlaps
  // the range decides, since it lands last: an exact match (same address, same size: the chunks of two image-wise calls
  // line up) is served from that producer's device buffer, with no copy at all -- every kernel of a batch runs on the
  // one compute stream, after its producer.  Any other overlap waits for the downloads to land and then uploads what
  // the host really holds.  A download also retires every entry of `uploads` it overlaps (note_download): that device
  // copy no longer matches what the host will hold.
  std::vector<Upload> pending;
  uint64_t h2d_bytes = 0, h2d_saved = 0;  // statistics since ctd_host_begin_batch (ctd_host_batch_stats)

  // ---- repeated batches as CUDA graphs ------------------------------------------------------------------------------
  // Every call of an open batch has a signature (entry point + every argument, pointers by value).  A finished batch
  // leaves its signature list in a small cache.  When the first call of a later batch matches a cached list, the batch
  // is EXPECTED to repeat it:
  //   * no graph yet (seen once): the calls run under stream capture -- same code path, the three streams forked from and
  //     joined back into the compute stream -- and ctd_host_end_batch instantiates, keeps and launches the graph;
  //   * graph cached: the calls only check their signature and return; ctd_host_end_batch launches the graph.
  // A call that breaks the expectation (different signature, fewer / more calls, a host buffer that is not pinned, a
  // workspace that would have to grow, an input overlapping an output in flight) ends it: the capture is dropped, the
  // calls recorded so far are issued the ordinary way, and the batch carries on as before.  Graphs hold workspace
  // addresses: they go when the workspace is reallocated or released.  Contract as before: host inputs must not change
  // while the batch is open (a replayed batch reads them at ctd_host_end_batch), and buffers of a replayed batch must
  // still be the pinned allocations they were.
  enum Mode { EAGER, CAPTURE, REPLAY };
  struct Call {
    std::string sig;
    std::function<int()> run;
  };
  struct Cached {
    std::vector<std::string> sigs;
    cudaGraphExec_t exec = nullptr;
    bool no_graph = false;  // broke a capture once: always issued the ordinary way
    uint64_t h2d = 0, saved = 0, stamp = 0;
  };
  static constexpr int MAX_CACHED = 16;
  Mode mode = EAGER;
  bool capturing = false;
  int cand = -1;
  uint64_t clock = 0;
  uint64_t n_captured = 0, n_replayed = 0, n_bailed = 0;  // ctd_host_graph_stats
  std::vector<Call> calls;
  std::vector<Cached> cache;

  void drop_graphs() {
    for (Cached& c : cache)
      if (c.exec) cudaGraphExecDestroy(c.exec);
    cache.clear();
    cand = -1;
  }
  int begin_capture() {
    CTD_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    capturing = true;
    CTD_CUDA(cudaEventRecord(ev_in[0], stream));  // fork: the copy streams join the capture
    CTD_CUDA(cudaStreamWaitEvent(s_in, ev_in[0], 0));
    CTD_CUDA(cudaStreamWaitEvent(s_out, ev_in[0], 0));
    return CTD_OK;
  }
  // join the copy streams and end the capture; *graph = nullptr when the capture was invalidated
  int end_capture(cudaGraph_t* graph) {
    *graph = nullptr;
    capturing = false;
    cudaEventRecord(ev_in[0], s_in);
    cudaStreamWaitEvent(stream, ev_in[0], 0);
    cudaEventRecord(ev_run[0], s_out);
    cudaStreamWaitEvent(stream, ev_run[0], 0);
    if (cudaStreamEndCapture(stream, graph) != cudaSuccess) {
      cudaGetLastError();
      *graph = nullptr;
    }
    return CTD_OK;
  }
  // the expectation failed: issue what has been recorded the ordinary way and carry on in EAGER mode
  int bail(bool never_again) {
    ++n_bailed;
    if (capturing) {
      cudaGraph_t g = nullptr;
      end_capture(&g);
      if (g) cudaGraphDestroy(g);
    }
    if (never_again && cand >= 0 && cand < (int)cache.size()) cache[cand].no_graph = true;
    mode = EAGER;
    cand = -1;
    used = 0;
    uploads.clear();
    pending.clear();
    h2d_bytes = h2d_saved = 0;
    for (Call& c : calls) {
      if (int rc = c.run()) return rc;
      c.run = nullptr;
    }
    return CTD_OK;
  }
  static bool pinned(const std::vector<const void*>& ptrs) {
    for (const void* p : ptrs) {
      if (!p) continue;
      cudaPointerAttributes a;
      if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
      }
      if (a.type != cudaMemoryTypeHost) return false;
    }
    return true;
  }
  int submit(std::string sig, const std::vector<const void*>& host_ptrs, std::function<int()> run);
  int end_batch(bool wait);

  static bool overlaps(const Upload& u, const void* host, size_t bytes) {
    const char *h0 = static_cast<const char*>(host), *p0 = static_cast<const char*>(u.host);
    return h0 < p0 + u.bytes && p0 < h0 + bytes;
  }
  void note_download(const void* host, size_t bytes, char* dev) {
    if (!deferred || !bytes) return;
    uploads.erase(std::remove_if(uploads.begin(), uploads.end(), [&](const Upload& u) { return overlaps(u, host, bytes); }),
                  uploads.end());
    pending.push_back({host, bytes, dev});
  }

  // device address holding `bytes` bytes of `host`: the earlier upload of this batch, or `dst` after enqueuing the copy
  int upload(cudaStream_t st, char* dst, const void* host, size_t bytes, char** dev) {
    *dev = dst;
    if (bytes == 0) return CTD_OK;
    if (deferred) {
      for (auto p = pending.rbegin(); p != pending.rend(); ++p) {
        if (!overlaps(*p, host, bytes)) continue;
        if (p->host == host && p->bytes == bytes) {
          *dev = p->dev;
          h2d_saved += bytes;
          return CTD_OK;
        }
        // partial overlap with an output in flight: let the downloads finish, then the host copy is current
        if (capturing) return CTD_RETRY_EAGER;
        CTD_CUDA(cudaStreamSynchronize(s_out));
        CTD_CUDA(cudaStreamSynchronize(stream));
        pending.clear();
        break;
      }
      for (const Upload& u : uploads)
        if (u.host == host && u.bytes == bytes) {
          *dev = u.dev;
          h2d_saved += bytes;
          return CTD_OK;
        }
      uploads.push_back({host, bytes, dst});
    }
    h2d_bytes += bytes;
    CTD_CUDA(cudaMemcpyAsync(dst, host, bytes, cudaMemcpyHostToDevice, st));
    return CTD_OK;
  }

  // workspace of one call: `bytes` fresh bytes behind everything still in flight
  int carve(size_t bytes, char** out) {
    const size_t need = (used + bytes + 255) & ~size_t(255);
    if (int rc = ensure(async_mode ? 2 * need : need)) return rc;  // a reallocation waits for everything and resets `used`
    slot_off = async_mode && slot ? (cap / 2) & ~size_t(255) : 0;
    *out = base + slot_off + used;
    return CTD_OK;
  }
  // end of a call: wait for the results unless a batch is open
  int finish(size_t bytes) {
    if (deferred) {
      used += bytes;
      return CTD_OK;
    }
    CTD_CUDA(cudaStreamSynchronize(s_out));
    CTD_CUDA(cudaStreamSynchronize(stream));
    return CTD_OK;
  }

  int ensure(size_t bytes) {
    int dev = 0;
    CTD_CUDA(cudaGetDevice(&dev));
    if (dev != device) {
      release();
      device = dev;
    }
    if (!stream) {
      if (capturing) return CTD_RETRY_EAGER;
      register_exit_hook();
      CTD_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
      CTD_CUDA(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
      CTD_CUDA(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
      for (int i = 0; i < MAX_CHUNKS; ++i) {
        CTD_CUDA(cudaEventCreateWithFlags(&ev_in[i], cudaEventDisableTiming));
        CTD_CUDA(cudaEventCreateWithFlags(&ev_run[i], cudaEventDisableTiming));
      }
      for (int i = 0; i < 2; ++i) {
        CTD_CUDA(cudaEventCreateWithFlags(&done_out[i], cudaEventDisableTiming));
        CTD_CUDA(cudaEventCreateWithFlags(&done_main[i], cudaEventDisableTiming));
        CTD_CUDA(cudaEventCreateWithFlags(&done_in[i], cudaEventDisableTiming));
      }
    }
    if (bytes > cap) {
      if (capturing) return CTD_RETRY_EAGER;  // cudaMalloc / cudaDeviceSynchronize cannot be captured
      drop_graphs();                          // they hold addresses of the old workspace
      if (base) {
        CTD_CUDA(cudaDeviceSynchronize());  // also completes every call and batch still in flight: their results are out
        busy[0] = busy[1] = false;
        cudaFree(base);
        base = nullptr;
        cap = 0;
        used = 0;
        uploads.clear();  // the device copies of this batch's earlier uploads went with the old workspace
        pending.clear();  // ... and every download has landed
      }
      const size_t want = bytes + bytes / 8 + (1 << 20);
      if (cudaMalloc(&base, want) != cudaSuccess) {
        cudaGetLastError();
        return fail(CTD_ERR_NOMEM, "host api: cannot allocate %zu bytes of device workspace", want);
      }
      cap = want;
    }
    return CTD_OK;
  }
  void release() {
    drop_graphs();
    if (stream) {
      cudaStreamSynchronize(stream);
      cudaStreamSynchronize(s_in);
      cudaStreamSynchronize(s_out);
      cudaStreamDestroy(stream);
      cudaStreamDestroy(s_in);
      cudaStreamDestroy(s_out);
      for (int i = 0; i < MAX_CHUNKS; ++i) {
        cudaEventDestroy(ev_in[i]);
        cudaEventDestroy(ev_run[i]);
      }
      for (int i = 0; i < 2; ++i) {
        cudaEventDestroy(done_out[i]);
        cudaEventDestroy(done_main[i]);
        cudaEventDestroy(done_in[i]);
      }
      busy[0] = busy[1] = false;
      async_mode = false;
      slot = 0;
      s_in = s_out = nullptr;
    }
    if (base) cudaFree(base);
    base = nullptr;
    cap = 0;
    stream = nullptr;
    device = -1;
  }
  // A host thread that ends gives its device workspace, streams and events back.  At process exit the destructors of
  // the exiting thread's thread_local objects run before any atexit handler or static destructor (so the CUDA runtime
  // is still up); g_process_exiting covers destructors that run later than that.
  ~Workspace() {
    if (g_process_exiting.load(std::memory_order_relaxed) || device < 0) return;
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess) {
      cudaGetLastError();
      return;
    }
    if (cudaSetDevice(device) == cudaSuccess) release();
    cudaSetDevice(cur);
    cudaGetLastError();
  }
};

static thread_local Workspace g_ws;

extern int g_host_graphs;  // ctd_set_option("host_graphs", 0): never capture / replay batches

// Signature of one call: entry point + arguments (pointers by value); the host pointers are also kept for the
// pinned-memory check in front of a capture.
struct Sig {
  std::string bytes;
  std::vector<const void*> host;
  explicit Sig(int op) { put(op); }
  template <typename T>
  Sig& put(T v) {
    bytes.append(reinterpret_cast<const char*>(&v), sizeof(T));
    return *this;
  }
  Sig& ptr(const void* p) {
    host.push_back(p);
    return put(p);
  }
};

int Workspace::submit(std::string sig, const std::vector<const void*>& host_ptrs, std::function<int()> run) {
  if (!deferred && (busy[0] || busy[1]))  // a synchronous call takes the workspace from its start: nothing may be in flight there
    if (int rc = wait_batches()) return rc;
  if (!deferred || !g_host_graphs) return run();
  sig.push_back((char)(slot + (async_mode ? 2 : 0)));  // a graph holds the addresses of the workspace half it was captured in
  const size_t i = calls.size();
  if (i == 0) {  // which cached batch does this one start like?
    cand = -1;
    for (int k = 0; k < (int)cache.size(); ++k)
      if (!cache[k].sigs.empty() && cache[k].sigs[0] == sig && (cand < 0 || cache[k].stamp > cache[cand].stamp)) cand = k;
    mode = EAGER;
    if (cand >= 0 && !cache[cand].no_graph && stream) {
      if (cache[cand].exec) {
        mode = REPLAY;
      } else {
        if (int rc = begin_capture()) {
          capturing = false;
          return rc;
        }
        mode = CAPTURE;
      }
    }
  }
  if (mode != EAGER) {
    bool ok = i < cache[cand].sigs.size() && cache[cand].sigs[i] == sig;
    bool never_again = false;
    if (!ok) {  // another cached batch that begins with the same calls (two kinds of step sharing their first calls)?
      int alt = -1;
      for (int k = 0; k < (int)cache.size(); ++k) {
        const Cached& a = cache[k];
        if (k == cand || a.no_graph || a.sigs.size() <= i || a.sigs[i] != sig) continue;
        bool same = true;
        for (size_t q = 0; q < i && same; ++q) same = a.sigs[q] == calls[q].sig;
        if (same && (alt < 0 || (a.exec != nullptr) > (cache[alt].exec != nullptr) ||
                     ((a.exec != nullptr) == (cache[alt].exec != nullptr) && a.stamp > cache[alt].stamp)))
          alt = k;
      }
      if (alt >= 0) {
        if (cache[alt].exec) {  // nothing of this batch has been issued yet (replay) or only into a capture (dropped)
          if (capturing) {
            cudaGraph_t g = nullptr;
            end_capture(&g);
            if (g) cudaGraphDestroy(g);
          }
          mode = REPLAY;
        } else if (mode == REPLAY) {  // capture this kind of batch instead: its first calls go into the capture now
          used = 0;
          uploads.clear();
          pending.clear();
          h2d_bytes = h2d_saved = 0;
          if (int rc = begin_capture()) {
            capturing = false;
            return rc;
          }
          mode = CAPTURE;
          for (size_t q = 0; q < i; ++q)
            if (int rc = calls[q].run()) {
              cand = alt;
              if (rc != CTD_RETRY_EAGER) {
                bail(true);
                return rc;
              }
              if (int rb = bail(true)) return rb;
              calls.push_back({std::move(sig), nullptr});
              return run();
            }
        }  // else: already capturing, and the captured prefix is this batch's too
        cand = alt;
        ok = true;
      }
    }
    if (ok && mode == CAPTURE && !pinned(host_ptrs)) {
      ok = false;
      never_again = true;  // pageable buffers: copies are staged by the driver, nothing to gain and not capturable
    }
    if (ok) {
      calls.push_back({sig, run});
      if (mode == REPLAY) return CTD_OK;
      const int rc = run();  // under capture
      if (rc == CTD_OK) return rc;
      calls.pop_back();
      if (rc != CTD_RETRY_EAGER) {  // a real error: the batch is over for the graph, the caller sees the status
        bail(true);
        return rc;
      }
      never_again = true;
    }
    if (int rc = bail(never_again)) return rc;
  }
  calls.push_back({std::move(sig), nullptr});
  return run();
}

int Workspace::end_batch(bool wait) {
  int rc = CTD_OK;
  bool launched = false;
  static const bool dbg = getenv("CTD_HOST_DEBUG") != nullptr;
  if (dbg) fprintf(stderr, "ctd_host_end_batch: %zu calls, mode %s, candidate %d of %zu cached\n", calls.size(),
                   mode == EAGER ? "eager" : (mode == CAPTURE ? "capture" : "replay"), cand, cache.size());
  if (mode != EAGER && calls.size() != cache[cand].sigs.size()) rc = bail(false);  // fewer calls than expected
  if (rc == CTD_OK && mode == CAPTURE) {
    cudaGraph_t g = nullptr;
    end_capture(&g);
    Cached& c = cache[cand];
    if (g && cudaGraphInstantiate(&c.exec, g, 0) == cudaSuccess) {
      c.h2d = h2d_bytes;
      c.saved = h2d_saved;
      mode = REPLAY;
      ++n_captured;
    } else {
      cudaGetLastError();
      c.exec = nullptr;
      rc = bail(true);
    }
    if (g) cudaGraphDestroy(g);
  }
  if (rc == CTD_OK && mode == REPLAY) {
    Cached& c = cache[cand];
    h2d_bytes = c.h2d;
    h2d_saved = c.saved;
    c.stamp = ++clock;
    cudaError_t e = cudaGraphLaunch(c.exec, stream);
    if (e != cudaSuccess) rc = fail(CTD_ERR_CUDA, "ctd_host_end_batch: graph launch: %s", cudaGetErrorString(e));
    launched = true;
    ++n_replayed;
  }
  if (rc == CTD_OK && !launched && g_host_graphs && !calls.empty()) {  // an ordinary batch: remember what it looked like
    int slot = -1;
    for (int k = 0; k < (int)cache.size() && slot < 0; ++k) {
      if (cache[k].sigs.size() != calls.size()) continue;
      bool same = true;
      for (size_t j = 0; j < calls.size() && same; ++j) same = cache[k].sigs[j] == calls[j].sig;
      if (same) slot = k;
    }
    if (slot < 0) {
      if ((int)cache.size() < MAX_CACHED) {
        cache.emplace_back();
        slot = (int)cache.size() - 1;
      } else {
        slot = 0;
        for (int k = 1; k < (int)cache.size(); ++k)
          if (cache[k].stamp < cache[slot].stamp) slot = k;
        if (cache[slot].exec) cudaGraphExecDestroy(cache[slot].exec);
        cache[slot] = Cached();
      }
      for (const Call& c : calls) cache[slot].sigs.push_back(c.sig);
    }
    cache[slot].stamp = ++clock;
  }
  deferred = false;
  if (stream && !wait && rc == CTD_OK) {  // leave it in flight: three events mark its end on the three streams
    async_mode = true;
    lo[slot] = slot_off;
    hi[slot] = slot_off + used;
    cudaError_t e1 = cudaEventRecord(done_out[slot], s_out), e2 = cudaEventRecord(done_main[slot], stream),
                e3 = cudaEventRecord(done_in[slot], s_in);
    const cudaError_t e = e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3);
    if (e != cudaSuccess) rc = fail(CTD_ERR_CUDA, "ctd_host_end_batch_async: %s", cudaGetErrorString(e));
    busy[slot] = rc == CTD_OK;
    last_ended = slot;
  }
  used = 0;
  uploads.clear();
  pending.clear();
  calls.clear();
  mode = EAGER;
  cand = -1;
  if (stream && (wait || rc != CTD_OK)) {  // the streams drain in order: this also completes an earlier batch still in flight
    cudaError_t e1 = cudaStreamSynchronize(s_out), e2 = cudaStreamSynchronize(stream), e3 = cudaStreamSynchronize(s_in);
    const cudaError_t e = e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3);
    if (e != cudaSuccess && rc == CTD_OK) rc = fail(CTD_ERR_CUDA, "ctd_host_end_batch: %s", cudaGetErrorString(e));
    busy[0] = busy[1] = false;
  }
  return rc;
}

// carve 256-byte aligned sub-buffers out of the workspace
struct Carver {
  std::vector<size_t> sizes;
  size_t total = 0;
  size_t add(size_t bytes) {
    const size_t off = total;
    total += (bytes + 255) & ~size_t(255);
    return off;
  }
};

// images [i0, i1) of chunk c when B images are cut into n chunks
static inline int64_t chunk_lo(int64_t B, int n, int c) { return B * c / n; }
extern int g_host_chunks_batch;
extern int g_host_chunks;  // ctd_set_option("host_chunks", n): upper bound on the pipeline depth (A/B runs)
extern int g_host_chunks_graph;
static inline int chunk_count(int64_t B, bool deferred) {
  // inside a batch the neighbouring calls already overlap with this one: fewer, larger copies win (measured: every
  // chunk is ~10 driver calls); in a batch that is being captured into a graph the calls cost nothing at replay
  const int want = g_ws.capturing ? g_host_chunks_graph : (deferred ? std::min(g_host_chunks, g_host_chunks_batch) : g_host_chunks);
  return (int)std::min<int64_t>(std::max<int64_t>(B, 1), std::min(std::max(want, 1), (int)Workspace::MAX_CHUNKS));
}

}  // namespace ctd

using namespace ctd;

// upload on the compute stream (the unpipelined ops); `devp` receives where the bytes are (an earlier copy of the batch or dst)
#define H2D(devp, dst, src, bytes) RUN(g_ws.upload(g_ws.stream, (dst), (src), (bytes), &(devp)))
#define D2H(dst, src, bytes) D2H_ON(g_ws.stream, dst, src, bytes)
#define D2H_ON(st, dst, src, bytes)                                                        \
  do {                                                                                     \
    CTD_CUDA(cudaMemcpyAsync((dst), (src), (bytes), cudaMemcpyDeviceToHost, (st)));        \
    g_ws.note_download((dst), (bytes), (char*)(src));                                      \
  } while (0)
#define RUN(call)                    \
  do {                               \
    if (int rc__ = (call)) return rc__; \
  } while (0)

static int photometric_host(const float* es, const float* ta, const float* go, float* out, float* gi, int64_t B,
                            int64_t C, int64_t H, int64_t W, int bs, int type, float eps) {
  CTD_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0, "photometric: negative size");
  const size_t nin = (size_t)(B * C * H * W) * sizeof(float), nout = (size_t)(B * H * W) * sizeof(float);
  Carver cv;
  const size_t o_es = cv.add(nin), o_ta = cv.add(nin), o_go = cv.add(go ? nout : 0), o_out = cv.add(out ? nout : 0),
               o_gi = cv.add(gi ? nin : 0);
  char* b = nullptr;
  RUN(g_ws.carve(cv.total, &b));
  if (nin) CTD_REQUIRE(es && ta, "photometric: null pointer");
  if (gi) CTD_REQUIRE(go || !nout, "photometric_bwd: null grad_out");
  if (B == 0) return CTD_OK;
  const int nch = chunk_count(B, g_ws.deferred);
  const size_t in_img = nin / B, out_img = nout / B;  // bytes per image
  for (int c = 0; c < nch; ++c) {
    const int64_t i0 = chunk_lo(B, nch, c), nb = chunk_lo(B, nch, c + 1) - i0;
    const size_t oi = (size_t)i0 * in_img, oo = (size_t)i0 * out_img;
    char *d_es = nullptr, *d_ta = nullptr, *d_go = nullptr;
    RUN(g_ws.upload(g_ws.s_in, b + o_es + oi, (const char*)es + oi, nb * in_img, &d_es));
    RUN(g_ws.upload(g_ws.s_in, b + o_ta + oi, (const char*)ta + oi, nb * in_img, &d_ta));
    RUN(g_ws.upload(g_ws.s_in, b + o_go + oo, (const char*)go + oo, gi ? nb * out_img : 0, &d_go));
    CTD_CUDA(cudaEventRecord(g_ws.ev_in[c], g_ws.s_in));
    CTD_CUDA(cudaStreamWaitEvent(g_ws.stream, g_ws.ev_in[c], 0));
    if (out && gi)
      RUN(ctd_photometric_fwd_bwd_f32((float*)d_es, (float*)d_ta, (float*)d_go, (float*)(b + o_out + oo), (float*)(b + o_gi + oi),
                                      nb, C, H, W, bs, type, eps, g_ws.stream));
    else if (out)
      RUN(ctd_photometric_fwd_f32((float*)d_es, (float*)d_ta, (float*)(b + o_out + oo), nb, C, H, W, bs, type, eps, g_ws.stream));
    else if (gi)
      RUN(ctd_photometric_bwd_f32((float*)d_es, (float*)d_ta, (float*)d_go, (float*)(b + o_gi + oi), nb, C, H, W, bs, type, eps,
                                  g_ws.stream));
    CTD_CUDA(cudaEventRecord(g_ws.ev_run[c], g_ws.stream));
    CTD_CUDA(cudaStreamWaitEvent(g_ws.s_out, g_ws.ev_run[c], 0));
    if (out && out_img) D2H_ON(g_ws.s_out, (char*)out + oo, b + o_out + oo, nb * out_img);
    if (gi && in_img) D2H_ON(g_ws.s_out, (char*)gi + oi, b + o_gi + oi, nb * in_img);
  }
  return g_ws.finish(cv.total);
}

CTD_API int ctd_host_photometric_fwd_f32(const float* es, const float* ta, float* out, int64_t B, int64_t C,
                                            int64_t H, int64_t W, int bs, int type, float eps) {
  CTD_REQUIRE(out || B * H * W == 0, "photometric_fwd: null output");
  Sig sg(1);
  sg.ptr(es).ptr(ta).ptr(out).put(B).put(C).put(H).put(W).put(bs).put(type).put(eps);
  return g_ws.submit(sg.bytes, sg.host, [=]() { return photometric_host(es, ta, nullptr, out, nullptr, B, C, H, W, bs, type, eps); });
}
CTD_API int ctd_host_photometric_bwd_f32(const float* es, const float* ta, const float* go, float* gi, int64_t B,
                                            int64_t C, int64_t H, int64_t W, int bs, int type, float eps) {
  CTD_REQUIRE(gi || B * C * H * W == 0, "photometric_bwd: null output");
  Sig sg(2);
  sg.ptr(es).ptr(ta).ptr(go).ptr(gi).put(B).put(C).put(H).put(W).put(bs).put(type).put(eps);
  return g_ws.submit(sg.bytes, sg.host, [=]() { return photometric_host(es, ta, go, nullptr, gi, B, C, H, W, bs, type, eps); });
}
CTD_API int ctd_host_photometric_fwd_bwd_f32(const float* es, const float* ta, const float* go, float* out,
                                                float* gi, int64_t B, int64_t C, int64_t H, int64_t W, int bs,
                                                int type, float eps) {
  CTD_REQUIRE((out && gi) || B * C * H * W == 0, "photometric_fwd_bwd: null output");
  Sig sg(3);
  sg.ptr(es).ptr(ta).ptr(go).ptr(out).ptr(gi).put(B).put(C).put(H).put(W).put(bs).put(type).put(eps);
  return g_ws.submit(sg.bytes, sg.host, [=]() { return photometric_host(es, ta, go, out, gi, B, C, H, W, bs, type, eps); });
}

// The reference caller's whole use of the loss (model/networks.py:376-377): loss map, d loss / d es for
// grad_out (= mask / sum(mask) up to a scalar, supplied by the caller) and the two masked-mean terms
// sums2 = (sum(mask * loss), sum(mask)) -- `out` may be NULL when the caller only wants the scalars and the gradient
// (the loss map then never crosses the bus: 4 bytes per pixel less to download).  Chunks produce their own partial
// sums on the device; one small kernel adds them in chunk order before the 8-byte download.
namespace ctd {
__global__ void add_pairs_kernel(const float* __restrict__ parts, int n, float* __restrict__ out2) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < n; ++i) {
      a += (double)parts[2 * i];
      b += (double)parts[2 * i + 1];
    }
    out2[0] = (float)a;
    out2[1] = (float)b;
  }
}
}  // namespace ctd

static int photometric_masked_host(const float* es, const float* ta, const float* go, const float* mask, float* out, float* gi,
                                   float* sums2, int64_t B, int64_t C, int64_t H, int64_t W, int bs, int type, float eps) {
  const size_t nin = (size_t)(B * C * H * W) * sizeof(float), nout = (size_t)(B * H * W) * sizeof(float);
  const int nch = chunk_count(B, g_ws.deferred);
  Carver cv;
  const size_t o_es = cv.add(nin), o_ta = cv.add(nin), o_go = cv.add(nout), o_mk = cv.add(nout), o_out = cv.add(nout),
               o_gi = cv.add(nin), o_parts = cv.add(sizeof(float) * 2 * (Workspace::MAX_CHUNKS + 1));
  char* b = nullptr;
  RUN(g_ws.carve(cv.total, &b));
  const size_t in_img = nin / B, out_img = nout / B;
  float* parts = reinterpret_cast<float*>(b + o_parts);
  for (int c = 0; c < nch; ++c) {
    const int64_t i0 = chunk_lo(B, nch, c), nb = chunk_lo(B, nch, c + 1) - i0;
    const size_t oi = (size_t)i0 * in_img, oo = (size_t)i0 * out_img;
    char *d_es = nullptr, *d_ta = nullptr, *d_go = nullptr, *d_mk = nullptr;
    RUN(g_ws.upload(g_ws.s_in, b + o_es + oi, (const char*)es + oi, nb * in_img, &d_es));
    RUN(g_ws.upload(g_ws.s_in, b + o_ta + oi, (const char*)ta + oi, nb * in_img, &d_ta));
    RUN(g_ws.upload(g_ws.s_in, b + o_go + oo, (const char*)go + oo, nb * out_img, &d_go));
    RUN(g_ws.upload(g_ws.s_in, b + o_mk + oo, (const char*)mask + oo, nb * out_img, &d_mk));
    CTD_CUDA(cudaEventRecord(g_ws.ev_in[c], g_ws.s_in));
    CTD_CUDA(cudaStreamWaitEvent(g_ws.stream, g_ws.ev_in[c], 0));
    RUN(ctd_photometric_fwd_bwd_masked_f32((float*)d_es, (float*)d_ta, (float*)d_go, (float*)d_mk, (float*)(b + o_out + oo),
                                           (float*)(b + o_gi + oi), parts + 2 * c, nb, C, H, W, bs, type, eps, g_ws.stream));
    if (c == nch - 1) {
      add_pairs_kernel<<<1, 32, 0, g_ws.stream>>>(parts, nch, parts + 2 * Workspace::MAX_CHUNKS);
      count_launch();
    }
    CTD_CUDA(cudaEventRecord(g_ws.ev_run[c], g_ws.stream));
    CTD_CUDA(cudaStreamWaitEvent(g_ws.s_out, g_ws.ev_run[c], 0));
    if (out) D2H_ON(g_ws.s_out, (char*)out + oo, b + o_out + oo, nb * out_img);
    D2H_ON(g_ws.s_out, (char*)gi + oi, b + o_gi + oi, nb * in_img);
    if (c == nch - 1) CTD_CUDA(cudaMemcpyAsync(sums2, parts + 2 * Workspace::MAX_CHUNKS, 2 * sizeof(float), cudaMemcpyDeviceToHost, g_ws.s_out));
  }
  return g_ws.finish(cv.total);
}

CTD_API int ctd_host_photometric_fwd_bwd_masked_f32(const float* es, const float* ta, const float* go, const float* mask,
                                                       float* out, float* gi, float* sums2, int64_t B, int64_t C, int64_t H,
                                                       int64_t W, int bs, int type, float eps) {
  CTD_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0, "photometric: negative size");
  CTD_REQUIRE(sums2, "photometric_fwd_bwd_masked: null sums2");
  if (B * H * W == 0) {  // host-side result, nothing to enqueue (and nothing for a replayed batch to miss)
    sums2[0] = sums2[1] = 0.f;
    return CTD_OK;
  }
  CTD_REQUIRE(es && ta && go && mask && gi, "photometric_fwd_bwd_masked: null pointer");
  Sig sg(4);
  sg.ptr(es).ptr(ta).ptr(go).ptr(mask).ptr(out).ptr(gi).ptr(sums2).put(B).put(C).put(H).put(W).put(bs).put(type).put(eps);
  return g_ws.submit(sg.bytes, sg.host,
                     [=]() { return photometric_masked_host(es, ta, go, mask, out, gi, sums2, B, C, H, W, bs, type, eps); });
}

static int xcorrvol_host(const float* in0, const float* in1, float* out, int64_t B, int64_t C, int64_t H, int64_t W, int64_t D,
                         int bs) {
  CTD_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0 && D >= 0, "xcorrvol: negative size");
  const size_t nin = (size_t)(B * C * H * W) * sizeof(float), nout = (size_t)(B * D * H * W) * sizeof(float);
  Carver cv;
  const size_t o0 = cv.add(nin), o1 = cv.add(nin), oo = cv.add(nout);
  char* b = nullptr;
  RUN(g_ws.carve(cv.total, &b));
  if (nin) CTD_REQUIRE(in0 && in1, "xcorrvol: null pointer");
  if (nout) CTD_REQUIRE(out, "xcorrvol: null output");
  if (B == 0) return CTD_OK;
  const int nch = chunk_count(B, g_ws.deferred);
  const size_t in_img = nin / B, out_img = nout / B;
  for (int c = 0; c < nch; ++c) {
    const int64_t i0 = chunk_lo(B, nch, c), nb = chunk_lo(B, nch, c + 1) - i0;
    const size_t oi = (size_t)i0 * in_img, ov = (size_t)i0 * out_img;
    char *d0 = nullptr, *d1 = nullptr;
    RUN(g_ws.upload(g_ws.s_in, b + o0 + oi, (const char*)in0 + oi, nb * in_img, &d0));
    RUN(g_ws.upload(g_ws.s_in, b + o1 + oi, (const char*)in1 + oi, nb * in_img, &d1));
    CTD_CUDA(cudaEventRecord(g_ws.ev_in[c], g_ws.s_in));
    CTD_CUDA(cudaStreamWaitEvent(g_ws.stream, g_ws.ev_in[c], 0));
    RUN(ctd_xcorrvol_f32((float*)d0, (float*)d1, (float*)(b + oo + ov), nb, C, H, W, D, bs, g_ws.stream));
    CTD_CUDA(cudaEventRecord(g_ws.ev_run[c], g_ws.stream));
    CTD_CUDA(cudaStreamWaitEvent(g_ws.s_out, g_ws.ev_run[c], 0));
    if (out_img) D2H_ON(g_ws.s_out, (char*)out + ov, b + oo + ov, nb * out_img);
  }
  return g_ws.finish(cv.total);
}

CTD_API int ctd_host_xcorrvol_f32(const float* in0, const float* in1, float* out, int64_t B, int64_t C, int64_t H,
                                     int64_t W, int64_t D, int bs) {
  Sig sg(5);
  sg.ptr(in0).ptr(in1).ptr(out).put(B).put(C).put(H).put(W).put(D).put(bs);
  return g_ws.submit(sg.bytes, sg.host, [=]() { return xcorrvol_host(in0, in1, out, B, C, H, W, D, bs); });
}

static int proj_nn_host(const float* xyz0, const float* xyz1, const float* K, int64_t* out, int64_t B, int64_t H, int64_t W,
                        int ps) {
  CTD_REQUIRE(B >= 0 && H >= 0 && W >= 0, "proj_nn: negative size");
  const size_t npt = (size_t)(B * H * W) * 3 * sizeof(float), nout = (size_t)(B * H * W) * sizeof(int64_t);
  Carver cv;
  const size_t o0 = cv.add(npt), o1 = cv.add(npt), ok = cv.add(9 * sizeof(float)), oo = cv.add(nout);
  char* b = nullptr;
  RUN(g_ws.carve(cv.total, &b));
  char *d0 = b + o0, *d1 = b + o1, *dk = b + ok;
  if (nout) {
    CTD_REQUIRE(xyz0 && xyz1 && K && out, "proj_nn: null pointer");
    H2D(d0, b + o0, xyz0, npt);
    H2D(d1, b + o1, xyz1, npt);
    H2D(dk, b + ok, K, 9 * sizeof(float));
  }
  RUN(ctd_proj_nn_f32((float*)d0, (float*)d1, (float*)dk, (int64_t*)(b + oo), B, H, W, ps, g_ws.stream));
  if (nout) D2H(out, b + oo, nout);
  return g_ws.finish(cv.total);
}

CTD_API int ctd_host_proj_nn_f32(const float* xyz0, const float* xyz1, const float* K, int64_t* out, int64_t B,
                                    int64_t H, int64_t W, int ps) {
  Sig sg(6);
  sg.ptr(xyz0).ptr(xyz1).ptr(K).ptr(out).put(B).put(H).put(W).put(ps);
  return g_ws.submit(sg.bytes, sg.host, [=]() { return proj_nn_host(xyz0, xyz1, K, out, B, H, W, ps); });
}

static int nn_host(const float* in0, const float* in1, int64_t* out, int64_t N0, int64_t N1) {
  CTD_REQUIRE(N0 >= 0 && N1 >= 0, "nn: negative size");
  const size_t n0 = (size_t)N0 * 3 * sizeof(float), n1 = (size_t)N1 * 3 * sizeof(float), no = (size_t)N0 * sizeof(int64_t);
  Carver cv;
  const size_t o0 = cv.add(n0), o1 = cv.add(n1), oo = cv.add(no);
  char* b = nullptr;
  RUN(g_ws.carve(cv.total, &b));
  char *d0 = b + o0, *d1 = b + o1;
  if (n0) {
    CTD_REQUIRE(in0 && out, "nn: null pointer");
    H2D(d0, b + o0, in0, n0);
  }
  if (n1) {
    CTD_REQUIRE(in1, "nn: null pointer");
    H2D(d1, b + o1, in1, n1);
  }
  RUN(ctd_nn_f32((float*)d0, (float*)d1, (int64_t*)(b + oo), N0, N1, g_ws.stream));
  if (no) D2H(out, b + oo, no);
  return g_ws.finish(cv.total);
}

CTD_API int ctd_host_nn_f32(const float* in0, const float* in1, int64_t* out, int64_t N0, int64_t N1) {
  Sig sg(7);
  sg.ptr(in0).ptr(in1).ptr(out).put(N0).put(N1);
  return g_ws.submit(sg.bytes, sg.host, [=]() { return nn_host(in0, in1, out, N0, N1); });
}

static int crosscheck_host(const int64_t* in0, const int64_t* in1, uint8_t* out, int64_t N0, int64_t N1) {
  CTD_REQUIRE(N0 >= 0 && N1 >= 0, "crosscheck: negative size");
  const size_t n0 = (size_t)N0 * sizeof(int64_t), n1 = (size_t)N1 * sizeof(int64_t), no = (size_t)N0;
  Carver cv;
  const size_t o0 = cv.add(n0), o1 = cv.add(n1), oo = cv.add(no);
  char* b = nullptr;
  RUN(g_ws.carve(cv.total, &b));
  char *d0 = b + o0, *d1 = b + o1;
  if (n0) {
    CTD_REQUIRE(in0 && out, "crosscheck: null pointer");
    H2D(d0, b + o0, in0, n0);
  }
  if (n1) {
    CTD_REQUIRE(in1, "crosscheck: null pointer");
    H2D(d1, b + o1, in1, n1);
  }
  RUN(ctd_crosscheck((int64_t*)d0, (int64_t*)d1, (uint8_t*)(b + oo), N0, N1, g_ws.stream));
  if (no) D2H(out, b + oo, no);
  return g_ws.finish(cv.total);
}

CTD_API int ctd_host_crosscheck(const int64_t* in0, const int64_t* in1, uint8_t* out, int64_t N0, int64_t N1) {
  Sig sg(8);
  sg.ptr(in0).ptr(in1).ptr(out).put(N0).put(N1);
  return g_ws.submit(sg.bytes, sg.host, [=]() { return crosscheck_host(in0, in1, out, N0, N1); });
}

static int lcn_host(const float* x, float* lcn, float* sd, int64_t N, int64_t H, int64_t W, int r, float eps) {
  CTD_REQUIRE(N >= 0 && H >= 0 && W >= 0, "lcn: negative size");
  const size_t n = (size_t)(N * H * W) * sizeof(float);
  Carver cv;
  const size_t ox = cv.add(n), ol = cv.add(n), os = cv.add(n);
  char* b = nullptr;
  RUN(g_ws.carve(cv.total, &b));
  if (n) CTD_REQUIRE(x && lcn && sd, "lcn: null pointer");
  if (N == 0 || n == 0) return CTD_OK;
  const int nch = chunk_count(N, g_ws.deferred);
  const size_t img = n / N;
  for (int c = 0; c < nch; ++c) {
    const int64_t i0 = chunk_lo(N, nch, c), nb = chunk_lo(N, nch, c + 1) - i0;
    const size_t o = (size_t)i0 * img;
    char* d_x = nullptr;
    RUN(g_ws.upload(g_ws.s_in, b + ox + o, (const char*)x + o, nb * img, &d_x));
    CTD_CUDA(cudaEventRecord(g_ws.ev_in[c], g_ws.s_in));
    CTD_CUDA(cudaStreamWaitEvent(g_ws.stream, g_ws.ev_in[c], 0));
    RUN(ctd_lcn_f32((float*)d_x, (float*)(b + ol + o), (float*)(b + os + o), nb, H, W, r, eps, g_ws.stream));
    CTD_CUDA(cudaEventRecord(g_ws.ev_run[c], g_ws.stream));
    CTD_CUDA(cudaStreamWaitEvent(g_ws.s_out, g_ws.ev_run[c], 0));
    D2H_ON(g_ws.s_out, (char*)lcn + o, b + ol + o, nb * img);
    D2H_ON(g_ws.s_out, (char*)sd + o, b + os + o, nb * img);
  }
  return g_ws.finish(cv.total);
}

CTD_API int ctd_host_lcn_f32(const float* x, float* lcn, float* sd, int64_t N, int64_t H, int64_t W, int r,
                                float eps) {
  Sig sg(9);
  sg.ptr(x).ptr(lcn).ptr(sd).put(N).put(H).put(W).put(r).put(eps);
  return g_ws.submit(sg.bytes, sg.host, [=]() { return lcn_host(x, lcn, sd, N, H, W, r, eps); });
}

CTD_API int ctd_host_begin_batch(void) {
  CTD_REQUIRE(!g_ws.deferred, "ctd_host_begin_batch: a batch is already open on this thread");
  if (g_ws.async_mode) {  // the other half of the workspace; at most two batches are in flight
    g_ws.slot ^= 1;
    if (int rc = g_ws.wait_slot(g_ws.slot)) return rc;
    const int other = g_ws.slot ^ 1;
    const size_t half = (g_ws.cap / 2) & ~size_t(255);
    const size_t my_lo = g_ws.slot ? half : 0, my_hi = g_ws.slot ? g_ws.cap : half;
    if (g_ws.busy[other] && g_ws.lo[other] < my_hi && my_lo < g_ws.hi[other])  // (the first asynchronous batch had the whole workspace)
      if (int rc = g_ws.wait_slot(other)) return rc;
  }
  g_ws.deferred = true;
  g_ws.used = 0;
  g_ws.uploads.clear();
  g_ws.pending.clear();
  g_ws.calls.clear();
  g_ws.mode = Workspace::EAGER;
  g_ws.cand = -1;
  g_ws.h2d_bytes = g_ws.h2d_saved = 0;
  return CTD_OK;
}

CTD_API int ctd_host_end_batch(void) {
  CTD_REQUIRE(g_ws.deferred, "ctd_host_end_batch: no batch is open on this thread");
  return g_ws.end_batch(true);
}

CTD_API int ctd_host_end_batch_async(void) {
  CTD_REQUIRE(g_ws.deferred, "ctd_host_end_batch_async: no batch is open on this thread");
  return g_ws.end_batch(false);
}

CTD_API int ctd_host_wait_batch(void) {
  CTD_REQUIRE(!g_ws.deferred, "ctd_host_wait_batch: a batch is open on this thread");
  const int oldest = g_ws.busy[g_ws.last_ended ^ 1] ? g_ws.last_ended ^ 1 : g_ws.last_ended;
  return g_ws.wait_slot(oldest);
}

CTD_API void ctd_host_batch_stats(uint64_t* h2d_bytes, uint64_t* h2d_bytes_saved) {
  if (h2d_bytes) *h2d_bytes = g_ws.h2d_bytes;
  if (h2d_bytes_saved) *h2d_bytes_saved = g_ws.h2d_saved;
}

CTD_API void ctd_host_graph_stats(uint64_t* captured, uint64_t* launched, uint64_t* bailed) {
  if (captured) *captured = g_ws.n_captured;
  if (launched) *launched = g_ws.n_replayed;
  if (bailed) *bailed = g_ws.n_bailed;
}

CTD_API void ctd_host_release(void) {
  if (g_ws.capturing) {
    cudaGraph_t g = nullptr;
    g_ws.end_capture(&g);
    if (g) cudaGraphDestroy(g);
  }
  g_ws.deferred = false;
  g_ws.used = 0;
  g_ws.calls.clear();
  g_ws.mode = Workspace::EAGER;
  g_ws.release();
}
