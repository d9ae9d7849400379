// ml_hostpath.cu -- ml_steric_local_host / ml_steric_global_host: the steric path on HOST buffers.
//
// What momlevel.steric(dset) does for variant="steric", domain="local" when the Dataset
// lives in host memory (src/momlevel/steric.py:84-184 with the reference state taken from
// time step 0, src/momlevel/reference.py:60-80): time steps are streamed through two device
// windows, the host->device copy of window k+1 running on a copy stream while the kernels of
// window k run on the compute stream.  Pinned (page-locked) host buffers make the copies
// truly asynchronous; pageable buffers work but serialise inside the driver.
#include <fcntl.h>
#include <sched.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "ml_host.cuh"

namespace {

// Worker threads of the packed transfer (below).  start() hands every worker the same job, the caller does
// its own share of the window meanwhile and then wait()s.
class Pool {
 public:
  ~Pool() {
    {
      std::lock_guard<std::mutex> l(m_);
      stop_ = true;
    }
    cv_start_.notify_all();
    for (auto& t : th_) t.join();
  }
  int size() const { return (int)th_.size(); }
  void ensure(int n) {
    std::lock_guard<std::mutex> l(m_);
    while ((int)th_.size() < n) {
      const int id = (int)th_.size();
      const uint64_t born = gen_;
      th_.emplace_back([this, id, born] { loop(id, born); });
    }
  }
  void start(int active, std::function<void(int)> job) {
    std::lock_guard<std::mutex> l(m_);
    job_ = std::move(job);
    active_ = std::min(active, (int)th_.size());
    running_ = active_;
    ++gen_;
    cv_start_.notify_all();
  }
  void wait() {
    std::unique_lock<std::mutex> l(m_);
    cv_done_.wait(l, [this] { return running_ == 0; });
  }

 private:
  void loop(int id, uint64_t seen) {
    for (;;) {
      std::function<void(int)> job;
      {
        std::unique_lock<std::mutex> l(m_);
        cv_start_.wait(l, [&] { return stop_ || gen_ != seen; });
        if (stop_) return;
        seen = gen_;
        if (id >= active_) continue;
        job = job_;
      }
      job(id);
      {
        std::lock_guard<std::mutex> l(m_);
        if (--running_ == 0) cv_done_.notify_all();
      }
    }
  }
  std::vector<std::thread> th_;
  std::mutex m_;
  std::condition_variable cv_start_, cv_done_;
  std::function<void(int)> job_;
  uint64_t gen_ = 0;
  int active_ = 0, running_ = 0;
  bool stop_ = false;
};

// Device staging buffers, pinned host staging, streams, events and the worker threads are kept per host
// thread between calls (a year of OM4p25 needs ~5 GB of windows; allocating and freeing them costs tens of
// milliseconds per call) and released by ml_host_release() or at thread exit.
// Device and pinned-host buffers of a thread's Resources, by name (a slot grows on demand and is kept between calls).
enum DevSlot {
  kDevWinT0, kDevWinS0, kDevWinT1, kDevWinS1,  // the two device windows of T and S
  kDevVol, kDevRho, kDevZi, kDevDepth, kDevP, kDevSums, kDevWs,
  kDevTref, kDevSref,                          // reference slabs held for the thermo- / halosteric variants
  kDevOut0,                                    // 6 slots: outputs [window parity][variant]
  kDevPackT0 = kDevOut0 + 6, kDevPackS0, kDevPackT1, kDevPackS1,  // packed rows [window parity][field]
  kDevWords, kDevBefore, kDevLvlOff, kDevFlags0, kDevFlags1,
  kDevSlots
};
enum HostSlot {
  kHostWords, kHostBefore, kHostLvlOff,
  kHostStageT0, kHostStageS0, kHostStageT1, kHostStageS1,  // pinned staging [window parity][field]; kHostStageT0 doubles as the ring
  kHostFlags,
  kHostOut0,                                               // 6 slots: bounce buffers of pageable outputs [parity][variant]
  kHostVol = kHostOut0 + 6,                                // bounce buffer of a pageable volcello
  kHostSlots_
};

#include "ml_hosttune.h"

struct Resources {
  static constexpr int kSlots = kDevSlots;
  static constexpr int kHostSlots = kHostSlots_;
  static constexpr int kRing = 3;  // dense rows in flight on the copy stream
  static constexpr int kStageRing = 6;  // packed rows between the packers and the copy engine (packing mode 3)
  void* buf[kSlots] = {nullptr};
  size_t cap[kSlots] = {0};
  void* hbuf[kHostSlots] = {nullptr};
  size_t hcap[kHostSlots] = {0};
  int device = -1;
  cudaStream_t copy = nullptr, comp = nullptr, back = nullptr;  // host->device, kernels, device->host
  cudaEvent_t copied[2] = {nullptr, nullptr}, freed[2] = {nullptr, nullptr};
  cudaEvent_t out_done[2] = {nullptr, nullptr};  // the outputs of a window of this parity have reached the host
  // win_start[w & 3]: the copy stream is done with window w - 1 (recorded right behind copied[] of that window; at the
  // first window: when its first copy is queued).  Timed against copied[] of window w it spans the window AND the idle
  // gap in front of it -- what a step costs -- and four of them keep a window's mark until its span has been read.
  cudaEvent_t win_start[4] = {nullptr, nullptr, nullptr, nullptr};
  PackTuner tuner;
  int tuned_choice[2] = {-1, -1};  // what the window of this parity ran with, for the tuner's report
  int64_t tuned_steps[2] = {0, 0};
  int last_pack_threads = 0;
  cudaEvent_t ring[kRing] = {nullptr};
  cudaEvent_t slot_done[kStageRing] = {nullptr};  // the copies out of a slot of the staging ring have finished
  Pool pool;
  // settings and accounting of the packed transfer (ml_host_set_packing and friends)
  int pack_mode = 1, pack_threads = 0;
  double last_packed_fraction = 0.0;
  double last_ms[4] = {0.0, 0.0, 0.0, 0.0};  // presence index, windows (host side), drain, whole call
  std::atomic<uint64_t> h2d_bytes{0};
  bool open_stream = false;  // a ml_host_stream_* computation is using the buffers
  void release() {
    for (int i = 0; i < kSlots; ++i) {
      if (buf[i]) cudaFree(buf[i]);
      buf[i] = nullptr;
      cap[i] = 0;
    }
    for (int i = 0; i < kHostSlots; ++i) {
      if (hbuf[i]) cudaFreeHost(hbuf[i]);
      hbuf[i] = nullptr;
      hcap[i] = 0;
    }
    for (int i = 0; i < 2; ++i) {
      if (copied[i]) cudaEventDestroy(copied[i]);
      if (freed[i]) cudaEventDestroy(freed[i]);
      if (out_done[i]) cudaEventDestroy(out_done[i]);
      copied[i] = freed[i] = out_done[i] = nullptr;
    }
    for (int i = 0; i < 4; ++i) {
      if (win_start[i]) cudaEventDestroy(win_start[i]);
      win_start[i] = nullptr;
    }
    for (int i = 0; i < kRing; ++i) {
      if (ring[i]) cudaEventDestroy(ring[i]);
      ring[i] = nullptr;
    }
    for (int i = 0; i < kStageRing; ++i) {
      if (slot_done[i]) cudaEventDestroy(slot_done[i]);
      slot_done[i] = nullptr;
    }
    if (copy) cudaStreamDestroy(copy);
    if (comp) cudaStreamDestroy(comp);
    if (back) cudaStreamDestroy(back);
    copy = comp = back = nullptr;
    device = -1;
  }
  ~Resources() { release(); }
  cudaError_t prepare() {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev != device) {
      release();
      device = dev;
    }
    if (!copy && (e = cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking)) != cudaSuccess) return e;
    if (!comp && (e = cudaStreamCreateWithFlags(&comp, cudaStreamNonBlocking)) != cudaSuccess) return e;
    if (!back && (e = cudaStreamCreateWithFlags(&back, cudaStreamNonBlocking)) != cudaSuccess) return e;
    for (int b = 0; b < 2; ++b) {
      if (!copied[b] && (e = cudaEventCreateWithFlags(&copied[b], 0)) != cudaSuccess) return e;  // timed: the tuner reads the span
      if (!freed[b] && (e = cudaEventCreateWithFlags(&freed[b], cudaEventDisableTiming)) != cudaSuccess) return e;
      if (!out_done[b] && (e = cudaEventCreateWithFlags(&out_done[b], cudaEventDisableTiming)) != cudaSuccess) return e;
    }
    for (int i = 0; i < 4; ++i)
      if (!win_start[i] && (e = cudaEventCreateWithFlags(&win_start[i], 0)) != cudaSuccess) return e;
    for (int i = 0; i < kRing; ++i)
      if (!ring[i] && (e = cudaEventCreateWithFlags(&ring[i], cudaEventDisableTiming)) != cudaSuccess) return e;
    for (int i = 0; i < kStageRing; ++i)
      if (!slot_done[i] && (e = cudaEventCreateWithFlags(&slot_done[i], cudaEventDisableTiming)) != cudaSuccess)
        return e;
    return cudaSuccess;
  }
  // slot i grows to at least `bytes`
  cudaError_t alloc(int i, void** p, size_t bytes) {
    if (cap[i] < bytes) {
      if (buf[i]) cudaFree(buf[i]);
      buf[i] = nullptr;
      cap[i] = 0;
      cudaError_t e = cudaMalloc(&buf[i], bytes);
      if (e != cudaSuccess) return e;
      cap[i] = bytes;
    }
    *p = buf[i];
    return cudaSuccess;
  }
  // pinned host slot i grows to at least `bytes`
  cudaError_t halloc(int i, void** p, size_t bytes) {
    if (hcap[i] < bytes) {
      if (hbuf[i]) cudaFreeHost(hbuf[i]);
      hbuf[i] = nullptr;
      hcap[i] = 0;
      cudaError_t e = cudaHostAlloc(&hbuf[i], bytes, cudaHostAllocDefault);
      if (e != cudaSuccess) return e;
      hcap[i] = bytes;
    }
    *p = hbuf[i];
    return cudaSuccess;
  }
};

// true for memory the driver does not know (malloc / numpy): copies from it are staged by the driver
bool is_pageable(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return a.type == cudaMemoryTypeUnregistered;
}

Resources& resources() {
  static thread_local Resources r;
  return r;
}

double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// memcpy by the worker threads (one thread moves ~10 GB/s, the memory system many times that)
void parallel_copy(Resources& r, void* dst, const void* src, size_t bytes, int threads) {
  threads = std::max(1, threads);
  if (bytes < (size_t)(8u << 20) || threads == 1) {
    memcpy(dst, src, bytes);
    return;
  }
  r.pool.ensure(threads);
  const size_t chunk = ((bytes + (size_t)threads - 1) / (size_t)threads + 63) & ~(size_t)63;
  r.pool.start(threads, [=](int id) {
    const size_t a = (size_t)id * chunk;
    if (a < bytes) memcpy((char*)dst + a, (const char*)src + a, std::min(chunk, bytes - a));
  });
  r.pool.wait();
}

// ---------------------------------------------------------------------------------------------------
// Packed transfer.  A window is nt_w * nz level rows of T and of S.  The reference never uses either
// field where the reference volcello is missing (steric.py:151-153, 163; derived.py:435-438), so a row
// may cross PCIe as its present cells only.  Compressing a row costs host memory bandwidth, moving it
// as it is costs PCIe time, and which of the two runs out first depends on the machine and on what
// else it is doing; so the rows of a window are put in order of how much of them is present and the
// two sides work towards each other: the calling thread queues the fullest rows as plain copies from
// the caller's buffer (at most kRing rows ahead of the copy engine), the workers compress the emptiest
// rows into pinned staging, segment by segment, and queue each one as soon as it is whole.  The
// window is done when they meet.  On the device k_unpack_rows spreads the compressed rows back into
// the dense window (NaN where the volume is missing) and the steric kernels run on it unchanged.
// ---------------------------------------------------------------------------------------------------
struct PackPlan {
  bool on = false;
  int mode = 0, threads = 0, nseg = 1;
  int64_t nz = 0, ncol = 0, ngrp = 0;
  uint64_t nwet = 0;            // present cells of one step
  uint32_t *words = nullptr, *before = nullptr;  // pinned host [nz][ngrp]
  uint64_t *lvloff = nullptr;   // pinned host [nz + 1]: present cells in the levels above
  std::vector<int> order;       // levels, fullest first
  int first_packable = 0;       // position in `order` of the first level worth compressing
  uint32_t *d_words = nullptr, *d_before = nullptr;
  uint64_t* d_lvloff = nullptr;
  float *stage[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // pinned [window parity][T,S]: [t][nwet]
  float *d_packed[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  uint8_t *flags[2] = {nullptr, nullptr}, *d_flags[2] = {nullptr, nullptr};  // [t][z]: 1 = row crossed packed
  int64_t rows_total = 0, rows_packed = 0;
  bool all_staged = false;  // pageable source: no row is copied straight from the caller's buffer
  bool tuned = false;       // the number of packing threads is the library's to choose, window by window (PackTuner)
  bool tuned_off = false;   // ... and it has settled on none: this call moves every row as it is, without an index
  // mode 3: packed rows wait for the copy engine in a ring of kStageRing row slots (T half, S half) that is
  // small enough to stay in the last-level cache, instead of in staging the size of the window
  bool ring = false;
  float* ring_buf = nullptr;
  int64_t ring_next = 0;                                    // rows that have taken a slot so far (under the lock)
  std::atomic<int64_t> slot_queued[Resources::kStageRing];  // rows whose copies out of the slot have been queued
  // mode 4: a row goes as it is only while no packed row is waiting for the copy stream
  bool packed_first = false;
  std::atomic<int> last_slot{-1};  // slot of the packed row queued last
};

constexpr double kPackableBelow = 0.9;  // a level with more of its cells present than this is never compressed
#ifdef ML_HOSTPATH_TEST_HOOKS
constexpr int64_t kSegmentGroups = 8;  // small rows are cut into several segments too
#else
constexpr int64_t kSegmentGroups = 2048;  // 32-column groups per segment of a row (64 K columns, 256 KB per field)
#endif

// tests/sim/hostpath_sim.cpp compiles this file with g++ against a simulated CUDA runtime (streams that run
// behind the host, events, pinned / pageable bookkeeping) to put the threads and the buffer recycling below under
// ThreadSanitizer on a box without a GPU; it brings its own launch_unpack().
#ifndef ML_HOSTPATH_TEST_HOOKS
__global__ void __launch_bounds__(256) k_unpack_rows(const float* __restrict__ pT, const float* __restrict__ pS,
                                                      float* __restrict__ T, float* __restrict__ S,
                                                      const uint32_t* __restrict__ words,
                                                      const uint32_t* __restrict__ before,
                                                      const uint64_t* __restrict__ lvloff,
                                                      const uint8_t* __restrict__ flags, int nz, int64_t ncol,
                                                      int64_t ngrp, uint64_t nwet, int xblocks) {
  const int row = blockIdx.x / xblocks;  // (t, z)
  if (!flags[row]) return;
  const int t = row / nz, z = row % nz;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t src0 = (uint64_t)t * nwet + lvloff[z];
  const size_t dst0 = (size_t)row * (size_t)ncol;
  const float nanf32 = __int_as_float(0x7fc00000);
  const int64_t gfirst = ((int64_t)(blockIdx.x % xblocks) * 8 + warp) * 4;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int64_t g = gfirst + k;
    if (g >= ngrp) break;
    const uint32_t m = words[(size_t)z * ngrp + g];
    const uint64_t src = src0 + before[(size_t)z * ngrp + g] + __popc(m & ((1u << lane) - 1u));
    const bool here = (m >> lane) & 1u;
    const float a = here ? pT[src] : nanf32;
    const float b = here ? pS[src] : nanf32;
    const int64_t col = g * 32 + lane;
    if (col < ncol) {
      T[dst0 + col] = a;
      S[dst0 + col] = b;
    }
  }
}

// The presence index of the reference volcello, made where the volume is going anyway: one 32-column word per
// group (bit = the cell is not NaN, as ml_pack_index_rows has it), the count of present cells in front of each
// group of its level, and the count of each level.  466 MB of an OM4p25 volume take ~0.1 ms here against 6 ms of
// eight host threads -- 20 ms when four ranks scan at once -- and the host's memory system is what the packed
// transfer is short of.
__global__ void __launch_bounds__(256) k_presence_words(const float* __restrict__ v, uint32_t* __restrict__ words,
                                                         int64_t ncol, int64_t ngrp) {
  const int64_t g = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (g >= ngrp) return;
  const int lane = threadIdx.x & 31;
  const int64_t z = blockIdx.y, col = g * 32 + lane;
  bool here = false;
  if (col < ncol) here = (__float_as_uint(v[(size_t)z * (size_t)ncol + (size_t)col]) & 0x7fffffffu) <= 0x7f800000u;
  const uint32_t m = __ballot_sync(0xffffffffu, here);
  if (lane == 0) words[(size_t)z * (size_t)ngrp + (size_t)g] = m;
}

__global__ void __launch_bounds__(1024) k_presence_before(const uint32_t* __restrict__ words, uint32_t* __restrict__ before,
                                                           uint64_t* __restrict__ count, int64_t ngrp) {
  __shared__ uint32_t warp_sum[32];
  const uint32_t* w = words + (size_t)blockIdx.x * (size_t)ngrp;
  uint32_t* b = before + (size_t)blockIdx.x * (size_t)ngrp;
  const int64_t per = (ngrp + 1023) / 1024;
  const int64_t g0 = min((int64_t)threadIdx.x * per, ngrp), g1 = min(g0 + per, ngrp);
  uint32_t mine = 0;
  for (int64_t g = g0; g < g1; ++g) mine += __popc(w[g]);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t up = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += up;
  }
  if (lane == 31) warp_sum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    uint32_t x = warp_sum[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t up = __shfl_up_sync(0xffffffffu, x, d);
      if (lane >= d) x += up;
    }
    warp_sum[lane] = x;
  }
  __syncthreads();
  uint32_t run = incl - mine + (warp ? warp_sum[warp - 1] : 0u);
  for (int64_t g = g0; g < g1; ++g) {
    b[g] = run;
    run += __popc(w[g]);
  }
  if (threadIdx.x == 1023) count[blockIdx.x] = run;
}

int launch_presence_index(cudaStream_t stream, const float* v, int64_t nz, int64_t ncol, int64_t ngrp, uint32_t* words,
                          uint32_t* before, uint64_t* count) {
  k_presence_words<<<dim3((unsigned)((ngrp + 7) / 8), (unsigned)nz), 256, 0, stream>>>(v, words, ncol, ngrp);
  int rc = ml::launched("k_presence_words");
  if (rc) return rc;
  k_presence_before<<<(unsigned)nz, 1024, 0, stream>>>(words, before, count, ngrp);
  return ml::launched("k_presence_before");
}

int launch_unpack(cudaStream_t stream, int nrows, int xblocks, const float* pT, const float* pS, float* T, float* S,
                  const uint32_t* words, const uint32_t* before, const uint64_t* lvloff, const uint8_t* flags, int nz,
                  int64_t ncol, int64_t ngrp, uint64_t nwet) {
  k_unpack_rows<<<(unsigned)((int64_t)nrows * xblocks), 256, 0, stream>>>(pT, pS, T, S, words, before, lvloff, flags, nz,
                                                                          ncol, ngrp, nwet, xblocks);
  return ml::launched("k_unpack_rows");
}
#endif

// Presence words of the reference volcello, the device copies of them and the staging buffers.
// Leaves plan.on false (every row crosses as it is) when packing is off, cannot help or cannot get
// its pinned memory.
int plan_packing(Resources& r, PackPlan& plan, int dtype, const void* d_v0, int64_t nz, int64_t ncol, int64_t spw,
                 bool allowed, bool pageable) {
  using namespace ml;
  plan.on = false;
  plan.mode = r.pack_mode;
  plan.all_staged = false;
  plan.tuned_off = false;
  if (!allowed || plan.mode == 0 || dtype != ML_F32) return ML_OK;
  if (nz > 65535) return ML_OK;  // a level is a grid row of the index kernels
  plan.nz = nz;
  plan.ncol = ncol;
  plan.ngrp = (ncol + 31) / 32;
  plan.threads = r.pack_threads > 0 ? std::min(r.pack_threads, 64) : default_threads();
  plan.tuned = r.pack_mode == 1 && r.pack_threads <= 0;
  if (plan.tuned) {
    const int cap = max_threads();
    if (r.tuner.nz != nz || r.tuner.ncol != ncol || r.tuner.threads[0] != default_threads()) r.tuner.reset(nz, ncol, default_threads(), cap);
    plan.threads = std::max(plan.threads, r.tuner.threads[2]);  // the pool holds the largest choice
    if (!pageable && r.tuner.settled_on_none()) {
      plan.tuned_off = true;
      r.last_pack_threads = 0;
      return ML_OK;
    }
  }
  plan.nseg = (int)std::max<int64_t>(1, std::min<int64_t>(64, plan.ngrp / kSegmentGroups));
  const size_t nw = (size_t)nz * (size_t)plan.ngrp;
  void *hw, *hb, *hl;
  if (r.halloc(kHostWords, &hw, nw * 4) != cudaSuccess || r.halloc(kHostBefore, &hb, nw * 4) != cudaSuccess ||
      r.halloc(kHostLvlOff, &hl, (size_t)(nz + 1) * 8) != cudaSuccess) {
    cudaGetLastError();
    return ML_OK;
  }
  plan.words = (uint32_t*)hw;
  plan.before = (uint32_t*)hb;
  plan.lvloff = (uint64_t*)hl;
  r.pool.ensure(plan.threads);
  // the index is made on the device, behind the upload of the volume on the copy stream, and comes back for the
  // packers; lvloff[1 ...] receives the level counts and is summed in place
  void *dw, *db, *dl;
  ML_CUDA(r.alloc(kDevWords, &dw, nw * 4));
  ML_CUDA(r.alloc(kDevBefore, &db, nw * 4));
  ML_CUDA(r.alloc(kDevLvlOff, &dl, (size_t)(nz + 1) * 8));
  plan.d_words = (uint32_t*)dw;
  plan.d_before = (uint32_t*)db;
  plan.d_lvloff = (uint64_t*)dl;
  {
    int rc = launch_presence_index(r.copy, (const float*)d_v0, nz, ncol, plan.ngrp, plan.d_words, plan.d_before, plan.d_lvloff + 1);
    if (rc) return rc;
  }
  ML_CUDA(cudaMemcpyAsync(plan.words, dw, nw * 4, cudaMemcpyDeviceToHost, r.copy));
  ML_CUDA(cudaMemcpyAsync(plan.before, db, nw * 4, cudaMemcpyDeviceToHost, r.copy));
  ML_CUDA(cudaMemcpyAsync(plan.lvloff + 1, plan.d_lvloff + 1, (size_t)nz * 8, cudaMemcpyDeviceToHost, r.copy));
  ML_CUDA(cudaStreamSynchronize(r.copy));
  std::vector<uint64_t> cnt((size_t)nz);
  plan.lvloff[0] = 0;
  for (int64_t z = 0; z < nz; ++z) {
    cnt[z] = plan.lvloff[z + 1];
    plan.lvloff[z + 1] = plan.lvloff[z] + cnt[z];
  }
  plan.nwet = plan.lvloff[nz];
  plan.order.resize((size_t)nz);
  for (int64_t z = 0; z < nz; ++z) plan.order[z] = (int)z;
  std::stable_sort(plan.order.begin(), plan.order.end(), [&](int a, int b) { return cnt[a] > cnt[b]; });
  plan.first_packable = (int)nz;
  for (int64_t i = 0; i < nz; ++i)
    if ((double)cnt[plan.order[i]] < kPackableBelow * (double)ncol) {
      plan.first_packable = (int)i;
      break;
    }
  if (pageable && plan.nwet != 0) {
    // Pageable source (a plain numpy array): a DMA from it is a synchronous, single-threaded bounce through the
    // driver at a fraction of the PCIe rate, so every row goes through the packers and the pinned staging,
    // full rows included.
    plan.all_staged = true;
    plan.first_packable = 0;
  }
  if (plan.first_packable == (int)nz || plan.nwet == 0) return ML_OK;  // nothing worth compressing
  const size_t stage_bytes = (size_t)spw * plan.nwet * 4;
  const size_t flag_bytes = (size_t)spw * (size_t)nz;
  plan.ring = plan.mode >= 3;
  plan.packed_first = plan.mode == 4;
  plan.last_slot.store(-1);
  plan.ring_next = 0;
  for (auto& q : plan.slot_queued) q.store(0, std::memory_order_relaxed);
  if (plan.ring) {
    void* h;
    if (r.halloc(kHostStageT0, &h, (size_t)Resources::kStageRing * 2 * (size_t)ncol * 4) != cudaSuccess) {
      cudaGetLastError();
      return ML_OK;
    }
    plan.ring_buf = (float*)h;
  }
  for (int b = 0; b < 2; ++b) {
    for (int f = 0; f < 2; ++f) {
      void *h = nullptr, *d;
      if (!plan.ring && r.halloc(kHostStageT0 + 2 * b + f, &h, stage_bytes) != cudaSuccess) {
        cudaGetLastError();
        return ML_OK;
      }
      ML_CUDA(r.alloc(kDevPackT0 + 2 * b + f, &d, stage_bytes));
      plan.stage[b][f] = (float*)h;
      plan.d_packed[b][f] = (float*)d;
    }
    void *hf, *df;
    if (r.halloc(kHostFlags, &hf, 2 * flag_bytes) != cudaSuccess) {
      cudaGetLastError();
      return ML_OK;
    }
    ML_CUDA(r.alloc(kDevFlags0 + b, &df, flag_bytes));
    plan.flags[b] = (uint8_t*)hf + (size_t)b * flag_bytes;
    plan.d_flags[b] = (uint8_t*)df;
  }
  ML_CUDA(cudaMemcpyAsync(plan.d_lvloff, plan.lvloff, (size_t)(nz + 1) * 8, cudaMemcpyHostToDevice, r.copy));
  r.h2d_bytes += (size_t)(nz + 1) * 8;
  plan.on = true;
  return ML_OK;
}

// One window of T and S to the device buffers dT / dS of parity b: on return every copy is queued on the
// copy stream, copied[b] is recorded behind them and the compute stream waits for it (and has expanded
// the rows that crossed packed).  T_w / S_w point at the window's first step in the caller's buffers.
int stage_window(Resources& r, PackPlan& plan, int b, int64_t w, const void* T_w, const void* S_w, int64_t nt_w,
                 size_t es, int64_t nz, int64_t ncol, void* dT, void* dS) {
  using namespace ml;
  const size_t bytes = (size_t)nt_w * (size_t)nz * (size_t)ncol * es;
  if (w >= 2) ML_CUDA(cudaStreamWaitEvent(r.copy, r.freed[b], 0));
  if (!plan.on) {
    ML_CUDA(cudaMemcpyAsync(dT, T_w, bytes, cudaMemcpyHostToDevice, r.copy));
    ML_CUDA(cudaMemcpyAsync(dS, S_w, bytes, cudaMemcpyHostToDevice, r.copy));
    r.h2d_bytes += 2 * bytes;
    ML_CUDA(cudaEventRecord(r.copied[b], r.copy));
    ML_CUDA(cudaStreamWaitEvent(r.comp, r.copied[b], 0));
    if (plan.tuned_off) r.tuner.idle_window();
    return ML_OK;
  }
  // the staging of this parity was last read by the copies of window w - 2
  if (w >= 2) ML_CUDA(cudaEventSynchronize(r.copied[b]));
  // how many threads pack this window: the caller's number, or -- left to the library -- what the tuner has found
  // fastest on this machine, under this load (PackTuner); a pageable source is staged in full whatever it says
  const bool tuned = plan.tuned && !plan.all_staged;
  int active = plan.threads;
  if (tuned) {
    if (w >= 2 && r.tuned_choice[b] >= 0) {  // the span of window w - 2 on the copy stream is known now
      float ms = 0.0f;
      if (cudaEventElapsedTime(&ms, r.win_start[(w - 2) & 3], r.copied[b]) == cudaSuccess)
        r.tuner.report(r.tuned_choice[b], (double)ms, r.tuned_steps[b]);
      else
        cudaGetLastError();
    }
    const int choice = r.tuner.choose();
    active = std::min(r.tuner.threads[choice], plan.threads);
    r.tuned_choice[b] = choice;
    r.tuned_steps[b] = nt_w;
    if (w == 0 || r.tuned_choice[b ^ 1] < 0) ML_CUDA(cudaEventRecord(r.win_start[w & 3], r.copy));  // else: behind window w - 1
  } else {
    r.tuned_choice[b] = -1;
  }
  r.last_pack_threads = active;

  const float* Th = (const float*)T_w;
  const float* Sh = (const float*)S_w;
  const int nrows = (int)(nt_w * nz);
  const size_t row_bytes = (size_t)ncol * 4;
  uint8_t* flags = plan.flags[b];
  memset(flags, 0, (size_t)nrows);
  // position i of the window's row order = step i % nt_w of level order[i / nt_w]
  auto row_of = [&](int i, int& t, int& z) {
    z = plan.order[i / (int)nt_w];
    t = i % (int)nt_w;
  };
  struct Shared {
    std::mutex m;
    int lo = 0, hi = 0, hi_min = 0, lo_end = 0;
    int cur = -1, next_seg = 0, cur_slot = 0;
    int packed = 0;
    std::atomic<int> err{(int)cudaSuccess};  // first CUDA error of any thread; set without the lock
  } sh;
  sh.hi = nrows - 1;
  sh.hi_min = plan.first_packable * (int)nt_w;
  sh.lo_end = (plan.mode == 2 || plan.all_staged) ? sh.hi_min : nrows;
  sh.next_seg = plan.nseg;  // no row open yet
  std::vector<std::atomic<int>> done((size_t)nrows);
  for (auto& d : done) d.store(0, std::memory_order_relaxed);
  const int dev = r.device;
  float *stT = plan.stage[b][0], *stS = plan.stage[b][1];
  float *dpT = plan.d_packed[b][0], *dpS = plan.d_packed[b][1];

  r.pool.start(active, [&, dev](int) {
    cudaSetDevice(dev);
    for (;;) {
      int pos, seg, slot;
      {
        std::lock_guard<std::mutex> l(sh.m);
        if (sh.next_seg >= plan.nseg) {
          if (sh.hi < sh.lo || sh.hi < sh.hi_min || sh.err.load() != (int)cudaSuccess) break;
          sh.cur = sh.hi--;
          sh.next_seg = 0;
          sh.packed++;
          if (plan.ring) {
            // the next slot of the ring, once the copy engine has emptied it.  Waiting here, with the lock held,
            // keeps every packer (they all want this row) no more than kStageRing rows ahead of the copies.
            const int64_t turn = plan.ring_next++;
            sh.cur_slot = (int)(turn % Resources::kStageRing);
            // the slot's previous row must have been queued (its last segment may still be with a thread that
            // lost its core) before the event below speaks for it
            while (plan.slot_queued[sh.cur_slot].load(std::memory_order_acquire) < turn / Resources::kStageRing &&
                   sh.err.load() == (int)cudaSuccess)
              std::this_thread::yield();
            const cudaError_t e = cudaEventSynchronize(r.slot_done[sh.cur_slot]);
            if (e != cudaSuccess) {
              sh.err.store((int)e);
              break;
            }
          }
        }
        pos = sh.cur;
        seg = sh.next_seg++;
        slot = sh.cur_slot;
      }
      int t, z;
      row_of(pos, t, z);
      const size_t src = ((size_t)t * (size_t)nz + (size_t)z) * (size_t)ncol;
      const size_t dst = (size_t)t * plan.nwet + plan.lvloff[z];
      const int64_t g0 = plan.ngrp * seg / plan.nseg, g1 = plan.ngrp * (seg + 1) / plan.nseg;
      float* rowT = plan.ring ? plan.ring_buf + (size_t)slot * 2 * (size_t)ncol : stT + dst;
      float* rowS = plan.ring ? rowT + (size_t)ncol : stS + dst;
      if (plan.ring)
        ml_pack_rows_cached(Th + src, Sh + src, plan.words + (size_t)z * plan.ngrp,
                            plan.before + (size_t)z * plan.ngrp, g0, g1, ncol, rowT, rowS);
      else
        ml_pack_rows(Th + src, Sh + src, plan.words + (size_t)z * plan.ngrp, plan.before + (size_t)z * plan.ngrp, g0,
                     g1, ncol, rowT, rowS);
      const int row = t * (int)nz + z;
      if (done[row].fetch_add(1, std::memory_order_acq_rel) + 1 == plan.nseg) {  // the row is whole: queue it
        const size_t nb = (size_t)(plan.lvloff[z + 1] - plan.lvloff[z]) * 4;
        flags[row] = 1;
        cudaError_t e = cudaSuccess;
        if (nb) {
          e = cudaMemcpyAsync(dpT + dst, rowT, nb, cudaMemcpyHostToDevice, r.copy);
          if (e == cudaSuccess) e = cudaMemcpyAsync(dpS + dst, rowS, nb, cudaMemcpyHostToDevice, r.copy);
          r.h2d_bytes += 2 * nb;
        }
        if (plan.ring && e == cudaSuccess) e = cudaEventRecord(r.slot_done[slot], r.copy);
        if (e != cudaSuccess) sh.err.store((int)e);
        if (plan.ring) {
          plan.last_slot.store(slot, std::memory_order_release);
          plan.slot_queued[slot].fetch_add(1, std::memory_order_release);
        }
      }
    }
  });

  // this thread: the fullest rows as they are, straight from the caller's buffer
  cudaError_t err = cudaSuccess;
  const int in_flight = plan.packed_first ? 1 : Resources::kRing;
  for (int issued = 0;; ++issued) {
    int pos;
    if (plan.packed_first) {
      // the copy stream belongs to the packed rows: wait until the one queued last has crossed (the stream is
      // in order, so then none is waiting) or until the rows have run out
      for (;;) {
        const int last = plan.last_slot.load(std::memory_order_acquire);
        if (last < 0) break;
        const cudaError_t q = cudaEventQuery(r.slot_done[last]);
        if (q == cudaSuccess) break;
        cudaGetLastError();  // cudaErrorNotReady is an answer, not a failure
        if (q != cudaErrorNotReady) {
          err = q;
          break;
        }
        {
          std::lock_guard<std::mutex> l(sh.m);
          if (sh.lo > sh.hi || sh.lo >= sh.lo_end) break;
        }
        std::this_thread::sleep_for(std::chrono::microseconds(20));
      }
      if (err != cudaSuccess) break;
    }
    {
      std::lock_guard<std::mutex> l(sh.m);
      if (sh.lo > sh.hi || sh.lo >= sh.lo_end) break;
      pos = sh.lo++;
    }
    int t, z;
    row_of(pos, t, z);
    const size_t off = ((size_t)t * (size_t)nz + (size_t)z) * (size_t)ncol;
    cudaEvent_t ev = r.ring[issued % in_flight];
    if (issued >= in_flight && (err = cudaEventSynchronize(ev)) != cudaSuccess) break;
    if ((err = cudaMemcpyAsync((float*)dT + off, Th + off, row_bytes, cudaMemcpyHostToDevice, r.copy)) != cudaSuccess) break;
    if ((err = cudaMemcpyAsync((float*)dS + off, Sh + off, row_bytes, cudaMemcpyHostToDevice, r.copy)) != cudaSuccess) break;
    r.h2d_bytes += 2 * row_bytes;
    if ((err = cudaEventRecord(ev, r.copy)) != cudaSuccess) break;
  }
  if (err != cudaSuccess) sh.err.store((int)err);  // stops the workers; wait for them before the locals they captured go
  r.pool.wait();
  if (sh.err.load() != (int)cudaSuccess) return cuda_fail((cudaError_t)sh.err.load(), "packed transfer");
  plan.rows_total += nrows;
  plan.rows_packed += sh.packed;

  if (sh.packed) {
    ML_CUDA(cudaMemcpyAsync(plan.d_flags[b], flags, (size_t)nrows, cudaMemcpyHostToDevice, r.copy));
    r.h2d_bytes += (size_t)nrows;
  }
  ML_CUDA(cudaEventRecord(r.copied[b], r.copy));
  if (tuned) ML_CUDA(cudaEventRecord(r.win_start[(w + 1) & 3], r.copy));  // the next window's interval starts here
  ML_CUDA(cudaStreamWaitEvent(r.comp, r.copied[b], 0));
  if (sh.packed) {
    const int xblocks = (int)((plan.ngrp + 31) / 32);
    if (int rc = launch_unpack(r.comp, nrows, xblocks, dpT, dpS, (float*)dT, (float*)dS, plan.d_words, plan.d_before,
                               plan.d_lvloff, plan.d_flags[b], (int)nz, ncol, plan.ngrp, plan.nwet))
      return rc;
  }
  return ML_OK;
}

}  // namespace

// Test entry (tests/test_host_logic.py, two processes on the CPU box): attach to the segment of a made-up job as
// `rank` of `ranks`, publish `ms4`, wait (at most wait_ms) until every rank has published, return the combined table,
// and leave only when every rank has read it.  Returns the number of ranks seen, or a negative status.
extern "C" int ml_host_tuner_share_selftest(const char* port, int rank, int ranks, int64_t nz, int64_t ncol, const double* ms4,
                                            double* combined4, int wait_ms) {
  if (port == nullptr || ms4 == nullptr || combined4 == nullptr || rank < 0 || rank >= ranks || ranks > SharedTuning::kMaxRanks)
    return ML_ERR_SHAPE;
  SharedTuning t(false);  // never the segment of the job this process may belong to
  t.ranks = ranks;
  t.attach("selftest", port, "selftest", rank);
  if (t.slots == nullptr) return ML_ERR_MODE;
  const int threads[4] = {4, 0, 8, 2};
  __atomic_store_n(&t.slots[rank].seen, 0, __ATOMIC_RELAXED);
  t.publish(nz, ncol, threads, ms4);
  auto count = [&](bool read) {
    int n = 0;
    for (int r = 0; r < ranks; ++r)
      n += __atomic_load_n(&t.slots[r].nz, __ATOMIC_ACQUIRE) == nz && (!read || __atomic_load_n(&t.slots[r].seen, __ATOMIC_ACQUIRE) == 1);
    return n;
  };
  const double t0 = now_ms();
  while (count(false) < ranks && now_ms() - t0 < (double)wait_ms) usleep(1000);
  const int seen = count(false);
  t.combine(nz, ncol, threads, ms4, combined4);
  __atomic_store_n(&t.slots[rank].seen, 1, __ATOMIC_RELEASE);
  while (count(true) < ranks && now_ms() - t0 < 2.0 * (double)wait_ms) usleep(1000);
  return seen;
}

extern "C" int ml_host_release(void) {
  resources().release();
  return ML_OK;
}

extern "C" int ml_host_set_packing(int mode, int threads) {
  if (mode < 0 || mode > 4) return ml::fail(ML_ERR_MODE, "packing mode %d is not 0 ... 4", mode);
  Resources& r = resources();
  r.pack_mode = mode;
  r.pack_threads = threads > 0 ? threads : 0;
  return ML_OK;
}

extern "C" double ml_host_last_packed_fraction(void) { return resources().last_packed_fraction; }

extern "C" int ml_host_last_pack_threads(void) { return resources().last_pack_threads; }

extern "C" uint64_t ml_host_last_h2d_bytes(void) { return resources().h2d_bytes.load(); }

extern "C" int ml_host_last_timings(double* ms4) {
  ML_REQUIRE_PTR(ms4);
  for (int i = 0; i < 4; ++i) ms4[i] = resources().last_ms[i];
  return ML_OK;
}

// ---------------------------------------------------------------------------------------------------
// Streamed computation: begin -> push (one block of time steps after the other, as they arrive) -> finish.
// The whole-array entry points below are begin + one push per window + finish, so there is one code path.
// ---------------------------------------------------------------------------------------------------
namespace {

struct HostStream {
  Resources* r = nullptr;
  std::thread::id owner;
  int domain = ML_DOMAIN_LOCAL, eos = 0, dtype = 0, vref_dtype = 0;
  size_t es = 4;
  int64_t nz = 0, ncol = 0, max_steps = 0;
  bool want[3] = {true, false, false};  // steric, thermosteric, halosteric
  bool selfref = true;                  // the reference state is step 0 of the first block
  bool want_rho_ref = false;
  bool want_sums = true;                // global domain: evaluate volo / masso of the reference state from step 0
  double coef = 0.0;
  int64_t blocks = 0, steps = 0;
  bool failed = false;
  PackPlan plan;
  void *dT[2] = {nullptr, nullptr}, *dS[2] = {nullptr, nullptr};
  void *dV = nullptr, *dRho = nullptr, *dZi = nullptr, *dDepth = nullptr, *dP = nullptr, *dSums = nullptr, *dWs = nullptr;
  void *dTref = nullptr, *dSref = nullptr;
  double* dOut[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};
  size_t ws_bytes = 0;
  // outputs of a block land in the caller's arrays directly (pinned) or through a pinned bounce buffer (pageable)
  struct Pending {
    double *user = nullptr, *bounce = nullptr;
    size_t bytes = 0;
  } pending[2][3];
  int nthreads = 1;
  bool release_previous = true;  // push(k) returns once block k - 1 has left the caller's memory
  double t_begin = 0.0, t_plan = 0.0;
};

// an error leaves copies and kernels in flight that read the caller's block and write buffers the next call reuses
int stream_fail(HostStream* hs, int rc) {
  if (hs->r) {
    cudaStreamSynchronize(hs->r->copy);
    cudaStreamSynchronize(hs->r->comp);
    cudaStreamSynchronize(hs->r->back);
  }
  hs->failed = true;
  return rc;
}

// pageable outputs of the block that used parity b: bounce buffer -> caller's array (the copies behind out_done[b] are done)
void flush_pending(HostStream* hs, int b) {
  for (int v = 0; v < 3; ++v) {
    HostStream::Pending& p = hs->pending[b][v];
    if (p.user != nullptr && p.bounce != nullptr && p.bytes) parallel_copy(*hs->r, p.user, p.bounce, p.bytes, hs->nthreads);
    p = HostStream::Pending();
  }
}

}  // namespace

extern "C" int ml_host_stream_begin(int domain, int eos, int dtype, int variants, const void* v_ref, int vref_dtype,
                                    const void* T_ref, const void* S_ref, const double* rho_ref, const double* z_i,
                                    const double* deptho,
                                    const double* p_level, double neg_inv_rhozero, int64_t nz, int64_t ncol,
                                    int64_t max_block_steps, int want_reference, void** stream_out) {
  using namespace ml;
  ML_REQUIRE_PTR(stream_out);
  *stream_out = nullptr;
  if (domain != ML_DOMAIN_LOCAL && domain != ML_DOMAIN_GLOBAL) return fail(ML_ERR_MODE, "unknown domain %d", domain);
  if (eos != ML_EOS_WRIGHT && eos != ML_EOS_LINEAR) return fail(ML_ERR_EOS, "unknown equation of state id %d", eos);
  if (dtype != ML_F32 && dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown dtype id %d", dtype);
  if (vref_dtype != ML_F32 && vref_dtype != ML_F64) return fail(ML_ERR_DTYPE, "unknown vref dtype id %d", vref_dtype);
  if ((variants & 7) == 0 || (variants & ~7)) return fail(ML_ERR_MODE, "variants mask %d: bit 0 steric, 1 thermosteric, 2 halosteric", variants);
  ML_REQUIRE_PTR(v_ref);
  ML_REQUIRE_PTR(p_level);
  const bool local = domain == ML_DOMAIN_LOCAL;
  if (local) {
    ML_REQUIRE_PTR(z_i);
    ML_REQUIRE_PTR(deptho);
  }
  if (nz <= 0 || ncol <= 0 || max_block_steps < 1)
    return fail(ML_ERR_SHAPE, "bad extents nz=%lld ncol=%lld block=%lld", (long long)nz, (long long)ncol, (long long)max_block_steps);
  // a supplied reference: the slabs that the thermo- / halosteric variants hold fixed, and (local) its density
  const bool supplied = T_ref != nullptr || S_ref != nullptr || rho_ref != nullptr;
  const bool others = (variants & 6) != 0;
  if (supplied) {
    if (local) ML_REQUIRE_PTR(rho_ref);
    if (others) {
      ML_REQUIRE_PTR(T_ref);
      ML_REQUIRE_PTR(S_ref);
    }
  }

  Resources& r = resources();
  if (r.open_stream) return fail(ML_ERR_MODE, "this thread already has an open host stream (finish or abort it first)");
  HostStream* hs = new HostStream();
  hs->r = &r;
  hs->owner = std::this_thread::get_id();
  hs->domain = domain;
  hs->eos = eos;
  hs->dtype = dtype;
  hs->es = (size_t)elem_size(dtype);
  hs->vref_dtype = vref_dtype;
  hs->nz = nz;
  hs->ncol = ncol;
  hs->max_steps = max_block_steps;
  for (int v = 0; v < 3; ++v) hs->want[v] = (variants >> v) & 1;
  hs->selfref = !supplied;
  hs->want_rho_ref = (want_reference & 1) != 0;
  hs->want_sums = (want_reference & 2) != 0 || local;
  hs->coef = neg_inv_rhozero;
  hs->nthreads = r.pack_threads > 0 ? std::min(r.pack_threads, 64) : default_threads();
  const size_t es = hs->es, lvl = (size_t)nz * (size_t)ncol, ves = (size_t)elem_size(vref_dtype);
  const size_t win_bytes = (size_t)max_block_steps * lvl * es;
  // a global stream that asks for two or more masses runs ml_steric_global_variants: three rows of partials per step
  const int nwanted = (variants & 1) + ((variants >> 1) & 1) + ((variants >> 2) & 1);
  hs->ws_bytes = ml_workspace_bytes(local ? 2 : std::max<int64_t>(2, (nwanted >= 2 ? 3 : 1) * max_block_steps), nz, ncol);
  auto bail = [&](int rc) {
    stream_fail(hs, rc);
    delete hs;
    return rc;
  };
#define ML_HS_CUDA(call)                                      \
  do {                                                        \
    cudaError_t e__ = (call);                                 \
    if (e__ != cudaSuccess) return bail(cuda_fail(e__, #call)); \
  } while (0)
  ML_HS_CUDA(r.prepare());
  for (int b = 0; b < 2; ++b) {
    ML_HS_CUDA(r.alloc(kDevWinT0 + 2 * b, &hs->dT[b], win_bytes));
    ML_HS_CUDA(r.alloc(kDevWinS0 + 2 * b, &hs->dS[b], win_bytes));
    const size_t out_bytes = (size_t)max_block_steps * (local ? (size_t)ncol : 1) * sizeof(double);
    for (int v = 0; v < 3; ++v) {
      void* d = nullptr;
      if (hs->want[v]) ML_HS_CUDA(r.alloc(kDevOut0 + 3 * b + v, &d, out_bytes));
      hs->dOut[b][v] = (double*)d;
    }
  }
  ML_HS_CUDA(r.alloc(kDevVol, &hs->dV, lvl * ves));
  ML_HS_CUDA(r.alloc(kDevP, &hs->dP, (size_t)nz * sizeof(double)));
  ML_HS_CUDA(r.alloc(kDevWs, &hs->dWs, hs->ws_bytes));
  ML_HS_CUDA(r.alloc(kDevSums, &hs->dSums, 2 * sizeof(double)));
  // the reference density: read by every local window; evaluated for the scalars of a self-referenced global series
  if (local || (!supplied && hs->want_sums)) ML_HS_CUDA(r.alloc(kDevRho, &hs->dRho, lvl * sizeof(double)));
  if (local) {
    ML_HS_CUDA(r.alloc(kDevZi, &hs->dZi, (size_t)(nz + 1) * sizeof(double)));
    ML_HS_CUDA(r.alloc(kDevDepth, &hs->dDepth, (size_t)ncol * sizeof(double)));
  }
  if (others) {
    ML_HS_CUDA(r.alloc(kDevTref, &hs->dTref, lvl * es));
    ML_HS_CUDA(r.alloc(kDevSref, &hs->dSref, lvl * es));
  }

  r.h2d_bytes = 0;
  r.last_packed_fraction = 0.0;
  hs->t_begin = now_ms();
  if (local) {
    ML_HS_CUDA(cudaMemcpyAsync(hs->dZi, z_i, (size_t)(nz + 1) * sizeof(double), cudaMemcpyHostToDevice, r.copy));
    ML_HS_CUDA(cudaMemcpyAsync(hs->dDepth, deptho, (size_t)ncol * sizeof(double), cudaMemcpyHostToDevice, r.copy));
    r.h2d_bytes += (size_t)(nz + 1 + ncol) * sizeof(double);
  }
  ML_HS_CUDA(cudaMemcpyAsync(hs->dP, p_level, (size_t)nz * sizeof(double), cudaMemcpyHostToDevice, r.copy));
  // Pageable memory (plain numpy) on either end of a copy makes it a synchronous bounce through the driver that
  // holds this thread -- and with it the pipeline -- for the length of the copy.  Unless packing is off such
  // operands go through pinned buffers of our own, filled / emptied by the worker threads.
  const void* v_src = v_ref;
  if (r.pack_mode != 0 && is_pageable(v_ref)) {
    void* hv;
    if (r.halloc(kHostVol, &hv, lvl * ves) == cudaSuccess) {
      parallel_copy(r, hv, v_ref, lvl * ves, hs->nthreads);
      v_src = hv;
    } else {
      cudaGetLastError();
    }
  }
  ML_HS_CUDA(cudaMemcpyAsync(hs->dV, v_src, lvl * ves, cudaMemcpyHostToDevice, r.copy));
  r.h2d_bytes += (size_t)nz * sizeof(double) + lvl * ves;
  if (supplied) {
    if (local) ML_HS_CUDA(cudaMemcpyAsync(hs->dRho, rho_ref, lvl * sizeof(double), cudaMemcpyHostToDevice, r.copy));
    if (others) {
      ML_HS_CUDA(cudaMemcpyAsync(hs->dTref, T_ref, lvl * es, cudaMemcpyHostToDevice, r.copy));
      ML_HS_CUDA(cudaMemcpyAsync(hs->dSref, S_ref, lvl * es, cudaMemcpyHostToDevice, r.copy));
    }
    r.h2d_bytes += (local ? lvl * sizeof(double) : 0) + (others ? 2 * lvl * es : 0);
  }
#undef ML_HS_CUDA
  // the packing plan is made at the first push: it depends on where the blocks live (pinned or pageable memory)
  r.open_stream = true;
  *stream_out = hs;
  return ML_OK;
}


// Referenced weakly: this file is also built on its own against a simulated runtime with stand-ins for the
// single-height entry points only (tests/sim), where the windows then take one ml_steric_global per mass.
extern "C" int ml_steric_global_variants(int, int, const void*, const void*, const void*, const void*, const void*, int,
                                         const double*, int64_t, int64_t, int64_t, double*, double*, double*, double*,
                                         void*, size_t, void*) __attribute__((weak));

extern "C" int ml_host_stream_push(void* stream, const void* T_block, const void* S_block, int64_t nt_block,
                                   double* out_steric, double* out_thermosteric, double* out_halosteric) {
  using namespace ml;
  ML_REQUIRE_PTR(stream);
  HostStream* hs = static_cast<HostStream*>(stream);
  if (hs->failed) return fail(ML_ERR_MODE, "the stream has failed; abort it");
  if (hs->owner != std::this_thread::get_id()) return fail(ML_ERR_MODE, "a host stream belongs to the thread that began it");
  ML_REQUIRE_PTR(T_block);
  ML_REQUIRE_PTR(S_block);
  if (nt_block < 1 || nt_block > hs->max_steps)
    return fail(ML_ERR_SHAPE, "block of %lld steps, the stream takes 1 ... %lld", (long long)nt_block, (long long)hs->max_steps);
  double* user_out[3] = {out_steric, out_thermosteric, out_halosteric};
  for (int v = 0; v < 3; ++v)
    if (hs->want[v] && user_out[v] == nullptr) return fail(ML_ERR_NULL, "output %d of the stream is NULL", v);
  Resources& r = *hs->r;
  const int64_t w = hs->blocks, nz = hs->nz, ncol = hs->ncol;
  const int b = (int)(w & 1);
  const bool local = hs->domain == ML_DOMAIN_LOCAL;
  const size_t lvl = (size_t)nz * (size_t)ncol, es = hs->es;
  const bool others = hs->want[1] || hs->want[2];
  const int eos = hs->eos, dtype = hs->dtype, vdt = hs->vref_dtype;
#define ML_HS_CUDA(call)                                                   \
  do {                                                                     \
    cudaError_t e__ = (call);                                              \
    if (e__ != cudaSuccess) return stream_fail(hs, cuda_fail(e__, #call)); \
  } while (0)
#define ML_HS_RC(call)                       \
  do {                                       \
    int rc__ = (call);                       \
    if (rc__) return stream_fail(hs, rc__);  \
  } while (0)
  if (w == 0) {
    // rho_ref is defined where the volume is missing too (reference.py:71), so a stream that hands it back moves
    // every row as it is; so does one whose reference volume is not stored like the fields
    const bool pageable = is_pageable(T_block) || is_pageable(S_block);
    ML_HS_RC(plan_packing(r, hs->plan, vdt == dtype ? dtype : ML_F64, hs->dV, nz, ncol, hs->max_steps, !hs->want_rho_ref,
                          pageable));
    hs->t_plan = now_ms();
  }
  if (w >= 2) {  // the outputs of block w - 2 have reached the host: its device output buffers and bounce buffers are free
    ML_HS_CUDA(cudaEventSynchronize(r.out_done[b]));
    flush_pending(hs, b);
  }
  ML_HS_RC(stage_window(r, hs->plan, b, w, T_block, S_block, nt_block, es, nz, ncol, hs->dT[b], hs->dS[b]));

  const double *dZi = (const double*)hs->dZi, *dDepth = (const double*)hs->dDepth, *dP = (const double*)hs->dP;
  const bool first_selfref = hs->selfref && w == 0;
  if (!local && first_selfref && hs->want_sums) {
    // the scalars of the reference state (reference.py:74-80) from step 0 of the first block
    ML_HS_RC(ml_reference_state(eos, dtype, hs->dT[0], hs->dS[0], hs->dV, dP, nz, ncol, (double*)hs->dRho, (double*)hs->dSums,
                                hs->dWs, hs->ws_bytes, r.comp));
  }
  if (first_selfref && others) {  // keep the reference slabs before window 0 is recycled (steric.py:115-121)
    ML_HS_CUDA(cudaMemcpyAsync(hs->dTref, hs->dT[0], lvl * es, cudaMemcpyDeviceToDevice, r.comp));
    ML_HS_CUDA(cudaMemcpyAsync(hs->dSref, hs->dS[0], lvl * es, cudaMemcpyDeviceToDevice, r.comp));
  }
  // a global window that asks for two or more masses: all of them from one pass (the reference slabs are device
  // copies, so this is never a self-reference call; the scalars came from ml_reference_state above)
  const bool one_pass = !local && hs->want[0] + hs->want[1] + hs->want[2] >= 2 && ml_steric_global_variants != nullptr;
  if (one_pass)
    ML_HS_RC(ml_steric_global_variants(eos, dtype, hs->dT[b], hs->dS[b], hs->dTref, hs->dSref, hs->dV, vdt, dP, nt_block, nz,
                                       ncol, hs->dOut[b][0], hs->dOut[b][1], hs->dOut[b][2], nullptr, hs->dWs, hs->ws_bytes,
                                       r.comp));
  for (int v = 0; v < 3 && !one_pass; ++v) {
    if (!hs->want[v]) continue;
    // thermosteric holds S at the reference slab, halosteric holds T
    const void* Tv = v == 2 ? hs->dTref : hs->dT[b];
    const void* Sv = v == 1 ? hs->dSref : hs->dS[b];
    const int tb = v == 2, sb = v == 1;
    double* out = hs->dOut[b][v];
    if (!local) {
      ML_HS_RC(ml_steric_global(eos, dtype, Tv, Sv, tb, sb, hs->dV, vdt, dP, nt_block, nz, ncol, out, hs->dWs, hs->ws_bytes,
                                r.comp));
    } else if (first_selfref) {
      // the window that starts at the reference step: the fused self-reference pass (for every variant, so that
      // each step-0 height is exactly zero; it rewrites rho_ref / sums with the same values)
      ML_HS_RC(ml_steric_local_selfref(eos, dtype, Tv, Sv, tb, sb, hs->dV, vdt, dZi, dDepth, dP, hs->coef, nt_block, nz, ncol,
                                       out, (double*)hs->dRho, (double*)hs->dSums, hs->dWs, hs->ws_bytes, r.comp));
    } else {
      ML_HS_RC(ml_steric_local(eos, dtype, Tv, Sv, tb, sb, (const double*)hs->dRho, hs->dV, vdt, dZi, dDepth, dP, hs->coef,
                               nt_block, nz, ncol, out, nullptr, r.comp));
    }
  }
  ML_HS_CUDA(cudaEventRecord(r.freed[b], r.comp));
  // the results of this block go home while the next blocks come in (PCIe carries both directions)
  ML_HS_CUDA(cudaStreamWaitEvent(r.back, r.freed[b], 0));
  const size_t out_bytes = (size_t)nt_block * (local ? (size_t)ncol : 1) * sizeof(double);
  for (int v = 0; v < 3; ++v) {
    if (!hs->want[v]) continue;
    double* dst = user_out[v];
    HostStream::Pending& pend = hs->pending[b][v];
    pend = HostStream::Pending();
    if (is_pageable(dst)) {  // a copy to pageable memory would hold this thread until the block's kernels are done
      void* hb;
      if (r.halloc(kHostOut0 + 3 * b + v, &hb, (size_t)hs->max_steps * (local ? (size_t)ncol : 1) * sizeof(double)) == cudaSuccess) {
        pend.user = dst;
        pend.bounce = (double*)hb;
        pend.bytes = out_bytes;
        dst = (double*)hb;
      } else {
        cudaGetLastError();
      }
    }
    ML_HS_CUDA(cudaMemcpyAsync(dst, hs->dOut[b][v], out_bytes, cudaMemcpyDeviceToHost, r.back));
  }
  ML_HS_CUDA(cudaEventRecord(r.out_done[b], r.back));
  // The caller may reuse the PREVIOUS block's memory once this call returns: its copies were queued in front of
  // this block's, so waiting for them does not stall the copy engine, which already has this block's rows to move.
  if (w >= 1 && hs->release_previous) ML_HS_CUDA(cudaEventSynchronize(r.copied[b ^ 1]));
#undef ML_HS_CUDA
#undef ML_HS_RC
  hs->blocks++;
  hs->steps += nt_block;
  return ML_OK;
}

extern "C" int ml_host_stream_finish(void* stream, double* rho_ref_out, double* sums_out) {
  using namespace ml;
  ML_REQUIRE_PTR(stream);
  HostStream* hs = static_cast<HostStream*>(stream);
  if (hs->owner != std::this_thread::get_id()) return fail(ML_ERR_MODE, "a host stream belongs to the thread that began it");
  Resources& r = *hs->r;
  int rc = ML_OK;
  const size_t lvl = (size_t)hs->nz * (size_t)hs->ncol;
  if (hs->failed) rc = fail(ML_ERR_MODE, "the stream has failed");
  if (rc == ML_OK && rho_ref_out != nullptr && !(hs->want_rho_ref && hs->dRho != nullptr))
    rc = fail(ML_ERR_MODE, "rho_ref_out needs want_rho_ref at ml_host_stream_begin");
  const double t_windows = now_ms();
  cudaError_t e = cudaSuccess;
  if (rc == ML_OK && hs->blocks > 0) {
    if (sums_out && hs->selfref && hs->want_sums) e = cudaMemcpyAsync(sums_out, hs->dSums, 2 * sizeof(double), cudaMemcpyDeviceToHost, r.comp);
    if (e == cudaSuccess && rho_ref_out)
      e = cudaMemcpyAsync(rho_ref_out, hs->dRho, lvl * sizeof(double), cudaMemcpyDeviceToHost, r.comp);
  }
  cudaError_t e2 = cudaStreamSynchronize(r.comp);
  cudaError_t e3 = cudaStreamSynchronize(r.back);
  cudaError_t e4 = cudaStreamSynchronize(r.copy);
  for (cudaError_t x : {e, e2, e3, e4})
    if (rc == ML_OK && x != cudaSuccess) rc = cuda_fail(x, "ml_host_stream_finish");
  if (rc == ML_OK) {
    flush_pending(hs, 0);
    flush_pending(hs, 1);
  }
  r.last_packed_fraction = hs->plan.rows_total ? (double)hs->plan.rows_packed / (double)hs->plan.rows_total : 0.0;
  const double t_end = now_ms();
  r.last_ms[0] = (hs->t_plan > 0.0 ? hs->t_plan : t_windows) - hs->t_begin;
  r.last_ms[1] = t_windows - (hs->t_plan > 0.0 ? hs->t_plan : t_windows);
  r.last_ms[2] = t_end - t_windows;
  r.last_ms[3] = t_end - hs->t_begin;
  r.open_stream = false;
  delete hs;
  return rc;
}

extern "C" int ml_host_stream_abort(void* stream) {
  if (stream == nullptr) return ML_OK;
  HostStream* hs = static_cast<HostStream*>(stream);
  stream_fail(hs, ML_OK);
  hs->r->open_stream = false;
  delete hs;
  return ML_OK;
}

// ---------------------------------------------------------------------------------------------------
// Whole arrays in host memory: begin + one push per window + finish.
// ---------------------------------------------------------------------------------------------------
static int run_windows(void* hs, const void* T, const void* S, size_t step_bytes, int64_t nt, int64_t spw, double* out[3],
                       size_t out_stride) {
  for (int64_t t = 0; t < nt; t += spw) {
    const int64_t n = t + spw <= nt ? spw : nt - t;
    double* o[3];
    for (int v = 0; v < 3; ++v) o[v] = out[v] ? out[v] + (size_t)t * out_stride : nullptr;
    int rc = ml_host_stream_push(hs, (const char*)T + (size_t)t * step_bytes, (const char*)S + (size_t)t * step_bytes, n, o[0],
                                 o[1], o[2]);
    if (rc) {
      ml_host_stream_abort(hs);
      return rc;
    }
  }
  return ML_OK;
}

static int steric_local_host_impl(int eos, int dtype, const void* T, const void* S, const void* v0, const double* z_i,
                                  const double* deptho, const double* p_level, double neg_inv_rhozero, int64_t nt,
                                  int64_t nz, int64_t ncol, int steps_per_window, double* eta, double* eta_thermo,
                                  double* eta_halo, double* rho_ref_out, double* sums_out) {
  using namespace ml;
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(eta);
  if (nt <= 0 || nz <= 0 || ncol <= 0 || steps_per_window < 1)
    return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld window=%d", (long long)nt, (long long)nz,
                (long long)ncol, steps_per_window);
  const int64_t spw = steps_per_window < nt ? steps_per_window : nt;
  const int variants = 1 | (eta_thermo ? 2 : 0) | (eta_halo ? 4 : 0);
  void* hs = nullptr;
  int rc = ml_host_stream_begin(ML_DOMAIN_LOCAL, eos, dtype, variants, v0, dtype, nullptr, nullptr, nullptr, z_i, deptho,
                                p_level, neg_inv_rhozero, nz, ncol, spw, rho_ref_out != nullptr ? 1 : 0, &hs);
  if (rc) return rc;
  static_cast<HostStream*>(hs)->release_previous = false;  // the caller's arrays outlive the call
  double* out[3] = {eta, eta_thermo, eta_halo};
  const size_t step_bytes = (size_t)nz * (size_t)ncol * (size_t)elem_size(dtype);
  if ((rc = run_windows(hs, T, S, step_bytes, nt, spw, out, (size_t)ncol))) return rc;
  return ml_host_stream_finish(hs, rho_ref_out, sums_out);
}

extern "C" int ml_steric_local_host(int eos, int dtype, const void* T, const void* S, const void* v0,
                                    const double* z_i, const double* deptho, const double* p_level,
                                    double neg_inv_rhozero, int64_t nt, int64_t nz, int64_t ncol,
                                    int steps_per_window, double* eta, double* rho_ref_out, double* sums_out) {
  return steric_local_host_impl(eos, dtype, T, S, v0, z_i, deptho, p_level, neg_inv_rhozero, nt, nz, ncol,
                                steps_per_window, eta, nullptr, nullptr, rho_ref_out, sums_out);
}

extern "C" int ml_steric_local_variants_host(int eos, int dtype, const void* T, const void* S, const void* v0,
                                             const double* z_i, const double* deptho, const double* p_level,
                                             double neg_inv_rhozero, int64_t nt, int64_t nz, int64_t ncol,
                                             int steps_per_window, double* eta_steric, double* eta_thermosteric,
                                             double* eta_halosteric, double* rho_ref_out, double* sums_out) {
  return steric_local_host_impl(eos, dtype, T, S, v0, z_i, deptho, p_level, neg_inv_rhozero, nt, nz, ncol,
                                steps_per_window, eta_steric, eta_thermosteric, eta_halosteric, rho_ref_out, sums_out);
}

// The global branch (src/momlevel/steric.py:134-147) on host buffers: per-step masses
// M(t) = sum rho(t) * volcello_ref (derived.py:435-438) with T, S streamed through the same two
// windows; the ln() formula stays with the caller, as for ml_steric_global.
extern "C" int ml_steric_global_host(int eos, int dtype, const void* T, const void* S, const void* v_ref,
                                     const double* p_level, int64_t nt, int64_t nz, int64_t ncol,
                                     int steps_per_window, double* masso) {
  using namespace ml;
  ML_REQUIRE_PTR(T);
  ML_REQUIRE_PTR(S);
  ML_REQUIRE_PTR(masso);
  if (nt <= 0 || nz <= 0 || ncol <= 0 || steps_per_window < 1)
    return fail(ML_ERR_SHAPE, "bad extents nt=%lld nz=%lld ncol=%lld window=%d", (long long)nt, (long long)nz,
                (long long)ncol, steps_per_window);
  const int64_t spw = steps_per_window < nt ? steps_per_window : nt;
  // the masses need the reference VOLUME only, which the caller hands in: no reference-state pass
  void* hs = nullptr;
  int rc = ml_host_stream_begin(ML_DOMAIN_GLOBAL, eos, dtype, 1, v_ref, dtype, nullptr, nullptr, nullptr, nullptr, nullptr,
                                p_level, 0.0, nz, ncol, spw, 0, &hs);
  if (rc) return rc;
  static_cast<HostStream*>(hs)->release_previous = false;
  double* out[3] = {masso, nullptr, nullptr};
  const size_t step_bytes = (size_t)nz * (size_t)ncol * (size_t)elem_size(dtype);
  if ((rc = run_windows(hs, T, S, step_bytes, nt, spw, out, 1))) return rc;
  return ml_host_stream_finish(hs, nullptr, nullptr);
}
