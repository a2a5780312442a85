// Host runtime and C ABI of liblwkzg_b200.so (declared in include/lwkzg.h).
//
// Mirrors the orchestration of /root/reference/src/lib.rs:245-858 -- same
// entry points, argument meaning, order of checks and error mapping (SURVEY
// App. A.11) -- with the arithmetic moved to the CUDA kernels in this
// directory.  The per-call SRS re-hydration of the reference
// (kzgsettings_to_structured_reference_string, src/srs.rs:258-280) becomes a
// device context that is built once per KZGSettings and stays resident in HBM.
//
// There is no CPU compute path in here: the host only parses text, moves bytes
// and launches kernels.
#include <cuda_runtime.h>
#include <fcntl.h>
#include <signal.h>
#include <sys/file.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/lwkzg.h"
#include "kernels.h"
#include "kernels_cells.h"
#include "kernels_setup.h"

namespace {

using namespace lw;

thread_local std::string tl_err;

void set_err(const std::string& s) { tl_err = s; }

#define CU_TRY(expr)                                                                      \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      set_err(std::string(#expr) + ": " + cudaGetErrorString(_e));                        \
      return false;                                                                       \
    }                                                                                     \
  } while (0)

struct Options {
  long window_bits = 16;     // fixed-base window; shrunk automatically to what free HBM allows
  long msm_blocks_per_blob = 0;
  long chunk_blobs = 256;
  long msm_algo = 1;         // 0 = XYZZ accumulation only, 1 = batched-affine accumulation for large batches
  long msm_ba_min_blobs = 5;         // measured (tools/batch_size_sweep.py): with blobs split over up to 8 blocks the batched-affine kernel wins from
                                     // five blobs up (4 blobs: 3.10 vs 2.78 ms, 6: 3.12 vs 3.83, 32: 3.9 vs 10.9, 64: 5.0 vs 12.1)
  long verify_super_blobs = 16384;   // blobs of a batched verification staged on the device at a time (2 GiB)
  long lincomb_points_in_g1 = 0;     // lwkzg_g1_lincomb: the caller vouches that every point is in the r-torsion (GLV split allowed)
  long verify_overlap_decode = 1;    // batched verification: blob hashes start beside the point decompression (possible since the decompression
                                     // kernels carry the hash kernels' shared-memory carve-out) instead of behind it
  long cache_config = 0;             // device-wide cudaDeviceSetCacheConfig hint applied when a context is built: 0 = leave alone, 1 = prefer shared,
                                     // 3 = prefer equal (see DESIGN 3.5: kernels with different shared-memory carve-outs do not share an SM)
  long verify_split_subgroup = 0;    // 1 = batched verification runs the r-torsion tests of the points beside the first blob hashes instead of in front
                                     // of them.  Measured and not kept as the default: device-resident 20.8 -> 20.8 ms, from pinned memory 21.2 -> 25 ms
                                     // (blob-hash kernels that run beside the thread-per-point kernels take several times longer)
  long verify_streams = 6;           // compute streams a batched verification spreads its chunks over (1..8).  Measured on B200, 4096 blobs:
                                     // 8 streams 25.5-27.8 ms device-resident (a chunk's hash kernel takes 13 ms instead of 2.5 now and then), 4-6
                                     // streams 21.0 ms, 3 streams 24.4 ms; from pinned memory 20.9-21.4 ms either way
  long share_table = 0;              // 1 = one digit table per (SRS, window, device) for every settings object and PROCESS that loads it
  long cell_window_bits = 13;        // window of the FK20 digit table (8192 points; 13 bits = 29 GiB), shrunk to what free HBM allows
  long cell_chunk_blobs = 888;       // blobs per pass of a cell batch: 2 x 444 = exactly two waves of the batched-affine MSM kernel, and 28 x 32 blobs
                                     // x 64 butterflies = 1792 warps per G1 FFT stage, one wave of the 16 x 148 warp slots the stage kernel gets
  long mode = 0;  // 0 = MODE_REFERENCE (what lambdaworks_kzg computes), 1 = MODE_CKZG_LE (what the YAML vectors encode),
                  // 2 = MODE_DENEB (the mainnet wire format: big-endian canonical scalars over the Lagrange SRS)
  Options() {
    if (const char* e = getenv("LWKZG_MODE")) mode = std::min(std::max(atol(e), 0L), 2L);
    if (const char* e = getenv("LWKZG_WINDOW_BITS")) window_bits = atol(e);
    if (const char* e = getenv("LWKZG_CHUNK_BLOBS")) chunk_blobs = std::min(std::max(atol(e), 1L), 1L << 20);
    if (const char* e = getenv("LWKZG_MSM_BLOCKS_PER_BLOB")) msm_blocks_per_blob = atol(e);
    if (const char* e = getenv("LWKZG_MSM_ALGO")) msm_algo = atol(e);
    if (const char* e = getenv("LWKZG_MSM_BA_MIN_BLOBS")) msm_ba_min_blobs = atol(e);
    if (const char* e = getenv("LWKZG_SHARE_TABLE")) share_table = atol(e) != 0;
    if (const char* e = getenv("LWKZG_CACHE_CONFIG")) cache_config = atol(e);
  }
};
Options& opts() {
  static Options o;
  return o;
}
std::mutex g_mu;  // guards the options

// Device buffer that grows on demand and is freed with its owner.  The owner synchronises the streams that use it first.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() {
    if (p) cudaFree(p);
  }
  bool ensure(size_t bytes) {
    if (bytes <= cap) return true;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    CU_TRY(cudaMalloc(&p, bytes));
    cap = bytes;
    return true;
  }
};

// Every device buffer of a workspace with the bytes one request needs, listed once per workspace: both "reserve" and
// "already fits" are answered from that list.
using BufList = std::vector<std::pair<DevBuf*, size_t>>;
bool reserve(const BufList& bufs) {
  for (const auto& b : bufs)
    if (!b.first->ensure(b.second)) return false;
  return true;
}
bool fits(const BufList& bufs) {
  for (const auto& b : bufs)
    if (b.first->cap < b.second) return false;
  return true;
}

// ------------------------------------------------------------------ pageable host buffers
// A c-kzg caller passes ordinary (pageable) memory.  cudaMemcpyAsync from pageable memory is a synchronous, single-
// threaded staged copy inside the driver (~11 GB/s measured: 512 MiB of blobs in 46 ms against 9.8 ms from pinned
// memory), so batches from pageable memory are staged here instead: a small pool of host threads copies each chunk
// into a ring of pinned buffers (aggregate host memcpy bandwidth), and the H2D copy from the ring is a real DMA that
// overlaps the staging of the next chunk.  (Byte moving only -- no arithmetic happens on the host.)
class HostStager {
 public:
  static HostStager& get() {
    static HostStager s;
    return s;
  }
  // dst[0, bytes) = src[0, bytes), split over the pool; returns when every slice has landed
  void copy(void* dst, const void* src, size_t bytes) {
    if (bytes < (size_t(1) << 20) || workers_.empty()) { memcpy(dst, src, bytes); return; }
    std::unique_lock<std::mutex> call(call_mu_);   // one parallel copy at a time
    const size_t parts = workers_.size() + 1;
    const size_t slice = ((bytes + parts - 1) / parts + 4095) & ~size_t(4095);
    {
      std::lock_guard<std::mutex> lk(mu_);
      dst_ = (uint8_t*)dst; src_ = (const uint8_t*)src; bytes_ = bytes; slice_ = slice;
      pending_ = (int)workers_.size();
      gen_++;
    }
    cv_.notify_all();
    memcpy(dst, src, std::min(slice, bytes));   // slice 0 on the calling thread
    std::unique_lock<std::mutex> lk(mu_);
    done_cv_.wait(lk, [&] { return pending_ == 0; });
  }
  ~HostStager() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      stop_ = true;
    }
    cv_.notify_all();
    for (auto& t : workers_) t.join();
  }

 private:
  HostStager() {
    unsigned hw = std::thread::hardware_concurrency();
    int n = (int)std::min(7u, hw > 2 ? hw / 2 - 1 : 0u);
    if (const char* e = getenv("LWKZG_STAGE_THREADS")) n = std::max(0, atoi(e) - 1);
    for (int i = 0; i < n; i++) workers_.emplace_back([this, i] { run(i + 1); });
  }
  void run(int idx) {
    uint64_t seen = 0;
    for (;;) {
      uint8_t* d; const uint8_t* s; size_t bytes, slice;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return stop_ || gen_ != seen; });
        if (stop_) return;
        seen = gen_;
        d = dst_; s = src_; bytes = bytes_; slice = slice_;
      }
      const size_t lo = std::min(bytes, slice * (size_t)idx), hi = std::min(bytes, lo + slice);
      if (hi > lo) memcpy(d + lo, s + lo, hi - lo);
      {
        std::lock_guard<std::mutex> lk(mu_);
        if (--pending_ == 0) done_cv_.notify_all();
      }
    }
  }
  std::vector<std::thread> workers_;
  std::mutex mu_, call_mu_;
  std::condition_variable cv_, done_cv_;
  uint8_t* dst_ = nullptr;
  const uint8_t* src_ = nullptr;
  size_t bytes_ = 0, slice_ = 0;
  int pending_ = 0;
  uint64_t gen_ = 0;
  bool stop_ = false;
};

bool is_pageable_host(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
  return a.type == cudaMemoryTypeUnregistered;
}

constexpr int RING_SLOTS = 3;
struct PinnedRing {   // per context: RING_SLOTS pinned buffers of one pipeline chunk each
  void* buf[RING_SLOTS] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev[RING_SLOTS] = {nullptr, nullptr, nullptr};
  bool used[RING_SLOTS] = {false, false, false};
  size_t cap = 0;
  bool ensure(size_t bytes) {
    if (bytes <= cap) return true;
    release();
    for (int i = 0; i < RING_SLOTS; i++) {
      CU_TRY(cudaMallocHost(&buf[i], bytes));
      CU_TRY(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
    }
    cap = bytes;
    return true;
  }
  void release() {
    for (int i = 0; i < RING_SLOTS; i++) {
      if (ev[i]) { cudaEventSynchronize(ev[i]); cudaEventDestroy(ev[i]); }
      if (buf[i]) cudaFreeHost(buf[i]);
      buf[i] = nullptr; ev[i] = nullptr; used[i] = false;
    }
    cap = 0;
  }
  // stage src into slot (seq % RING_SLOTS) -- after the copy that last used the slot has finished -- and enqueue the
  // H2D copy from there on `st`
  bool h2d(void* d_dst, const void* src, size_t bytes, uint64_t seq, cudaStream_t st) {
    const int k = (int)(seq % RING_SLOTS);
    if (used[k]) CU_TRY(cudaEventSynchronize(ev[k]));
    HostStager::get().copy(buf[k], src, bytes);
    CU_TRY(cudaMemcpyAsync(d_dst, buf[k], bytes, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaEventRecord(ev[k], st));
    used[k] = true;
    return true;
  }
};

constexpr uint64_t CTX_MAGIC = 0x4c574b5a47423230ull;  // "LWKZGB20"
constexpr int NSLOT = 4;

struct Slot {
  cudaStream_t st = nullptr, aux = nullptr;
  cudaEvent_t ev_in = nullptr, ev_aux = nullptr, ev_done = nullptr, ev_fork = nullptr;
  DevBuf ba_scratch;  // accumulators + prefix products of the batched-affine MSM kernel
  DevBuf blobs, q, partials, states, z, y, ybe, c48, cin48, p48, caff, status, status2, zbe;
};

struct CellCtx;                       // PeerDAS state (cells_host.inl), built on the first cell call
void destroy_cell_ctx(CellCtx* cc);

struct Ctx {
  FFTSettings fs_prefix;  // MUST be first: KZGSettings.fs points here
  uint64_t magic;
  int device;
  int c, nwin;
  bool srs_valid;     // every g1 value on the curve (else every call errors, like the reference's re-hydration)
  bool srs_in_g1;     // every g1 value in the r-torsion
  bool g2_valid;      // g2[0], g2[1] on the twist
  int mode;           // semantic mode captured when the context was built
  bool lagrange() const { return mode != 0; }   // evaluation-form blobs over a Lagrange SRS, c-kzg error codes
  bool be_wire() const { return mode == 2; }    // MODE_DENEB: big-endian field elements and hash headers
  void* d_roots;      // Lagrange modes: bit-reversed 4096th roots of unity (Montgomery)
  void* d_gen;        // Lagrange modes: the G1 generator (c-kzg verifies against G, not against g1_values[0] = L_0)
  void* d_srs;        // 4096 affine Montgomery
  void* d_mono = nullptr;     // the MONOMIAL SRS [tau^i]G (= d_srs in MODE_REFERENCE; kept by the loader in the Lagrange modes): FK20, cell verification
  bool mono_owned = false;
  CellCtx* cell = nullptr;
  void* d_table;      // fixed-base digit table
  int table_share = 0;        // 0 = private, 1 = built here and published ("share_table"), 2 = attached to another process's, 3 = another settings object's
  uint64_t table_key = 0;
  void* d_prep0;      // prepared g2[0] / g2[1] line coefficients
  void* d_prep1;
  Slot slot[NSLOT];
  // batched-verification workspace (sized for the largest batch seen)
  DevBuf vb_cin, vb_pin, vb_caff, vb_piaff, vb_c48r, vb_p48r, vb_z, vb_y, vb_tuples, vb_status, vb_r, vb_partial, vb_scratch, vb_ok, vb_zy_in;
  size_t vb_n = 0;  // items currently held by the workspace (phase1 -> phase2)
  // the batch challenge r is one sequential SHA-256 over all tuples: it is absorbed chunk by chunk on its own
  // stream while later chunks are still being copied and evaluated
  cudaStream_t hash_st = nullptr, copy_st = nullptr;
  cudaEvent_t ev_hash = nullptr;
  std::vector<cudaEvent_t> ev_pool;   // per chunk: blob copy landed / tuples written
  DevBuf vb_hstate, vb_blobs, vb_states, vb_status2, vb_sub;
  // pinned host staging for batch results: a D2H copy into pageable memory would block the host
  // until the chunk's kernels finish and serialise the two pipeline slots
  void* h_stage = nullptr;
  size_t h_stage_cap = 0;
  PinnedRing ring;            // staging of pageable caller buffers (blobs)
  uint64_t ring_seq = 0;
  std::mutex mu;
  // lwkzg_set_devices: contexts of the same settings on the other GPUs (built on the first multi-device call; owned
  // by this, the primary, context) and the host arrays they were built from
  const g1_t* g1_host = nullptr;
  const g2_t* g2_host = nullptr;
  std::vector<Ctx*> replicas;
  std::mutex replicas_mu;
};

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

// ------------------------------------------------------------------ g1/g2 value layout
// src/srs.rs:131-213: canonical integers, u64 limbs most-significant first.
void canon_to_blst_fp(blst_fp* out, const uint32_t* le12) {
  for (int k = 0; k < 6; k++) out->l[k] = ((uint64_t)le12[11 - 2 * k] << 32) | (uint64_t)le12[10 - 2 * k];
}
void blst_fp_to_canon(uint32_t* le12, const blst_fp* in) {
  for (int k = 0; k < 6; k++) {
    le12[11 - 2 * k] = (uint32_t)(in->l[k] >> 32);
    le12[10 - 2 * k] = (uint32_t)in->l[k];
  }
}

// ------------------------------------------------------------------ shared digit tables ("share_table")
// SURVEY 8 f2 asks for a table cache.  On this hardware the table is REBUILT faster than any disk could deliver it
// (100 GiB in 3.8 s = 26 GiB/s), so what is worth caching is the copy already in HBM: with "share_table" a table is
// keyed by (SRS contents, window, device), shared by every settings object of a process (reference count) and by
// every PROCESS on the same GPU through a CUDA IPC handle published in /dev/shm -- N verifier or fuzzer processes
// (the reference's fuzz harness runs `-workers` processes, fuzz/Makefile:53-58) hold ONE table instead of N and attach
// in milliseconds.  The first loader owns the memory and must outlive the others (CUDA IPC rule); a stale file left
// by a dead owner is ignored and replaced.
uint64_t fnv1a(const void* p, size_t n, uint64_t h = 1469598103934665603ull);
struct SharedTable { void* p; int refs; bool ipc_import; bool published; };
std::mutex g_table_mu;
std::map<uint64_t, SharedTable>& table_registry() {
  static std::map<uint64_t, SharedTable> m;
  return m;
}
struct TableFile {
  uint64_t magic, key, entries;
  int32_t pid, c;
  cudaIpcMemHandle_t handle;
};
constexpr uint64_t TABLE_FILE_MAGIC = 0x4c574b5a5442314cull;
std::string table_path(uint64_t key) {
  char buf[96];
  snprintf(buf, sizeof(buf), "/dev/shm/lwkzg_b200_%016llx.tbl", (unsigned long long)key);
  return buf;
}
void release_table(Ctx* c) {
  if (c->table_share == 0) { cudaFree(c->d_table); c->d_table = nullptr; return; }
  std::lock_guard<std::mutex> lk(g_table_mu);
  auto it = table_registry().find(c->table_key);
  if (it != table_registry().end() && --it->second.refs == 0) {
    if (it->second.ipc_import) cudaIpcCloseMemHandle(it->second.p);
    else cudaFree(it->second.p);
    if (it->second.published) unlink(table_path(c->table_key).c_str());
    table_registry().erase(it);
  }
  c->d_table = nullptr;
}

// ------------------------------------------------------------------ context
void destroy_ctx(Ctx* c) {
  if (!c) return;
  for (Ctx* r : c->replicas) destroy_ctx(r);
  c->replicas.clear();
  DeviceGuard g(c->device);
  for (auto& s : c->slot) {
    if (s.st) cudaStreamSynchronize(s.st);
    if (s.aux) cudaStreamSynchronize(s.aux);
    if (s.ev_in) cudaEventDestroy(s.ev_in);
    if (s.ev_aux) cudaEventDestroy(s.ev_aux);
    if (s.ev_done) cudaEventDestroy(s.ev_done);
    if (s.ev_fork) cudaEventDestroy(s.ev_fork);
    if (s.st) cudaStreamDestroy(s.st);
    if (s.aux) cudaStreamDestroy(s.aux);
  }
  if (c->hash_st) cudaStreamSynchronize(c->hash_st);
  if (c->ev_hash) cudaEventDestroy(c->ev_hash);
  for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
  if (c->copy_st) { cudaStreamSynchronize(c->copy_st); cudaStreamDestroy(c->copy_st); }
  if (c->hash_st) cudaStreamDestroy(c->hash_st);
  if (c->cell) destroy_cell_ctx(c->cell);
  c->cell = nullptr;
  if (c->d_mono && c->mono_owned) cudaFree(c->d_mono);
  if (c->d_srs) cudaFree(c->d_srs);
  if (c->d_table) release_table(c);
  if (c->d_prep0) cudaFree(c->d_prep0);
  if (c->d_prep1) cudaFree(c->d_prep1);
  if (c->d_roots) cudaFree(c->d_roots);
  if (c->d_gen) cudaFree(c->d_gen);
  if (c->h_stage) cudaFreeHost(c->h_stage);
  c->ring.release();
  c->magic = 0;
  delete c;
}

bool build_ctx_inner(Ctx* c, const g1_t* g1, const g2_t* g2, int mode, long window_override) {
  CU_TRY(cudaGetDevice(&c->device));
  {
    long cfg;
    {
      std::lock_guard<std::mutex> lk(g_mu);
      cfg = opts().cache_config;
    }
    if (cfg == 1) cudaDeviceSetCacheConfig(cudaFuncCachePreferShared);
    else if (cfg == 2) cudaDeviceSetCacheConfig(cudaFuncCachePreferL1);
    else if (cfg == 3) cudaDeviceSetCacheConfig(cudaFuncCachePreferEqual);
  }
  int lo = 0, hi = 0;
  CU_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  for (auto& s : c->slot) {
    CU_TRY(cudaStreamCreateWithPriority(&s.st, cudaStreamNonBlocking, lo));
    CU_TRY(cudaStreamCreateWithPriority(&s.aux, cudaStreamNonBlocking, hi));  // SHA midstate: latency critical
    CU_TRY(cudaEventCreateWithFlags(&s.ev_in, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&s.ev_aux, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&s.ev_fork, cudaEventDisableTiming));
  }
  CU_TRY(cudaStreamCreateWithPriority(&c->hash_st, cudaStreamNonBlocking, hi));
  CU_TRY(cudaStreamCreateWithPriority(&c->copy_st, cudaStreamNonBlocking, hi));
  CU_TRY(cudaEventCreateWithFlags(&c->ev_hash, cudaEventDisableTiming));
  cudaStream_t st = c->slot[0].st;

  // ---- SRS import
  std::vector<uint32_t> canon((size_t)N_POINTS * 24);
  for (int i = 0; i < N_POINTS; i++) {
    blst_fp_to_canon(&canon[(size_t)i * 24], &g1[i].x);
    blst_fp_to_canon(&canon[(size_t)i * 24 + 12], &g1[i].y);
  }
  void* d_canon = nullptr;
  int* d_flags = nullptr;
  CU_TRY(cudaMalloc(&d_canon, canon.size() * 4));
  CU_TRY(cudaMalloc(&d_flags, 2 * N_POINTS * sizeof(int)));
  CU_TRY(cudaMalloc(&c->d_srs, (size_t)N_POINTS * AFFINE_BYTES));
  CU_TRY(cudaMemcpyAsync(d_canon, canon.data(), canon.size() * 4, cudaMemcpyHostToDevice, st));
  launch_srs_import(c->d_srs, d_canon, d_flags, d_flags + N_POINTS, N_POINTS, st);
  std::vector<int> flags(2 * N_POINTS);
  CU_TRY(cudaMemcpyAsync(flags.data(), d_flags, flags.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
  CU_TRY(cudaStreamSynchronize(st));
  cudaFree(d_canon);
  cudaFree(d_flags);
  c->srs_valid = true;
  c->srs_in_g1 = true;
  for (int i = 0; i < N_POINTS; i++) {
    if (flags[i]) c->srs_valid = false;
    if (flags[N_POINTS + i]) c->srs_in_g1 = false;
  }

  // ---- G2: g2[0], g2[1] -> prepared Miller-loop lines
  c->g2_valid = false;
  {
    std::vector<uint32_t> g2canon((size_t)TRUSTED_SETUP_NUM_G2_POINTS * 48);   // per call: contexts are built concurrently
    for (int k = 0; k < TRUSTED_SETUP_NUM_G2_POINTS; k++) {
      blst_fp_to_canon(&g2canon[(size_t)k * 48], &g2[k].x.fp[0]);
      blst_fp_to_canon(&g2canon[(size_t)k * 48 + 12], &g2[k].x.fp[1]);
      blst_fp_to_canon(&g2canon[(size_t)k * 48 + 24], &g2[k].y.fp[0]);
      blst_fp_to_canon(&g2canon[(size_t)k * 48 + 36], &g2[k].y.fp[1]);
    }
    void* d_g2 = nullptr;
    int* d_bad = nullptr;
    const size_t g2_bytes = g2canon.size() * sizeof(uint32_t);
    CU_TRY(cudaMalloc(&d_g2, g2_bytes));
    CU_TRY(cudaMalloc(&d_bad, (2 + TRUSTED_SETUP_NUM_G2_POINTS) * sizeof(int)));
    CU_TRY(cudaMalloc(&c->d_prep0, g2_prepared_bytes()));
    CU_TRY(cudaMalloc(&c->d_prep1, g2_prepared_bytes()));
    CU_TRY(cudaMemcpyAsync(d_g2, g2canon.data(), g2_bytes, cudaMemcpyHostToDevice, st));
    launch_g2_prepare(c->d_prep0, d_bad, d_g2, st);
    launch_g2_prepare(c->d_prep1, d_bad + 1, (const uint8_t*)d_g2 + 48 * 4, st);
    launch_g2_check(d_bad + 2, d_g2, TRUSTED_SETUP_NUM_G2_POINTS, st);
    int bad[2 + TRUSTED_SETUP_NUM_G2_POINTS];
    for (int& b : bad) b = 1;
    CU_TRY(cudaMemcpyAsync(bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    cudaFree(d_g2);
    cudaFree(d_bad);
    c->g2_valid = !bad[0] && !bad[1];
    // the reference re-hydrates all 65 G2 values on every call and fails if any
    // is off the twist (src/srs.rs:258-280)
    for (int k = 0; k < TRUSTED_SETUP_NUM_G2_POINTS; k++)
      if (bad[2 + k]) c->srs_valid = false;
  }

  c->mode = mode;
  if (mode == 0) c->d_mono = c->d_srs;
  if (mode != 0) {
    // allocated before the early return below: every Lagrange-mode kernel may assume they exist
    CU_TRY(cudaMalloc(&c->d_roots, (size_t)N_POINTS * 32));
    launch_le_roots(c->d_roots, st);
    CU_TRY(cudaMalloc(&c->d_gen, AFFINE_BYTES));
    launch_write_generator(c->d_gen, st);
  }
  if (!c->srs_valid) {  // usable only to report C_KZG_ERROR, like the reference
    CU_TRY(cudaStreamSynchronize(st));
    return true;
  }

  // ---- fixed-base digit table; shrink the window if HBM is short
  long want_c;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    want_c = window_override > 0 ? window_override : opts().window_bits;
  }
  if (want_c < 4) want_c = 4;
  if (want_c > 16) want_c = 16;
  size_t free_b = 0, total_b = 0;
  CU_TRY(cudaMemGetInfo(&free_b, &total_b));
  bool share;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    share = opts().share_table != 0 && window_override == 0;
  }
  uint64_t base_key = 0;
  int lock_fd = -1;
  if (share) {
    // key: SRS contents (as imported: the Lagrange points in the Lagrange modes), device identity
    char bus[32] = {0};
    cudaDeviceGetPCIBusId(bus, sizeof(bus), c->device);
    base_key = fnv1a(g1, sizeof(g1_t) * N_POINTS);
    base_key = fnv1a(bus, sizeof(bus), base_key);
    // one loader at a time per machine: a second process waits for the first one's build and then attaches
    lock_fd = open("/dev/shm/lwkzg_b200.lock", O_CREAT | O_RDWR, 0600);
    if (lock_fd >= 0) flock(lock_fd, LOCK_EX);
  }
  auto unlock = [&]() { if (lock_fd >= 0) { flock(lock_fd, LOCK_UN); close(lock_fd); lock_fd = -1; } };
  if (share) {
    std::lock_guard<std::mutex> lk(g_table_mu);
    for (int cb = (int)want_c; cb >= 4 && !c->d_table; cb--) {
      const uint64_t key = base_key * 31 + (uint64_t)cb;
      auto it = table_registry().find(key);
      if (it != table_registry().end()) {   // another settings object of this process
        it->second.refs++;
        c->d_table = it->second.p;
        c->table_share = 3;
        c->table_key = key;
        c->c = cb;
        break;
      }
      TableFile tf;
      FILE* f = fopen(table_path(key).c_str(), "rb");
      if (!f) continue;
      const bool got = fread(&tf, sizeof(tf), 1, f) == 1;
      fclose(f);
      if (!got || tf.magic != TABLE_FILE_MAGIC || tf.key != key || tf.c != cb || tf.entries != table_entries(cb, N_POINTS)) continue;
      if (tf.pid == (int32_t)getpid() || (kill(tf.pid, 0) != 0 && errno == ESRCH)) continue;   // ours but unregistered, or a dead owner
      void* p = nullptr;
      if (cudaIpcOpenMemHandle(&p, tf.handle, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); continue; }
      table_registry()[key] = SharedTable{p, 1, true, false};
      c->d_table = p;
      c->table_share = 2;
      c->table_key = key;
      c->c = cb;
    }
  }
  if (c->d_table) {
    c->nwin = table_num_windows(c->c);
    unlock();
    CU_TRY(cudaStreamSynchronize(st));
    return true;
  }
  int cbits = (int)want_c;
  for (;; cbits--) {
    const size_t need = (size_t)table_entries(cbits, N_POINTS) * AFFINE_BYTES;
    if (need + (size_t(8) << 30) <= free_b || cbits <= 4) break;   // keep room for the batch slots and the verify workspace
  }
  c->c = cbits;
  c->nwin = table_num_windows(cbits);
  const size_t entries = (size_t)table_entries(cbits, N_POINTS);
  if (entries >= (size_t(1) << 31)) { unlock(); set_err("table index does not fit 31 bits"); return false; }   // entry | sign << 31 (msm.cu)
  bool built = [&]() -> bool {
    CU_TRY(cudaMalloc(&c->d_table, entries * AFFINE_BYTES));
    void* d_bases = nullptr;
    CU_TRY(cudaMalloc(&d_bases, (size_t)c->nwin * N_POINTS * AFFINE_BYTES));
    launch_table_bases(d_bases, c->d_srs, c->c, c->nwin, N_POINTS, st);
    launch_table_fill(c->d_table, d_bases, c->c, c->nwin, N_POINTS, table_top_count(c->c), st);
    CU_TRY(cudaStreamSynchronize(st));
    CU_TRY(cudaGetLastError());
    cudaFree(d_bases);
    return true;
  }();
  if (built && share) {
    std::lock_guard<std::mutex> lk(g_table_mu);
    const uint64_t key = base_key * 31 + (uint64_t)cbits;
    TableFile tf;
    memset(&tf, 0, sizeof(tf));
    tf.magic = TABLE_FILE_MAGIC;
    tf.key = key;
    tf.entries = entries;
    tf.pid = (int32_t)getpid();
    tf.c = cbits;
    bool published = false;
    if (cudaIpcGetMemHandle(&tf.handle, c->d_table) == cudaSuccess) {
      const std::string path = table_path(key), tmp = path + ".tmp";
      FILE* f = fopen(tmp.c_str(), "wb");
      if (f) {
        published = fwrite(&tf, sizeof(tf), 1, f) == 1;
        fclose(f);
        published = published && rename(tmp.c_str(), path.c_str()) == 0;
      }
    } else {
      cudaGetLastError();
    }
    table_registry()[key] = SharedTable{c->d_table, 1, false, published};
    c->table_share = 1;
    c->table_key = key;
  }
  unlock();
  return built;
}

long current_mode() {
  std::lock_guard<std::mutex> lk(g_mu);
  return opts().mode;
}

Ctx* build_ctx(const g1_t* g1, const g2_t* g2, int mode = -1, long window_override = 0) {
  if (mode < 0) mode = (int)current_mode();
  Ctx* c = new Ctx();
  memset(&c->fs_prefix, 0, sizeof(c->fs_prefix));
  c->magic = CTX_MAGIC;
  c->d_srs = c->d_table = c->d_prep0 = c->d_prep1 = c->d_roots = c->d_gen = nullptr;
  c->mode = mode;
  c->c = c->nwin = 0;
  c->srs_valid = c->srs_in_g1 = c->g2_valid = false;
  c->g1_host = g1;
  c->g2_host = g2;
  if (!build_ctx_inner(c, g1, g2, mode, window_override)) {
    std::string e = tl_err;
    destroy_ctx(c);
    set_err(e);
    return nullptr;
  }
  return c;
}

// lazily created contexts for hand-assembled KZGSettings (fs == NULL)
struct LazyKey {
  const void* g1;
  const void* g2;
  uint64_t hash;
  bool operator<(const LazyKey& o) const {
    if (g1 != o.g1) return g1 < o.g1;
    if (g2 != o.g2) return g2 < o.g2;
    return hash < o.hash;
  }
};
std::map<LazyKey, Ctx*>& lazy_map() {
  static std::map<LazyKey, Ctx*> m;
  return m;
}
uint64_t fnv1a(const void* p, size_t n, uint64_t h) {
  const uint64_t* w = (const uint64_t*)p;  // all inputs are multiples of 8 bytes
  for (size_t i = 0; i < n / 8; i++) {
    h ^= w[i];
    h *= 1099511628211ull;
  }
  return h;
}

std::mutex g_lazy_mu;  // guards the lazy-context cache across lookup, build and insert (never taken while holding g_mu)

// Contexts are destroyed only with their own lock held, so a call that is still running on one finishes first.
// (Calling into settings that are being freed concurrently is a caller error here as it is in c-kzg.)
void destroy_ctx_locked(Ctx* c) {
  if (!c) return;
  { std::lock_guard<std::mutex> lk(c->mu); }
  destroy_ctx(c);
}

Ctx* ctx_of(const KZGSettings* s) {
  if (!s || !s->g1_values || !s->g2_values) {
    set_err("null KZGSettings");
    return nullptr;
  }
  if (s->fs) {
    Ctx* c = reinterpret_cast<Ctx*>(s->fs);
    if (c->magic == CTX_MAGIC) return c;
  }
  LazyKey key{s->g1_values, s->g2_values, 0};
  key.hash = fnv1a(s->g1_values, sizeof(g1_t) * N_POINTS);
  key.hash = fnv1a(s->g2_values, sizeof(g2_t) * 2, key.hash);
  // the lock is held while the context is built: a second thread making its first call on the same settings
  // waits here and then finds the finished context instead of building (and leaking) its own
  std::lock_guard<std::mutex> lk(g_lazy_mu);
  auto it = lazy_map().find(key);
  if (it != lazy_map().end()) return it->second;
  // drop stale contexts registered for the same pointers (the caller rewrote the arrays)
  for (auto j = lazy_map().begin(); j != lazy_map().end();) {
    if (j->first.g1 == key.g1 && j->first.g2 == key.g2) {
      destroy_ctx_locked(j->second);
      j = lazy_map().erase(j);
    } else {
      ++j;
    }
  }
  Ctx* c = build_ctx(s->g1_values, s->g2_values);
  if (c) lazy_map()[key] = c;
  return c;
}

// ------------------------------------------------------------------ pipeline
enum class Mode { Commit, CommitProve, BlobProof, PointProof };

// The fixed-base MSM of one chunk: batched-affine accumulation (one block per blob) when the batch is
// large enough to fill the GPU that way, XYZZ accumulation (window-split, many blocks per blob) for
// latency-bound small calls.
bool use_batch_affine(int n) {
  std::lock_guard<std::mutex> lk(g_mu);
  return opts().msm_algo == 1 && n >= opts().msm_ba_min_blobs;
}

// Size of the pipeline chunk that starts at blob `off` of an n-blob call.  Uniform: tapered and mixed plans
// (384/256/192/192, 512/256/128/128, ...) were measured on B200 and make no difference -- a step is bound by
// the total block work of its MSMs, not by the order they are issued in.
size_t chunk_at(size_t off, size_t n, size_t chunk) { return std::min(chunk, n - off); }

// blocks resident at once for the batched-affine kernel (3 per SM)
int ba_block_slots() {
  static int slots[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 444;
  if (!slots[dev]) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    slots[dev] = 3 * sms;
  }
  return slots[dev];
}

int auto_bpb(int n) {
  if (use_batch_affine(n)) {
    // a batch that would leave block slots empty is split further: 2, 4 or 8 blocks per blob, each taking a share
    // of every thread's points (a block's fold of its 64 accumulators per thread is the price: not beyond 8)
    int split = 1;
    while (split < 8 && n * split * 2 <= ba_block_slots()) split *= 2;
    return split;
  }
  long o;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    o = opts().msm_blocks_per_blob;
  }
  if (o > 0) return (int)o;
  int target = (1024 + n - 1) / n;  // measured best on B200: 2 blocks per blob at 512-blob chunks
  int b = 1;
  while (b < target) b <<= 1;
  return std::min(b, 128);
}

void run_msm(Slot& s, const Ctx* c, const void* d_scalars, bool be_input, int n, int bpb, cudaStream_t st);

// the buffers of a pipeline slot for a chunk of n blobs split bpb ways (need_blobs: the blobs are copied in)
BufList slot_buffers(Slot& s, int n, int bpb, bool need_blobs) {
  const size_t m = (size_t)n;
  BufList bufs;
  if (use_batch_affine(n)) bufs.push_back({&s.ba_scratch, msm_ba_scratch_bytes(n * bpb)});
  if (need_blobs) bufs.push_back({&s.blobs, m * BLOB_BYTES});
  bufs.insert(bufs.end(), {{&s.q, m * BLOB_BYTES}, {&s.partials, m * bpb * XYZZ_BYTES}, {&s.states, m * 32}, {&s.z, m * 32}, {&s.y, m * 32},
                           {&s.ybe, m * 32}, {&s.c48, m * 48}, {&s.cin48, m * 48}, {&s.p48, m * 48}, {&s.caff, m * AFFINE_BYTES},
                           {&s.status, m * sizeof(int)}, {&s.status2, m * sizeof(int)}, {&s.zbe, m * 32}});
  return bufs;
}

void run_msm(Slot& s, const Ctx* c, const void* d_scalars, bool be_input, int n, int bpb, cudaStream_t st) {
  if (bpb <= 8 && use_batch_affine(n) && s.ba_scratch.cap >= msm_ba_scratch_bytes(n * bpb))
    launch_msm_gather_ba(s.partials.p, c->d_table, c->c, d_scalars, be_input, n, s.ba_scratch.p, st, bpb);
  else
    launch_msm_gather(s.partials.p, c->d_table, c->c, d_scalars, be_input, n, bpb, st);
}

// Enqueue one chunk on slot.st (+ slot.aux for the SHA midstate).  All pointers
// are device pointers.  Outputs: d_c48 (Commit/CommitProve), d_p48 (all but
// Commit), d_ybe (PointProof), d_status (BlobProof: decode status of the given
// commitments; else zero-filled).
bool enqueue_chunk(Ctx* c, Slot& s, Mode mode, const void* d_blobs, int n, void* d_c48, void* d_p48, void* d_ybe, int* d_status,
                   const void* d_commit_in48, const void* d_z_in_be) {
  const int bpb = auto_bpb(n);
  cudaStream_t st = s.st;
  const bool le = c->lagrange();
  if (le) {
    // MODE_CKZG_LE (SURVEY App. B): canonical little-endian scalars = the limbs as they lie in memory,
    // Lagrange table, barycentric evaluation, evaluation-form quotient, BADARGS for invalid input.
    // MODE_DENEB: the same over big-endian scalars (be) with the final spec's hash layout
    const bool be = c->be_wire();
    int* stt = d_status ? d_status : (int*)s.status.p;
    CU_TRY(cudaMemsetAsync(stt, 0, (size_t)n * sizeof(int), st));
    launch_le_blob_check(stt, d_blobs, n, st, be);
    if (mode == Mode::Commit) {
      run_msm(s, c, d_blobs, be, n, bpb, st);
      launch_msm_finalize(d_c48, nullptr, s.partials.p, bpb, n, st);
      return true;
    }
    const void* commit_for_hash = nullptr;
    if (mode == Mode::CommitProve || mode == Mode::BlobProof) {
      CU_TRY(cudaEventRecord(s.ev_fork, st));
      CU_TRY(cudaStreamWaitEvent(s.aux, s.ev_fork, 0));
      launch_challenge_midstate(s.states.p, d_blobs, n, s.aux, mode == Mode::BlobProof, be);
      CU_TRY(cudaEventRecord(s.ev_aux, s.aux));
    }
    if (mode == Mode::CommitProve) {
      run_msm(s, c, d_blobs, be, n, bpb, st);
      launch_msm_finalize(d_c48, nullptr, s.partials.p, bpb, n, st);
      commit_for_hash = d_c48;
    } else if (mode == Mode::BlobProof) {
      launch_g1_decompress(nullptr, nullptr, (int*)s.status2.p, d_commit_in48, n, st, true);
      launch_status_or(stt, (const int*)s.status2.p, n, st);
      commit_for_hash = d_commit_in48;  // c-kzg hashes the commitment bytes as given
    }
    if (mode == Mode::PointProof) {
      CU_TRY(cudaMemsetAsync(s.status2.p, 0, (size_t)n * sizeof(int), st));
      launch_le_fr_parse(s.z.p, (int*)s.status2.p, d_z_in_be, n, st, be);
      launch_status_or(stt, (const int*)s.status2.p, n, st);
    } else {
      CU_TRY(cudaStreamWaitEvent(st, s.ev_aux, 0));
      launch_challenge_finish(s.z.p, s.states.p, d_blobs, commit_for_hash, n, st, !be);
    }
    launch_le_eval_quot(s.q.p, nullptr, d_ybe, d_blobs, s.z.p, c->d_roots, n, st, be);
    run_msm(s, c, s.q.p, false, n, bpb, st);
    launch_msm_finalize(d_p48, nullptr, s.partials.p, bpb, n, st);
    return true;
  }
  if (mode == Mode::Commit) {
    run_msm(s, c, d_blobs, true, n, bpb, st);
    launch_msm_finalize(d_c48, nullptr, s.partials.p, bpb, n, st);
    if (d_status) CU_TRY(cudaMemsetAsync(d_status, 0, (size_t)n * sizeof(int), st));
    return true;
  }
  const void* commit_for_hash = nullptr;
  if (mode == Mode::CommitProve || mode == Mode::BlobProof) {
    // fork: SHA-256 midstate over the blob on the high-priority aux stream
    CU_TRY(cudaEventRecord(s.ev_fork, st));
    CU_TRY(cudaStreamWaitEvent(s.aux, s.ev_fork, 0));
    launch_challenge_midstate(s.states.p, d_blobs, n, s.aux, mode == Mode::BlobProof);
    CU_TRY(cudaEventRecord(s.ev_aux, s.aux));
  }
  if (mode == Mode::CommitProve) {
    run_msm(s, c, d_blobs, true, n, bpb, st);
    launch_msm_finalize(d_c48, nullptr, s.partials.p, bpb, n, st);
    commit_for_hash = d_c48;
    if (d_status) CU_TRY(cudaMemsetAsync(d_status, 0, (size_t)n * sizeof(int), st));
    if (!c->srs_in_g1) {
      // compute_blob_kzg_proof re-validates its commitment argument
      // (lib.rs:373): only matters for hand-made setups with points outside G1
      launch_g1_decompress(nullptr, nullptr, d_status ? d_status : (int*)s.status.p, d_c48, n, st);
    }
  } else if (mode == Mode::BlobProof) {
    // lib.rs:373-378: decode the commitment first; the hash sees its canonical re-encoding (utils.rs:138)
    launch_g1_decompress(nullptr, s.c48.p, d_status ? d_status : (int*)s.status.p, d_commit_in48, n, st);
    commit_for_hash = s.c48.p;
  }
  if (mode == Mode::PointProof) {
    launch_fr_from_be(s.z.p, d_z_in_be, n, st);
    if (d_status) CU_TRY(cudaMemsetAsync(d_status, 0, (size_t)n * sizeof(int), st));
  } else {
    CU_TRY(cudaStreamWaitEvent(st, s.ev_aux, 0));
    launch_challenge_finish(s.z.p, s.states.p, d_blobs, commit_for_hash, n, st);
  }
  launch_poly_eval_quot(s.q.p, nullptr, d_ybe, d_blobs, s.z.p, n, st);
  run_msm(s, c, s.q.p, false, n, bpb, st);
  launch_msm_finalize(d_p48, nullptr, s.partials.p, bpb, n, st);
  return true;
}

// ------------------------------------------------------------------ devices (lwkzg_set_devices)
std::vector<int>& device_list() {   // guarded by g_mu; empty = whatever device the settings were loaded on
  static std::vector<int> d;
  return d;
}

// Replica of c on the current device: same SRS, same window, same mode.  The host arrays hold the Lagrange points in
// the Lagrange modes, so the replica also gets a copy of the monomial points the primary context kept (FK20, cell
// verification).  NULL when any of it fails.
Ctx* build_replica(const Ctx* c) {
  Ctx* r = build_ctx(c->g1_host, c->g2_host, c->mode, c->c);
  if (!r || r->d_mono || !c->d_mono) return r;
  const size_t bytes = (size_t)N_POINTS * AFFINE_BYTES;
  cudaStream_t st = r->slot[0].st;
  if (cudaMalloc(&r->d_mono, bytes) != cudaSuccess) { destroy_ctx(r); return nullptr; }
  r->mono_owned = true;
  if (cudaMemcpyPeerAsync(r->d_mono, r->device, c->d_mono, c->device, bytes, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) {
    destroy_ctx(r);
    return nullptr;
  }
  return r;
}

// The contexts a call over n items runs on: the primary one plus a replica per other device of lwkzg_set_devices,
// built side by side on first use.  The call shards only when every context gets at least two items; otherwise it
// runs on the primary context alone and no replica is built for it.
std::vector<Ctx*> ctxs_for(Ctx* c, size_t n) {
  std::vector<int> devs;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    devs = device_list();
  }
  std::vector<Ctx*> out{c};
  const size_t g = 1 + devs.size() - std::count(devs.begin(), devs.end(), c->device);
  if (devs.size() <= 1 || !c->srs_valid || n < 2 * g) return out;
  std::lock_guard<std::mutex> lk(c->replicas_mu);
  std::vector<int> missing;
  for (int d : devs) {
    if (d == c->device) continue;
    bool have = false;
    for (Ctx* r : c->replicas) have = have || r->device == d;
    if (!have) missing.push_back(d);
  }
  if (!missing.empty()) {
    std::vector<Ctx*> built(missing.size(), nullptr);
    std::vector<std::thread> th;
    for (size_t k = 0; k < missing.size(); k++)
      th.emplace_back([&, k]() {
        if (cudaSetDevice(missing[k]) != cudaSuccess) return;
        built[k] = build_replica(c);
      });
    for (auto& t : th) t.join();
    for (Ctx* b : built)
      if (b) c->replicas.push_back(b);
  }
  for (int d : devs) {
    if (d == c->device) continue;
    for (Ctx* r : c->replicas)
      if (r->device == d && r->srs_valid) { out.push_back(r); break; }
  }
  return out;
}

// contiguous shard k of n items over g workers (SURVEY 8e)
void shard_of(size_t n, size_t g, size_t k, size_t& first, size_t& count) {
  const size_t base = n / g, rem = n % g;
  count = base + (k < rem ? 1 : 0);
  first = k * base + std::min(k, rem);
}

// fn(k, ctxs[k], first, count) for every shard of n items over the contexts, with that context's device current: one
// host thread per context, or inline on the calling thread when there is only one.  Returns the first failing code
// and its shard's error message.
template <class Fn>
C_KZG_RET for_shards(const std::vector<Ctx*>& ctxs, size_t n, const Fn& fn) {
  const size_t g = ctxs.size();
  std::vector<C_KZG_RET> rcs(g, C_KZG_OK);
  std::vector<std::string> errs(g);
  auto shard = [&](size_t k) {
    size_t first, count;
    shard_of(n, g, k, first, count);
    DeviceGuard dg(ctxs[k]->device);
    rcs[k] = fn(k, ctxs[k], first, count);
    if (rcs[k] != C_KZG_OK) errs[k] = tl_err;
  };
  if (g == 1) {
    shard(0);
  } else {
    std::vector<std::thread> th;
    for (size_t k = 0; k < g; k++) th.emplace_back(shard, k);
    for (auto& t : th) t.join();
  }
  for (size_t k = 0; k < g; k++)
    if (rcs[k] != C_KZG_OK) { set_err(errs[k]); return rcs[k]; }
  return C_KZG_OK;
}

// Host-buffer batches of independent items (commitments, proofs, cells, recovery: no exchange between shards) over
// the devices of lwkzg_set_devices.  run(ctx, first, count, status + first) does one shard on one device and fills
// one status code per item.  An unusable SRS fails every item.  With status == NULL the first failing item's code is
// returned, with `what` as the error message.
template <class Run>
C_KZG_RET sharded_batch(Ctx* c, size_t n, int* status, const char* what, const Run& run) {
  if (!c->srs_valid) {
    set_err("SRS re-hydration failed: g1_values holds a point that is not on the curve");
    if (status) for (size_t i = 0; i < n; i++) status[i] = C_KZG_ERROR;
    return C_KZG_ERROR;
  }
  std::vector<int> st_own;
  int* st = status;
  if (!st) { st_own.assign(n, 0); st = st_own.data(); }
  C_KZG_RET rc = for_shards(ctxs_for(c, n), n, [&](size_t, Ctx* x, size_t first, size_t count) { return run(x, first, count, st + first); });
  if (rc != C_KZG_OK) return rc;
  if (!status) {
    for (size_t i = 0; i < n; i++)
      if (st[i]) { set_err(what); return (C_KZG_RET)st[i]; }
  }
  return C_KZG_OK;
}

// Host-buffer batch driver on ONE device: chunked, double-buffered over the stream slots so
// the H2D copy of chunk k+1 overlaps the kernels of chunk k.  `status` receives one code per item.
C_KZG_RET host_batch_on(Ctx* c, Mode mode, size_t n, const Blob* blobs, const Bytes48* commit_in, const Bytes32* z_in,
                        Bytes48* c_out, Bytes48* p_out, Bytes32* y_out, int* status) {
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard dg(c->device);
  long chunk;
  {
    std::lock_guard<std::mutex> lk2(g_mu);
    chunk = std::max(1L, opts().chunk_blobs);
  }
  // outputs land in (pinned) temporaries so that failed items leave caller memory untouched
  // (lib.rs:275-281, 334-341) and the D2H copies stay asynchronous
  const size_t stage_bytes = n * (48 + 48 + 32 + sizeof(int));
  if (stage_bytes > c->h_stage_cap) {
    if (c->h_stage) cudaFreeHost(c->h_stage);
    c->h_stage = nullptr;
    c->h_stage_cap = 0;
    if (cudaMallocHost(&c->h_stage, stage_bytes) != cudaSuccess) { set_err("cudaMallocHost failed"); return C_KZG_MALLOC; }
    c->h_stage_cap = stage_bytes;
  }
  Bytes48* c_tmp = (Bytes48*)c->h_stage;
  Bytes48* p_tmp = c_tmp + n;
  Bytes32* y_tmp = (Bytes32*)(p_tmp + n);
  int* st_host = (int*)(y_tmp + n);
  memset(st_host, 0, n * sizeof(int));
  auto fail = [&]() {
    for (auto& sl : c->slot) { cudaStreamSynchronize(sl.st); cudaStreamSynchronize(sl.aux); }
    return C_KZG_ERROR;
  };
  // blobs in pageable memory go through the pinned ring (see HostStager); tiny calls are not worth the ring
  const bool pageable = n * BLOB_BYTES >= (size_t(4) << 20) && is_pageable_host(blobs) &&
                        c->ring.ensure(std::min<size_t>(n, (size_t)chunk) * BLOB_BYTES);
  size_t k = 0;
  for (size_t off = 0, m_sz = 0; off < n; off += m_sz, k++) {
    m_sz = chunk_at(off, n, (size_t)chunk);
    int m = (int)m_sz;
    Slot& sl = c->slot[k % NSLOT];
    if (cudaStreamSynchronize(sl.st) != cudaSuccess) { set_err("stream sync failed"); return fail(); }
    if (!reserve(slot_buffers(sl, m, auto_bpb(m), true))) return fail();
    if (pageable) {
      if (!c->ring.h2d(sl.blobs.p, blobs + off, (size_t)m * BLOB_BYTES, c->ring_seq++, sl.st)) return fail();
    } else if (cudaMemcpyAsync(sl.blobs.p, blobs + off, (size_t)m * BLOB_BYTES, cudaMemcpyHostToDevice, sl.st) != cudaSuccess) { set_err("H2D failed"); return fail(); }
    if (mode == Mode::BlobProof && cudaMemcpyAsync(sl.cin48.p, commit_in + off, (size_t)m * 48, cudaMemcpyHostToDevice, sl.st) != cudaSuccess) { set_err("H2D failed"); return fail(); }
    if (mode == Mode::PointProof && cudaMemcpyAsync(sl.zbe.p, z_in + off, (size_t)m * 32, cudaMemcpyHostToDevice, sl.st) != cudaSuccess) { set_err("H2D failed"); return fail(); }
    void* d_c48 = (mode == Mode::BlobProof) ? nullptr : sl.c48.p;
    if (!enqueue_chunk(c, sl, mode, sl.blobs.p, m, d_c48, sl.p48.p, y_out ? sl.ybe.p : nullptr, (int*)sl.status.p, sl.cin48.p, sl.zbe.p)) return fail();
    cudaError_t ce = cudaSuccess;
    if (c_out && ce == cudaSuccess) ce = cudaMemcpyAsync(&c_tmp[off], sl.c48.p, (size_t)m * 48, cudaMemcpyDeviceToHost, sl.st);
    if (p_out && ce == cudaSuccess) ce = cudaMemcpyAsync(&p_tmp[off], sl.p48.p, (size_t)m * 48, cudaMemcpyDeviceToHost, sl.st);
    if (y_out && ce == cudaSuccess) ce = cudaMemcpyAsync(&y_tmp[off], sl.ybe.p, (size_t)m * 32, cudaMemcpyDeviceToHost, sl.st);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(&st_host[off], sl.status.p, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, sl.st);
    if (ce != cudaSuccess) { set_err(std::string("D2H failed: ") + cudaGetErrorString(ce)); return fail(); }
  }
  for (auto& sl : c->slot) {
    cudaError_t e = cudaStreamSynchronize(sl.st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(sl.aux);
    if (e != cudaSuccess) { set_err(std::string("kernel failure: ") + cudaGetErrorString(e)); return C_KZG_ERROR; }
  }
  if (cudaGetLastError() != cudaSuccess) { set_err("CUDA launch failure"); return C_KZG_ERROR; }
  for (size_t i = 0; i < n; i++) {
    if (st_host[i] == 0) {
      if (c_out) c_out[i] = c_tmp[i];
      if (p_out) p_out[i] = p_tmp[i];
      if (y_out) y_out[i] = y_tmp[i];
    }
    status[i] = st_host[i];
  }
  return C_KZG_OK;
}

// Host-buffer batch driver: one device, or -- after lwkzg_set_devices -- contiguous shards of the batch on every
// listed GPU, one host thread and stream set per device, no exchange between them (SURVEY 8e: commit / proof
// batches are independent units).
C_KZG_RET host_batch(Mode mode, const KZGSettings* s, size_t n, const Blob* blobs, const Bytes48* commit_in, const Bytes32* z_in,
                     Bytes48* c_out, Bytes48* p_out, Bytes32* y_out, int* status) {
  if (n == 0) return C_KZG_OK;
  Ctx* c = ctx_of(s);
  if (!c) return C_KZG_ERROR;
  return sharded_batch(c, n, status, "invalid input item", [&](Ctx* x, size_t first, size_t count, int* st) {
    return host_batch_on(x, mode, count, blobs + first, commit_in ? commit_in + first : nullptr, z_in ? z_in + first : nullptr,
                         c_out ? c_out + first : nullptr, p_out ? p_out + first : nullptr, y_out ? y_out + first : nullptr, st);
  });
}

// Device-buffer batch driver, asynchronous with respect to the host: forks from
// `user` onto the two internal slots and joins back.
C_KZG_RET device_batch(Mode mode, const KZGSettings* s, size_t n, const void* d_blobs, const void* d_commit_in, void* d_c_out,
                       void* d_p_out, void* d_status, cudaStream_t user) {
  if (n == 0) return C_KZG_OK;
  Ctx* c = ctx_of(s);
  if (!c) return C_KZG_ERROR;
  if (!c->srs_valid) { set_err("SRS re-hydration failed"); return C_KZG_ERROR; }
  std::lock_guard<std::mutex> lk(c->mu);
  DeviceGuard dg(c->device);
  long chunk;
  {
    std::lock_guard<std::mutex> lk2(g_mu);
    chunk = std::max(1L, opts().chunk_blobs);
  }
  // buffers must be big enough BEFORE anything is enqueued (a realloc would
  // pull memory from under kernels still in flight on another slot): plan the
  // chunks first and size every slot for the largest request it will see
  // (a small remainder chunk may need MORE block partials than a full one)
  std::vector<std::pair<size_t, size_t>> plan;
  for (size_t off = 0; off < n;) {
    const size_t m = chunk_at(off, n, (size_t)chunk);
    plan.emplace_back(off, m);
    off += m;
  }
  // The host only waits for earlier work when a buffer really has to grow: back-to-back calls (also from
  // different user streams) then queue behind each other on the slot streams and the tail of one batch
  // overlaps the head of the next.
  std::vector<BufList> bufs;
  bool all_fit = true;
  for (size_t k = 0; k < plan.size(); k++) {
    bufs.push_back(slot_buffers(c->slot[k % NSLOT], (int)plan[k].second, auto_bpb((int)plan[k].second), false));
    all_fit = all_fit && fits(bufs.back());
  }
  if (!all_fit) {
    for (auto& sl : c->slot) { cudaStreamSynchronize(sl.st); cudaStreamSynchronize(sl.aux); }
    for (const BufList& b : bufs)
      if (!reserve(b)) return C_KZG_ERROR;
  }
  cudaEvent_t ev_user;
  if (cudaEventCreateWithFlags(&ev_user, cudaEventDisableTiming) != cudaSuccess) { set_err("event"); return C_KZG_ERROR; }
  cudaEventRecord(ev_user, user);
  for (auto& sl : c->slot) cudaStreamWaitEvent(sl.st, ev_user, 0);
  size_t k = 0;
  bool ok = true;
  for (; k < plan.size() && ok; k++) {
    const size_t off = plan[k].first;
    const int m = (int)plan[k].second;
    Slot& sl = c->slot[k % NSLOT];
    const uint8_t* b = (const uint8_t*)d_blobs + off * BLOB_BYTES;
    void* co = d_c_out ? (uint8_t*)d_c_out + off * 48 : (mode == Mode::CommitProve ? sl.c48.p : nullptr);
    void* po = d_p_out ? (uint8_t*)d_p_out + off * 48 : nullptr;
    const void* ci = d_commit_in ? (const uint8_t*)d_commit_in + off * 48 : nullptr;
    int* so = d_status ? (int*)d_status + off : (int*)sl.status.p;
    ok = enqueue_chunk(c, sl, mode, b, m, co, po, nullptr, so, ci, nullptr);
    if (ok && (mode == Mode::BlobProof || c->lagrange())) {   // the only ways an item can fail: bad commitment / non-canonical blob
      if (co && d_c_out) launch_zero_failed(co, 48, so, m, sl.st);
      if (po) launch_zero_failed(po, 48, so, m, sl.st);
    }
  }
  for (auto& sl : c->slot) {
    cudaEventRecord(sl.ev_done, sl.st);
    cudaStreamWaitEvent(user, sl.ev_done, 0);
  }
  cudaEventDestroy(ev_user);
  if (!ok || cudaGetLastError() != cudaSuccess) { if (ok) set_err("CUDA launch failure"); return C_KZG_ERROR; }
  return C_KZG_OK;
}

// ------------------------------------------------------------------ setup loading
bool hex_nibble(char ch, uint8_t& v) {
  if (ch >= '0' && ch <= '9') { v = (uint8_t)(ch - '0'); return true; }
  if (ch >= 'a' && ch <= 'f') { v = (uint8_t)(ch - 'a' + 10); return true; }
  if (ch >= 'A' && ch <= 'F') { v = (uint8_t)(ch - 'A' + 10); return true; }
  return false;
}
// hex::decode_to_slice semantics: exact length, hex digits only
bool hex_line(const std::string& ln, uint8_t* out, size_t nbytes) {
  if (ln.size() != 2 * nbytes) return false;
  for (size_t i = 0; i < nbytes; i++) {
    uint8_t a, b;
    if (!hex_nibble(ln[2 * i], a) || !hex_nibble(ln[2 * i + 1], b)) return false;
    out[i] = (uint8_t)(a << 4 | b);
  }
  return true;
}
// str::parse::<usize>: optional '+', digits only, no whitespace
bool parse_usize(const std::string& ln, size_t& v) {
  size_t i = 0;
  if (i < ln.size() && ln[i] == '+') i++;
  if (i >= ln.size()) return false;
  v = 0;
  for (; i < ln.size(); i++) {
    if (ln[i] < '0' || ln[i] > '9') return false;
    if (v > (SIZE_MAX - 9) / 10) return false;
    v = v * 10 + (size_t)(ln[i] - '0');
  }
  return true;
}

// Decode + validate compressed points on the device, then lay out KZGSettings
// exactly as src/srs.rs:99-153 / src/lib.rs:724-758 do.  n1 / n2 may be
// smaller than 4096 / 65 for the file loader (tests/trusted_setup_4.txt): the
// arrays are always allocated full size and zero-padded so later calls stay
// memory safe (they then fail SRS re-hydration -> C_KZG_ERROR).
C_KZG_RET settings_from_compressed(KZGSettings* out, const uint8_t* g1_bytes, size_t n1, const uint8_t* g2_bytes, size_t n2) {
  size_t a1 = std::max<size_t>(n1, N_POINTS), a2 = std::max<size_t>(n2, TRUSTED_SETUP_NUM_G2_POINTS);
  void *d_in1 = nullptr, *d_in2 = nullptr, *d_c1 = nullptr, *d_c2 = nullptr;
  int* d_st = nullptr;
  std::vector<uint32_t> c1(n1 * 24), c2(n2 * 48);
  std::vector<int> st(n1 + n2);
  auto cleanup = [&]() {
    cudaFree(d_in1); cudaFree(d_in2); cudaFree(d_c1); cudaFree(d_c2); cudaFree(d_st);
  };
  auto run = [&]() -> bool {
    CU_TRY(cudaMalloc(&d_in1, std::max<size_t>(n1, 1) * 48));
    CU_TRY(cudaMalloc(&d_in2, std::max<size_t>(n2, 1) * 96));
    CU_TRY(cudaMalloc(&d_c1, std::max<size_t>(n1, 1) * 96));
    CU_TRY(cudaMalloc(&d_c2, std::max<size_t>(n2, 1) * 192));
    CU_TRY(cudaMalloc(&d_st, (n1 + n2 + 1) * sizeof(int)));
    if (n1) CU_TRY(cudaMemcpy(d_in1, g1_bytes, n1 * 48, cudaMemcpyHostToDevice));
    if (n2) CU_TRY(cudaMemcpy(d_in2, g2_bytes, n2 * 96, cudaMemcpyHostToDevice));
    launch_setup_decode_g1(d_c1, d_st, d_in1, (int)n1, 0);
    launch_setup_decode_g2(d_c2, d_st + n1, d_in2, (int)n2, 0);
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaGetLastError());
    if (n1) CU_TRY(cudaMemcpy(c1.data(), d_c1, n1 * 96, cudaMemcpyDeviceToHost));
    if (n2) CU_TRY(cudaMemcpy(c2.data(), d_c2, n2 * 192, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(st.data(), d_st, (n1 + n2) * sizeof(int), cudaMemcpyDeviceToHost));
    return true;
  };
  bool ok = run();
  cleanup();
  if (!ok) return C_KZG_ERROR;
  for (size_t i = 0; i < n1; i++)
    if (st[i] != 0) { set_err("invalid G1 point in trusted setup"); return C_KZG_ERROR; }
  for (size_t i = 0; i < n2; i++)
    if (st[n1 + i] == 2) { set_err("invalid G2 point in trusted setup"); return C_KZG_ERROR; }

  g1_t* g1 = (g1_t*)calloc(a1, sizeof(g1_t));
  g2_t* g2 = (g2_t*)calloc(a2, sizeof(g2_t));
  if (!g1 || !g2) { free(g1); free(g2); return C_KZG_MALLOC; }
  for (size_t i = 0; i < n1; i++) {
    canon_to_blst_fp(&g1[i].x, &c1[i * 24]);
    canon_to_blst_fp(&g1[i].y, &c1[i * 24 + 12]);
    g1[i].z.l[5] = 1;  // z = 1, most-significant-first limbs (srs.rs:131-153; also for infinity)
  }
  for (size_t i = n1; i < a1; i++) g1[i].z.l[5] = 1;
  for (size_t i = 0; i < n2; i++) {
    canon_to_blst_fp(&g2[i].x.fp[0], &c2[i * 48]);
    canon_to_blst_fp(&g2[i].x.fp[1], &c2[i * 48 + 12]);
    canon_to_blst_fp(&g2[i].y.fp[0], &c2[i * 48 + 24]);
    canon_to_blst_fp(&g2[i].y.fp[1], &c2[i * 48 + 36]);
    if (st[n1 + i] == 0) g2[i].z.fp[0].l[5] = 1;  // affine z = 1 + 0u ; infinity keeps z = 0
  }
  const int mode = (int)current_mode();
  if (mode != 0 && n1 == N_POINTS) {
    // c-kzg's load_trusted_setup stores the SRS in Lagrange form, bit-reversed
    // (the step the reference left as a TODO, lib.rs:760-770): L_i = sum_j (1/n) w_i^-j [tau^j]G,
    // computed as 4096 fixed-base MSMs over a temporary 8-bit table of the monomial points.
    Ctx* tmp = build_ctx(g1, g2, 0, 8);
    if (!tmp || !tmp->srs_valid) { if (tmp) destroy_ctx(tmp); free(g1); free(g2); set_err("Lagrange conversion failed"); return C_KZG_ERROR; }
    std::vector<uint32_t> lag((size_t)N_POINTS * 24);
    bool good = [&]() -> bool {
      void *d_rows = nullptr, *d_aff = nullptr, *d_canon = nullptr;
      Slot& sl = tmp->slot[0];
      const int bpb = 1;
      if (!reserve(slot_buffers(sl, N_POINTS, bpb, false))) return false;
      CU_TRY(cudaMalloc(&d_rows, (size_t)N_POINTS * BLOB_BYTES));
      CU_TRY(cudaMalloc(&d_aff, (size_t)N_POINTS * AFFINE_BYTES));
      CU_TRY(cudaMalloc(&d_canon, (size_t)N_POINTS * 96));
      launch_le_idft_rows(d_rows, sl.st);
      run_msm(sl, tmp, d_rows, false, N_POINTS, bpb, sl.st);
      launch_msm_finalize(nullptr, d_aff, sl.partials.p, bpb, N_POINTS, sl.st);
      launch_affine_to_canon(d_canon, d_aff, N_POINTS, sl.st);
      CU_TRY(cudaMemcpyAsync(lag.data(), d_canon, (size_t)N_POINTS * 96, cudaMemcpyDeviceToHost, sl.st));
      CU_TRY(cudaStreamSynchronize(sl.st));
      CU_TRY(cudaGetLastError());
      cudaFree(d_rows); cudaFree(d_aff); cudaFree(d_canon);
      return true;
    }();
    destroy_ctx(tmp);
    if (!good) { free(g1); free(g2); return C_KZG_ERROR; }
    for (size_t i = 0; i < (size_t)N_POINTS; i++) {
      canon_to_blst_fp(&g1[i].x, &lag[i * 24]);
      canon_to_blst_fp(&g1[i].y, &lag[i * 24 + 12]);
    }
  }
  Ctx* c = build_ctx(g1, g2, mode);
  if (!c) { free(g1); free(g2); return C_KZG_ERROR; }
  if (mode != 0 && n1 == N_POINTS && c->srs_valid) {
    // the Lagrange modes keep the monomial points too (c-kzg's g1_values_monomial): FK20 and cell verification need them
    bool good = [&]() -> bool {
      DeviceGuard dg(c->device);
      void* d_canon = nullptr;
      int* d_flags = nullptr;
      CU_TRY(cudaMalloc(&d_canon, (size_t)N_POINTS * 96));
      CU_TRY(cudaMalloc(&d_flags, 2 * N_POINTS * sizeof(int)));
      CU_TRY(cudaMalloc(&c->d_mono, (size_t)N_POINTS * AFFINE_BYTES));
      c->mono_owned = true;
      // on the kernel's own stream: a plain cudaMemcpy from pageable memory may return before the DMA has landed, and
      // a non-blocking stream does not wait for the legacy stream
      CU_TRY(cudaMemcpyAsync(d_canon, c1.data(), (size_t)N_POINTS * 96, cudaMemcpyHostToDevice, c->slot[0].st));
      launch_srs_import(c->d_mono, d_canon, d_flags, d_flags + N_POINTS, N_POINTS, c->slot[0].st);
      std::vector<int> flags(N_POINTS);
      CU_TRY(cudaMemcpyAsync(flags.data(), d_flags, N_POINTS * sizeof(int), cudaMemcpyDeviceToHost, c->slot[0].st));
      CU_TRY(cudaStreamSynchronize(c->slot[0].st));
      CU_TRY(cudaGetLastError());
      cudaFree(d_canon);
      cudaFree(d_flags);
      for (int f : flags)
        if (f) { set_err("monomial SRS import failed"); return false; }
      return true;
    }();
    if (!good) { destroy_ctx(c); free(g1); free(g2); return C_KZG_ERROR; }
  }
  out->fs = reinterpret_cast<FFTSettings*>(c);
  out->g1_values = g1;
  out->g2_values = g2;
  return C_KZG_OK;
}

// ------------------------------------------------------------------ verification
// blobs of a batched verification are staged on the device "verify_super_blobs" at a time (default 16384 = 2 GiB)
size_t vb_super_blobs() {
  std::lock_guard<std::mutex> lk(g_mu);
  return (size_t)std::max(1L, opts().verify_super_blobs);
}
bool vb_reserve(Ctx* c, size_t n, bool stage_blobs = true) {
  const size_t VB_SUPER_BLOBS = stage_blobs ? vb_super_blobs() : 0;
  return c->vb_cin.ensure(n * 48) && c->vb_pin.ensure(n * 48) && c->vb_caff.ensure(n * AFFINE_BYTES) && c->vb_piaff.ensure(n * AFFINE_BYTES) &&
         c->vb_c48r.ensure(n * 48) && c->vb_p48r.ensure(n * 48) && c->vb_z.ensure(n * 32) && c->vb_y.ensure(n * 32) && c->vb_tuples.ensure(n * 160) &&
         c->vb_status.ensure(n * sizeof(int)) && c->vb_r.ensure(32) && c->vb_partial.ensure(288) && c->vb_ok.ensure(sizeof(int)) &&
         c->vb_zy_in.ensure(n * 64) && c->vb_scratch.ensure(batch_partials_scratch_bytes((int)n)) &&
         c->vb_hstate.ensure(batch_challenge_state_bytes()) && c->vb_blobs.ensure(std::max<size_t>(std::min<size_t>(n, VB_SUPER_BLOBS), 1) * (stage_blobs ? (size_t)BLOB_BYTES : 16)) &&
         c->vb_states.ensure(n * 32) && c->vb_status2.ensure(n * sizeof(int));
}

// Per-blob preparation of a batched verification (lib.rs:562-596): decode C_i
// and pi_i, z_i = challenge(blob_i, C_i), y_i = p_i(z_i); everything stays in
// the context's verify workspace.  Host blobs are streamed through the two
// slots in chunks.  Returns false on CUDA failure; invalid items are reported
// through vb_status.
// hash_r: also derive the batch challenge r (utils.rs:166-206) into vb_r, absorbing each chunk's tuples as soon as
// they exist.
// defer_subgroup: the points are decoded without their r-torsion tests -- the single-proof kernel runs them itself,
// beside its scalar multiplications (verify_single_from_workspace(..., true))
bool verify_prepare(Ctx* c, const Blob* blobs, const Bytes48* commitments, const Bytes48* proofs, size_t n, bool hash_r = false,
                    bool dev_inputs = false, bool defer_subgroup = false) {
  c->vb_n = 0;   // whatever a previous phase 1 left in the workspace is about to be overwritten
  // the reference re-hydrates the SRS before anything else in every entry point (lib.rs:256-262, 420-426, 468-474,
  // 548-554): an unusable SRS is an error whatever the other arguments are -- and the kernels below need it
  if (!c->srs_valid || !c->g2_valid) { set_err("SRS re-hydration failed"); return false; }
  if (!vb_reserve(c, n, !dev_inputs)) return false;
  long chunk;
  {
    std::lock_guard<std::mutex> lk2(g_mu);
    chunk = std::max(1L, opts().chunk_blobs);
  }
  cudaStream_t s0 = c->slot[0].st;
  const bool le = c->lagrange(), be = c->be_wire();
  const int wire = c->mode;
  const cudaMemcpyKind in_kind = dev_inputs ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  // commitments on s0, proofs on the hash stream (idle until the first tuples exist): the two decompressions are
  // latency-bound thread-per-point kernels and run side by side
  CU_TRY(cudaMemcpyAsync(c->vb_cin.p, commitments, n * 48, in_kind, s0));
  CU_TRY(cudaMemcpyAsync(c->vb_pin.p, proofs, n * 48, in_kind, c->hash_st));
  // Large batches: decoding (a square root) gates the blob hashes, the r-torsion tests (two thirds of a decompression)
  // do not -- they run beside the first chunks on the two compute streams the chunks leave free and are merged into
  // the status array at the end.
  bool split, overlap_decode;
  {
    std::lock_guard<std::mutex> lk2(g_mu);
    overlap_decode = opts().verify_overlap_decode != 0;
    split = opts().verify_split_subgroup != 0 && n > 64 && opts().verify_streams <= 2 * NSLOT - 2;
  }
  if (split && !c->vb_sub.ensure(2 * n * sizeof(int))) return false;
  launch_g1_decompress(c->vb_caff.p, c->vb_c48r.p, (int*)c->vb_status.p, c->vb_cin.p, (int)n, s0, le, !split && !defer_subgroup);
  // proofs: decode status into the (still unused) tuples buffer, then merge
  launch_g1_decompress(c->vb_piaff.p, c->vb_p48r.p, (int*)c->vb_tuples.p, c->vb_pin.p, (int)n, c->hash_st, le, !split && !defer_subgroup);
  CU_TRY(cudaEventRecord(c->ev_hash, c->hash_st));
  CU_TRY(cudaStreamWaitEvent(s0, c->ev_hash, 0));
  launch_status_or((int*)c->vb_status.p, (const int*)c->vb_tuples.p, (int)n, s0);
  // the blob copies and SHA midstates do not need the decoded points: only the challenge tail does, so the
  // slot streams wait for the decompression through an event instead of the host waiting here
  CU_TRY(cudaEventRecord(c->slot[0].ev_in, s0));
  if (split) {
    cudaStream_t sa = c->slot[NSLOT - 1].st, sb = c->slot[NSLOT - 1].aux;
    CU_TRY(cudaStreamWaitEvent(sa, c->slot[0].ev_in, 0));
    CU_TRY(cudaStreamWaitEvent(sb, c->slot[0].ev_in, 0));
    launch_g1_subgroup_check((int*)c->vb_sub.p, c->vb_caff.p, (int)n, sa, le);
    launch_g1_subgroup_check((int*)c->vb_sub.p + n, c->vb_piaff.p, (int)n, sb, le);
    CU_TRY(cudaEventRecord(c->slot[NSLOT - 1].ev_done, sa));
    CU_TRY(cudaEventRecord(c->slot[NSLOT - 1].ev_aux, sb));
  }
  // Blobs land in a verify-owned staging area big enough for a whole super-batch, so no chunk ever waits for a
  // buffer: one copy stream issues the H2D copies back to back, and each chunk's kernels (SHA midstate ->
  // challenge -> evaluation -> tuple) start on one of 2 * NSLOT compute streams as soon as its copy has landed.
  // The copy engine is the only thing that runs the whole time.
  const size_t super = dev_inputs ? n : std::min<size_t>(n, vb_super_blobs());   // device blobs are read in place
  // (measured and not kept: small first chunks, so that the batch-challenge hash -- one sequential SHA-256 over
  // all tuples, ~1 us per 64-byte block, as long as the blob copies -- starts absorbing 1.5 ms earlier: the hash
  // then runs slower beside the extra kernels and the batch ends 0.4 ms later, profiles/r02_verify_notes.md)
  auto chunk_len = [&](size_t, size_t left) -> size_t { return std::min((size_t)chunk, left); };
  auto need_events = [&](size_t count) -> bool {
    while (c->ev_pool.size() < count) {
      cudaEvent_t e;
      CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      c->ev_pool.push_back(e);
    }
    return true;
  };
  cudaStream_t cs[2 * NSLOT];
  // how many of them are used: with the copy stream, the hash stream and the caller's stream, more than eight streams
  // share hardware queues (CUDA_DEVICE_MAX_CONNECTIONS defaults to 8) and chunks serialise behind the sequential
  // batch-challenge launches of a stream they have nothing to do with
  int ncs;
  {
    std::lock_guard<std::mutex> lk2(g_mu);
    ncs = (int)std::min<long>(std::max<long>(opts().verify_streams, 1), 2 * NSLOT);
  }
  for (int i = 0; i < NSLOT; i++) { cs[2 * i] = c->slot[i].st; cs[2 * i + 1] = c->slot[i].aux; }
  auto sync_all = [&]() -> bool {
    CU_TRY(cudaStreamSynchronize(c->copy_st));
    for (auto st : cs) CU_TRY(cudaStreamSynchronize(st));
    return true;
  };
  static const bool trace = getenv("LWKZG_VERIFY_TRACE") != nullptr;
  cudaEvent_t tr[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> trace_chunks;
  if (trace) {
    for (auto& e : tr) cudaEventCreate(&e);
    cudaEventRecord(tr[0], c->copy_st);
    cudaEventRecord(tr[3], s0);   // end of point decompression (s0 has only that queued so far)
  }
  const bool pageable = !dev_inputs && n * BLOB_BYTES >= (size_t(4) << 20) && is_pageable_host(blobs) &&
                        c->ring.ensure(std::min<size_t>(n, (size_t)chunk) * BLOB_BYTES);
  size_t k = 0;
  int hashed_blocks = 0;   // 64-byte blocks of the batch-challenge message absorbed so far
  for (size_t base = 0; base < n; base += super) {
    if (base > 0 && !sync_all()) return false;   // the staging area is about to be overwritten
    const size_t top = std::min(n, base + super);
    size_t j = 0;
    for (size_t off = base, m_sz = 0; off < top; off += m_sz, k++, j++) {
      m_sz = chunk_len(off, top - off);
      const int m = (int)m_sz;
      if (!need_events(2 * j + 2)) return false;
      const uint8_t* d_blobs = dev_inputs ? (const uint8_t*)blobs + off * BLOB_BYTES : (const uint8_t*)c->vb_blobs.p + (off - base) * BLOB_BYTES;
      void* d_states = (uint8_t*)c->vb_states.p + off * 32;
      cudaEvent_t ev_copied = c->ev_pool[2 * j], ev_tuples = c->ev_pool[2 * j + 1];
      cudaStream_t st = cs[(k + 1) % ncs];   // chunk 0 not on s0: its hash runs beside the commitment decompression
      if (!dev_inputs) {
        if (pageable) {
          if (!c->ring.h2d((void*)d_blobs, blobs + off, (size_t)m * BLOB_BYTES, c->ring_seq++, c->copy_st)) return false;
        } else {
          CU_TRY(cudaMemcpyAsync((void*)d_blobs, blobs + off, (size_t)m * BLOB_BYTES, cudaMemcpyHostToDevice, c->copy_st));
        }
      }
      CU_TRY(cudaEventRecord(ev_copied, c->copy_st));
      CU_TRY(cudaStreamWaitEvent(st, ev_copied, 0));
      cudaEvent_t tc[3] = {nullptr, nullptr, nullptr};
      // (measured: a hash kernel that starts while the two decompression kernels are still running takes 9-15 ms
      // instead of 2.7 -- so every chunk waits for them, ~2 ms after the call began, before anything else)
      // (small batches use the warp-per-blob hash, which does not show this, and want the overlap)
      if (!overlap_decode && n > 64) CU_TRY(cudaStreamWaitEvent(st, c->slot[0].ev_in, 0));
      if (trace) { for (auto& e : tc) cudaEventCreate(&e); cudaEventRecord(tc[0], st); }
      launch_challenge_midstate(d_states, d_blobs, m, st, true, be);
      if (trace) cudaEventRecord(tc[1], st);
      if (overlap_decode || n <= 64) CU_TRY(cudaStreamWaitEvent(st, c->slot[0].ev_in, 0));
      if (le) {
        int* st2 = (int*)c->vb_status2.p + off;
        CU_TRY(cudaMemsetAsync(st2, 0, (size_t)m * sizeof(int), st));
        launch_le_blob_check(st2, d_blobs, m, st, be);
        launch_status_or((int*)c->vb_status.p + off, st2, m, st);
        launch_challenge_finish((uint8_t*)c->vb_z.p + off * 32, d_states, d_blobs, (const uint8_t*)c->vb_cin.p + off * 48, m, st, !be);
        launch_le_eval_quot(nullptr, (uint8_t*)c->vb_y.p + off * 32, nullptr, d_blobs, (const uint8_t*)c->vb_z.p + off * 32, c->d_roots, m, st, be);
      } else {
        launch_challenge_finish((uint8_t*)c->vb_z.p + off * 32, d_states, d_blobs, (const uint8_t*)c->vb_c48r.p + off * 48, m, st);
        launch_poly_eval_quot(nullptr, (uint8_t*)c->vb_y.p + off * 32, nullptr, d_blobs, (const uint8_t*)c->vb_z.p + off * 32, m, st);
      }
      launch_make_tuples((uint8_t*)c->vb_tuples.p + off * 160, (const uint8_t*)c->vb_c48r.p + off * 48, (const uint8_t*)c->vb_z.p + off * 32,
                         (const uint8_t*)c->vb_y.p + off * 32, (const uint8_t*)c->vb_p48r.p + off * 48, m, st, le && !be);
      if (trace) { cudaEventRecord(tc[2], st); for (auto e : tc) trace_chunks.push_back(e); }
      if (hash_r) {
        // chunks reach the hash stream in order; each launch absorbs the blocks its chunk completed
        CU_TRY(cudaEventRecord(ev_tuples, st));
        CU_TRY(cudaStreamWaitEvent(c->hash_st, ev_tuples, 0));
        const bool last = off + (size_t)m >= n;
        const int ready = batch_challenge_blocks_ready(off + (size_t)m);
        launch_batch_challenge_part(c->vb_r.p, c->vb_hstate.p, c->vb_tuples.p, n, hashed_blocks, ready, k == 0, last, c->hash_st, wire);
        hashed_blocks = ready;
      }
    }
  }
  if (trace) { cudaEventRecord(tr[1], c->copy_st); cudaEventRecord(tr[2], c->hash_st); cudaEventRecord(tr[4], cs[k % ncs]); }
  if (split) {
    CU_TRY(cudaStreamWaitEvent(s0, c->slot[NSLOT - 1].ev_done, 0));
    CU_TRY(cudaStreamWaitEvent(s0, c->slot[NSLOT - 1].ev_aux, 0));
    launch_status_or((int*)c->vb_status.p, (const int*)c->vb_sub.p, (int)n, s0);
    launch_status_or((int*)c->vb_status.p, (const int*)c->vb_sub.p + n, (int)n, s0);
  }
  if (!sync_all()) return false;
  if (trace) {
    cudaStreamSynchronize(c->hash_st);
    float a = 0, b = 0, d = 0, e = 0;
    cudaEventElapsedTime(&a, tr[0], tr[1]);
    cudaEventElapsedTime(&b, tr[0], tr[2]);
    cudaEventElapsedTime(&d, tr[0], tr[3]);
    cudaEventElapsedTime(&e, tr[0], tr[4]);
    fprintf(stderr, "[lwkzg] prepare n=%zu: decompress done at %.2f ms, copies done at %.2f ms, last chunk's tuples at %.2f ms, challenge hash done at %.2f ms\n", n, d, a, e, b);
    for (size_t q = 0; q + 2 < trace_chunks.size() + 0 && n > 1; q += 3) {
      float x = 0, y = 0, z = 0;
      cudaEventElapsedTime(&x, tr[0], trace_chunks[q]);
      cudaEventElapsedTime(&y, tr[0], trace_chunks[q + 1]);
      cudaEventElapsedTime(&z, tr[0], trace_chunks[q + 2]);
      fprintf(stderr, "[lwkzg]   chunk %zu: hash starts %.2f, hash done %.2f, tuples %.2f\n", q / 3, x, y, z);
    }
    for (auto e : trace_chunks) cudaEventDestroy(e);
    for (auto& ev : tr) cudaEventDestroy(ev);
  }
  if (hash_r) CU_TRY(cudaStreamSynchronize(c->hash_st));
  CU_TRY(cudaGetLastError());
  c->vb_n = n;
  return true;
}

// first non-zero per-item code of the verify workspace (0 = all items valid)
bool first_bad_status(Ctx* c, size_t n, int& code) {
  std::vector<int> st(n);
  CU_TRY(cudaMemcpy(st.data(), c->vb_status.p, n * sizeof(int), cudaMemcpyDeviceToHost));
  code = 0;
  for (int v : st)
    if (v) { code = v; break; }
  return true;
}
C_KZG_RET bad_code(int code) { return code == 1 ? C_KZG_BADARGS : C_KZG_ERROR; }

// single-proof verification with everything already decoded in the workspace (item 0).  deferred_subgroup: C and pi
// were decoded without their r-torsion tests; the kernel runs them on its second warp, beside the scalar
// multiplications, and reports a failure through vb_status[0] -> `bad` (0 = fine)
bool verify_single_from_workspace(Ctx* c, bool& ok, bool deferred_subgroup = false, int* bad = nullptr) {
  cudaStream_t s0 = c->slot[0].st;
  // reference: KZG::verify subtracts y * srs[0] (= G for a monomial setup); c-kzg uses the generator itself
  launch_verify_single((int*)c->vb_ok.p, c->vb_caff.p, c->vb_piaff.p, c->vb_z.p, c->vb_y.p, c->lagrange() ? c->d_gen : c->d_srs, c->d_prep0, c->d_prep1,
                       c->lagrange() || c->srs_in_g1, s0, deferred_subgroup ? (int*)c->vb_status.p : nullptr, c->lagrange() ? 1 : 2);
  int out[2] = {0, 0};
  CU_TRY(cudaMemcpyAsync(&out[0], c->vb_ok.p, sizeof(int), cudaMemcpyDeviceToHost, s0));
  if (deferred_subgroup) CU_TRY(cudaMemcpyAsync(&out[1], c->vb_status.p, sizeof(int), cudaMemcpyDeviceToHost, s0));
  CU_TRY(cudaStreamSynchronize(s0));
  CU_TRY(cudaGetLastError());
  ok = out[0] != 0;
  if (bad) *bad = out[1];
  return true;
}

struct CtxLock {
  Ctx* c;
  std::unique_lock<std::mutex> lk;
  DeviceGuard dg;
  explicit CtxLock(Ctx* ctx) : c(ctx), lk(ctx->mu), dg(ctx->device) {}
};

#include "cells_host.inl"

}  // namespace

// =================================================================== C ABI
extern "C" {

const char* lwkzg_last_error(void) { return tl_err.c_str(); }
const char* lwkzg_version(void) { return "lwkzg-b200 0.2 (sm_100a)"; }
uint64_t lwkzg_kernel_launches(void) { return lw::launches(); }

int lwkzg_set_option(const char* name, long value) {
  std::lock_guard<std::mutex> lk(g_mu);
  std::string n(name ? name : "");
  if (n == "window_bits") { if (value < 4 || value > 16) return 1; opts().window_bits = value; return 0; }
  if (n == "msm_blocks_per_blob") { if (value < 0 || value > 256 || (value > 64 && (value & (value - 1)))) return 1; opts().msm_blocks_per_blob = value; return 0; }
  if (n == "chunk_blobs") { if (value < 1 || value > (1 << 20)) return 1; opts().chunk_blobs = value; return 0; }
  if (n == "mode") { if (value < 0 || value > 2) return 1; opts().mode = value; return 0; }
  if (n == "msm_algo") { if (value != 0 && value != 1) return 1; opts().msm_algo = value; return 0; }
  if (n == "msm_ba_min_blobs") { if (value < 1) return 1; opts().msm_ba_min_blobs = value; return 0; }
  if (n == "verify_super_blobs") { if (value < 1) return 1; opts().verify_super_blobs = value; return 0; }
  if (n == "lincomb_points_in_g1") { if (value != 0 && value != 1) return 1; opts().lincomb_points_in_g1 = value; return 0; }
  if (n == "share_table") { if (value != 0 && value != 1) return 1; opts().share_table = value; return 0; }
  if (n == "verify_streams") { if (value < 1 || value > 8) return 1; opts().verify_streams = value; return 0; }
  if (n == "verify_split_subgroup") { if (value != 0 && value != 1) return 1; opts().verify_split_subgroup = value; return 0; }
  if (n == "cache_config") { if (value < 0 || value > 3) return 1; opts().cache_config = value; return 0; }
  if (n == "verify_overlap_decode") { if (value != 0 && value != 1) return 1; opts().verify_overlap_decode = value; return 0; }
  if (n == "cell_window_bits") { if (value < 4 || value > 14) return 1; opts().cell_window_bits = value; return 0; }
  if (n == "cell_chunk_blobs") { if (value < 1 || value > 65536) return 1; opts().cell_chunk_blobs = value; return 0; }
  if (n == "msm_ba_variant") { if (value < 0 || value >= msm_ba_num_variants()) return 1; msm_ba_set_variant((int)value); return 0; }
  return 1;
}
long lwkzg_get_option(const char* name) {
  std::lock_guard<std::mutex> lk(g_mu);
  std::string n(name ? name : "");
  if (n == "window_bits") return opts().window_bits;
  if (n == "msm_blocks_per_blob") return opts().msm_blocks_per_blob;
  if (n == "chunk_blobs") return opts().chunk_blobs;
  if (n == "mode") return opts().mode;
  if (n == "msm_algo") return opts().msm_algo;
  if (n == "msm_ba_min_blobs") return opts().msm_ba_min_blobs;
  if (n == "verify_super_blobs") return opts().verify_super_blobs;
  if (n == "lincomb_points_in_g1") return opts().lincomb_points_in_g1;
  if (n == "share_table") return opts().share_table;
  if (n == "verify_streams") return opts().verify_streams;
  if (n == "verify_split_subgroup") return opts().verify_split_subgroup;
  if (n == "cache_config") return opts().cache_config;
  if (n == "verify_overlap_decode") return opts().verify_overlap_decode;
  if (n == "cell_window_bits") return opts().cell_window_bits;
  if (n == "cell_chunk_blobs") return opts().cell_chunk_blobs;
  if (n == "msm_ba_threads") return msm_ba_threads();   // read-only: threads per blob of the batched-affine kernel
  if (n == "msm_ba_slots") return msm_ba_slots();       // read-only: affine accumulators per thread
  return -1;
}

double lwkzg_imad_peak(int variant) { return lw::run_imad_peak(variant); }

C_KZG_RET load_trusted_setup(KZGSettings* out, const uint8_t* g1_bytes, size_t n1, const uint8_t* g2_bytes, size_t n2) {
  if (n1 != TRUSTED_SETUP_NUM_G1_POINTS || n2 != TRUSTED_SETUP_NUM_G2_POINTS) return C_KZG_BADARGS;  // lib.rs:716-718
  if (!out || !g1_bytes || !g2_bytes) return C_KZG_ERROR;
  return settings_from_compressed(out, g1_bytes, n1, g2_bytes, n2);
}

C_KZG_RET load_trusted_setup_file(KZGSettings* out, FILE* in) {
  if (!out || !in) return C_KZG_ERROR;
  std::string contents;
  char buf[65536];
  size_t got;
  while ((got = fread(buf, 1, sizeof(buf), in)) > 0) contents.append(buf, got);
  // str::lines(): split on '\n', strip one trailing '\r'
  std::vector<std::string> lines;
  size_t pos = 0;
  while (pos < contents.size()) {
    size_t nl = contents.find('\n', pos);
    std::string ln = contents.substr(pos, nl == std::string::npos ? std::string::npos : nl - pos);
    if (!ln.empty() && ln.back() == '\r') ln.pop_back();
    lines.push_back(ln);
    if (nl == std::string::npos) break;
    pos = nl + 1;
  }
  size_t n1 = 0, n2 = 0;
  if (lines.size() < 2 || !parse_usize(lines[0], n1) || !parse_usize(lines[1], n2)) { set_err("invalid trusted setup header"); return C_KZG_ERROR; }
  if (n1 > (1u << 20) || n2 > (1u << 20)) { set_err("implausible point counts"); return C_KZG_ERROR; }
  // srs.rs:54-79: lines beyond n1+n2 are ignored, a short file just yields fewer points
  size_t avail = lines.size() - 2;
  size_t m1 = std::min(n1, avail), m2 = std::min(n2, avail - m1);
  std::vector<uint8_t> g1b(m1 * 48 + 1), g2b(m2 * 96 + 1);
  for (size_t i = 0; i < m1; i++)
    if (!hex_line(lines[2 + i], &g1b[i * 48], 48)) { set_err("bad G1 hex line"); return C_KZG_ERROR; }
  for (size_t i = 0; i < m2; i++)
    if (!hex_line(lines[2 + m1 + i], &g2b[i * 96], 96)) { set_err("bad G2 hex line"); return C_KZG_ERROR; }
  return settings_from_compressed(out, g1b.data(), m1, g2b.data(), m2);
}

C_KZG_RET free_trusted_setup(KZGSettings* s) {
  if (!s) return C_KZG_OK;
  if (s->fs) {
    Ctx* c = reinterpret_cast<Ctx*>(s->fs);
    if (c->magic == CTX_MAGIC) destroy_ctx_locked(c);
    s->fs = nullptr;
  } else {
    std::lock_guard<std::mutex> lk(g_lazy_mu);
    for (auto j = lazy_map().begin(); j != lazy_map().end();) {
      if (j->first.g1 == s->g1_values && j->first.g2 == s->g2_values) {
        destroy_ctx_locked(j->second);
        j = lazy_map().erase(j);
      } else {
        ++j;
      }
    }
  }
  free(s->g1_values);  // lib.rs:824-825
  free(s->g2_values);
  s->g1_values = nullptr;
  s->g2_values = nullptr;
  return C_KZG_OK;
}

// ---- batch API (host buffers)
C_KZG_RET lwkzg_blob_to_kzg_commitment_batch(KZGCommitment* out, const Blob* blobs, size_t n, const KZGSettings* s, int* status) {
  return host_batch(Mode::Commit, s, n, blobs, nullptr, nullptr, out, nullptr, nullptr, status);
}
C_KZG_RET lwkzg_compute_blob_kzg_proof_batch(KZGProof* out, const Blob* blobs, const Bytes48* commitments, size_t n, const KZGSettings* s, int* status) {
  return host_batch(Mode::BlobProof, s, n, blobs, commitments, nullptr, nullptr, out, nullptr, status);
}
C_KZG_RET lwkzg_compute_kzg_proof_batch(KZGProof* proofs, Bytes32* ys, const Blob* blobs, const Bytes32* zs, size_t n, const KZGSettings* s, int* status) {
  return host_batch(Mode::PointProof, s, n, blobs, nullptr, zs, nullptr, proofs, ys, status);
}
C_KZG_RET lwkzg_commit_and_prove_batch(KZGCommitment* commitments, KZGProof* proofs, const Blob* blobs, size_t n, const KZGSettings* s, int* status) {
  return host_batch(Mode::CommitProve, s, n, blobs, nullptr, nullptr, commitments, proofs, nullptr, status);
}

// ---- batch API (device buffers)
C_KZG_RET lwkzg_commit_and_prove_batch_device(void* d_commitments, void* d_proofs, const void* d_blobs, size_t n, const KZGSettings* s, void* stream, void* d_status) {
  return device_batch(Mode::CommitProve, s, n, d_blobs, nullptr, d_commitments, d_proofs, d_status, (cudaStream_t)stream);
}
C_KZG_RET lwkzg_blob_to_kzg_commitment_batch_device(void* d_commitments, const void* d_blobs, size_t n, const KZGSettings* s, void* stream, void* d_status) {
  return device_batch(Mode::Commit, s, n, d_blobs, nullptr, d_commitments, nullptr, d_status, (cudaStream_t)stream);
}
C_KZG_RET lwkzg_compute_blob_kzg_proof_batch_device(void* d_proofs, const void* d_blobs, const void* d_commitments, size_t n, const KZGSettings* s, void* stream, void* d_status) {
  return device_batch(Mode::BlobProof, s, n, d_blobs, d_commitments, nullptr, d_proofs, d_status, (cudaStream_t)stream);
}

C_KZG_RET lwkzg_synth_blobs_device(void* d_blobs, uint64_t first_blob, size_t n, void* stream) {
  lw::launch_synth_blobs(d_blobs, first_blob, n, (cudaStream_t)stream);
  return cudaGetLastError() == cudaSuccess ? C_KZG_OK : C_KZG_ERROR;
}

// ---- the c-kzg-4844 single-item entry points = the n = 1 case of the batch drivers
C_KZG_RET blob_to_kzg_commitment(KZGCommitment* out, const Blob* blob, const KZGSettings* s) {
  return host_batch(Mode::Commit, s, 1, blob, nullptr, nullptr, out, nullptr, nullptr, nullptr);
}
C_KZG_RET compute_kzg_proof(KZGProof* proof_out, Bytes32* y_out, const Blob* blob, const Bytes32* z_bytes, const KZGSettings* s) {
  return host_batch(Mode::PointProof, s, 1, blob, nullptr, z_bytes, nullptr, proof_out, y_out, nullptr);
}
C_KZG_RET compute_blob_kzg_proof(KZGProof* out, const Blob* blob, const Bytes48* commitment_bytes, const KZGSettings* s) {
  return host_batch(Mode::BlobProof, s, 1, blob, commitment_bytes, nullptr, nullptr, out, nullptr, nullptr);
}

// ---- verification
C_KZG_RET verify_kzg_proof(bool* ok, const Bytes48* commitment_bytes, const Bytes32* z_bytes, const Bytes32* y_bytes, const Bytes48* proof_bytes,
                           const KZGSettings* s) {
  if (!ok) return C_KZG_ERROR;
  *ok = false;  // lib.rs:415-417
  Ctx* c = ctx_of(s);
  if (!c) return C_KZG_ERROR;
  CtxLock L(c);
  c->vb_n = 0;   // the workspace no longer holds a phase-1 result
  if (!c->srs_valid || !c->g2_valid) { set_err("SRS re-hydration failed"); return C_KZG_ERROR; }
  if (!vb_reserve(c, 1)) return C_KZG_ERROR;
  cudaStream_t s0 = c->slot[0].st;
  uint8_t zy[64];
  memcpy(zy, z_bytes, 32);
  memcpy(zy + 32, y_bytes, 32);
  bool good = [&]() -> bool {
    CU_TRY(cudaMemcpyAsync(c->vb_cin.p, commitment_bytes, 48, cudaMemcpyHostToDevice, s0));
    CU_TRY(cudaMemcpyAsync(c->vb_pin.p, proof_bytes, 48, cudaMemcpyHostToDevice, c->hash_st));
    CU_TRY(cudaMemcpyAsync(c->vb_zy_in.p, zy, 64, cudaMemcpyHostToDevice, s0));
    const bool le = c->lagrange(), be = c->be_wire();
    // the two point decompressions (sqrt + subgroup check, ~2 ms each on one thread) run side by side
    // (decoding only: the r-torsion tests, two thirds of a decompression, run inside the verification kernel beside
    // its scalar multiplications)
    launch_g1_decompress(c->vb_caff.p, nullptr, (int*)c->vb_status.p, c->vb_cin.p, 1, s0, le, false);
    launch_g1_decompress(c->vb_piaff.p, nullptr, (int*)c->vb_tuples.p, c->vb_pin.p, 1, c->hash_st, le, false);
    CU_TRY(cudaEventRecord(c->ev_hash, c->hash_st));
    CU_TRY(cudaStreamWaitEvent(s0, c->ev_hash, 0));
    launch_status_or((int*)c->vb_status.p, (const int*)c->vb_tuples.p, 1, s0);
    if (le) {
      CU_TRY(cudaMemsetAsync(c->vb_tuples.p, 0, 2 * sizeof(int), s0));
      launch_le_fr_parse(c->vb_z.p, (int*)c->vb_tuples.p, c->vb_zy_in.p, 1, s0, be);
      launch_le_fr_parse(c->vb_y.p, (int*)c->vb_tuples.p + 1, (const uint8_t*)c->vb_zy_in.p + 32, 1, s0, be);
      launch_status_or((int*)c->vb_status.p, (const int*)c->vb_tuples.p, 1, s0);
      launch_status_or((int*)c->vb_status.p, (const int*)c->vb_tuples.p + 1, 1, s0);
    } else {
      launch_fr_from_be(c->vb_z.p, c->vb_zy_in.p, 1, s0);
      launch_fr_from_be(c->vb_y.p, (const uint8_t*)c->vb_zy_in.p + 32, 1, s0);
    }
    return true;
  }();
  if (!good) return C_KZG_ERROR;
  // no host round trip in between: the verification kernel is queued right behind the decoding (a rejected point is
  // decoded as infinity, so it runs on well-defined values either way) and the status word -- decode errors,
  // non-canonical field elements, points outside G1 -- is read together with the result
  int bad = 0;
  bool res = false;
  if (!verify_single_from_workspace(c, res, true, &bad)) return C_KZG_ERROR;
  if (bad) { set_err("invalid commitment, proof or field element bytes"); return bad_code(bad); }
  *ok = res;
  return C_KZG_OK;
}

static C_KZG_RET verify_blob_single(bool* ok, const Blob* blob, const Bytes48* commitment_bytes, const Bytes48* proof_bytes, const KZGSettings* s,
                                    bool dev_inputs) {
  if (!ok) return C_KZG_ERROR;
  *ok = false;  // lib.rs:463-465
  Ctx* c = ctx_of(s);
  if (!c) return C_KZG_ERROR;
  CtxLock L(c);
  if (!verify_prepare(c, blob, commitment_bytes, proof_bytes, 1, false, dev_inputs, true)) return C_KZG_ERROR;
  int bad = 0;
  if (!first_bad_status(c, 1, bad)) return C_KZG_ERROR;
  if (bad) { set_err("invalid commitment, proof or field element bytes"); return bad_code(bad); }
  bool res = false;
  c->vb_n = 0;
  if (!verify_single_from_workspace(c, res, true, &bad)) return C_KZG_ERROR;
  if (bad) { set_err("commitment or proof is not in G1"); return bad_code(bad); }
  *ok = res;
  return C_KZG_OK;
}

// ---- the three phases of a batched verification, on a context whose lock the caller holds.  The batched call, the
// same call over several GPUs and the distributed phase entry points below are all assembled from these.

// Phase 1: per-item preparation into the workspace (hash_r: the batch challenge r into vb_r as well), the first invalid
// item's code, then -- when tuples_out is given -- the 160-byte tuples copied there on s0 and waited for.
static C_KZG_RET phase1_on(Ctx* c, const Blob* blobs, const Bytes48* commitments, const Bytes48* proofs, size_t n, bool inputs_on_device,
                           bool hash_r, void* tuples_out, bool out_on_device) {
  if (!verify_prepare(c, blobs, commitments, proofs, n, hash_r, inputs_on_device)) return C_KZG_ERROR;
  int bad = 0;
  if (!first_bad_status(c, n, bad)) return C_KZG_ERROR;
  if (bad) { set_err("invalid commitment, proof or field element bytes"); return bad_code(bad); }
  if (!tuples_out) return C_KZG_OK;
  // on the context's stream and waited for: a plain cudaMemcpy between device buffers may still be running when it
  // returns, on the legacy stream, which the library's non-blocking streams (phase 2 reads these tuples) do not wait for
  cudaStream_t s0 = c->slot[0].st;
  if (cudaMemcpyAsync(tuples_out, c->vb_tuples.p, n * 160, out_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s0) != cudaSuccess ||
      cudaStreamSynchronize(s0) != cudaSuccess) {
    set_err("tuple copy failed");
    return C_KZG_ERROR;
  }
  return C_KZG_OK;
}

// Phase 2: the partial sums of items [first, first + count) with weights r^(first + i), r already in vb_r, into
// vb_partial.  When partial_out is given, the 288 bytes are copied there and waited for.
static bool phase2_on(Ctx* c, size_t first, size_t count, void* partial_out, bool out_on_device) {
  if (!c->vb_partial.ensure(288) || !c->vb_scratch.ensure(batch_partials_scratch_bytes((int)std::max<size_t>(count, 1)))) return false;
  cudaStream_t s0 = c->slot[0].st;
  launch_batch_partials(c->vb_partial.p, c->vb_r.p, c->vb_caff.p, c->vb_piaff.p, c->vb_z.p, c->vb_y.p, first, (int)count, c->vb_scratch.p, s0,
                        c->slot[0].aux, c->slot[0].ev_fork, c->slot[0].ev_aux);
  if (!partial_out) return true;
  CU_TRY(cudaMemcpyAsync(partial_out, c->vb_partial.p, 288, out_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s0));
  CU_TRY(cudaStreamSynchronize(s0));
  CU_TRY(cudaGetLastError());
  return true;
}

// Phase 3: the sum of `count` partial sums (host or device memory) and the 2-pairing check
static C_KZG_RET phase3_on(Ctx* c, bool* ok, const void* partials288, bool on_device, size_t count) {
  cudaStream_t s0 = c->slot[0].st;
  DevBuf staged;   // the partial sums, when they come from host memory
  if (!on_device && !staged.ensure(std::max<size_t>(count, 1) * 288)) { set_err("cudaMalloc failed"); return C_KZG_MALLOC; }
  int okv = 0;
  bool good = [&]() -> bool {
    if (!c->vb_ok.ensure(sizeof(int))) return false;
    if (!on_device) CU_TRY(cudaMemcpyAsync(staged.p, partials288, count * 288, cudaMemcpyHostToDevice, s0));
    launch_batch_final((int*)c->vb_ok.p, on_device ? partials288 : staged.p, (int)count, c->d_prep0, c->d_prep1, s0);
    CU_TRY(cudaMemcpyAsync(&okv, c->vb_ok.p, sizeof(int), cudaMemcpyDeviceToHost, s0));
    CU_TRY(cudaStreamSynchronize(s0));
    CU_TRY(cudaGetLastError());
    return true;
  }();
  if (!good) return C_KZG_ERROR;
  *ok = okv != 0;
  return C_KZG_OK;
}

// verify_blob_kzg_proof_batch over the GPUs of lwkzg_set_devices (SURVEY 8e): the distributed phases, with one host
// thread per device instead of one process.  Phase 1 on every shard; the tuples meet in host memory and the primary
// device derives r (one sequential hash over ALL tuples, utils.rs:166-206) and hands it to the others; phase 2 on
// every shard; phase 3 on the primary device over the g partial sums.  Both exchanges are a few hundred KB at most.
// Group addition is exact: the boolean does not depend on the sharding.
static C_KZG_RET verify_blob_batch_multi(bool* ok, const Blob* blobs, const Bytes48* cs, const Bytes48* ps, size_t n, std::vector<Ctx*>& ctxs) {
  const size_t g = ctxs.size();
  Ctx* c0 = ctxs[0];
  std::vector<std::unique_lock<std::mutex>> locks;
  for (Ctx* c : ctxs) locks.emplace_back(c->mu);
  std::vector<uint8_t> tuples(n * 160), partials(g * 288);
  C_KZG_RET rc = for_shards(ctxs, n, [&](size_t, Ctx* c, size_t first, size_t count) {
    return phase1_on(c, blobs + first, cs + first, ps + first, count, false, false, tuples.data() + first * 160, false);
  });
  uint32_t r_host[8];
  if (rc == C_KZG_OK) {
    DeviceGuard dg(c0->device);
    cudaStream_t s0 = c0->slot[0].st;
    DevBuf all;
    auto derive_r = [&]() -> bool {
      CU_TRY(cudaMemcpyAsync(all.p, tuples.data(), n * 160, cudaMemcpyHostToDevice, s0));
      launch_batch_challenge(c0->vb_r.p, all.p, n, s0, c0->mode);
      CU_TRY(cudaMemcpyAsync(r_host, c0->vb_r.p, 32, cudaMemcpyDeviceToHost, s0));
      CU_TRY(cudaStreamSynchronize(s0));
      return true;
    };
    if (!all.ensure(n * 160)) { set_err("cudaMalloc failed"); rc = C_KZG_MALLOC; }
    else if (!derive_r()) rc = C_KZG_ERROR;
  }
  if (rc == C_KZG_OK) {
    rc = for_shards(ctxs, n, [&](size_t k, Ctx* c, size_t first, size_t count) {
      const bool good = cudaMemcpyAsync(c->vb_r.p, r_host, 32, cudaMemcpyHostToDevice, c->slot[0].st) == cudaSuccess &&
                        phase2_on(c, first, count, partials.data() + k * 288, false);
      return good ? C_KZG_OK : C_KZG_ERROR;
    });
  }
  for (Ctx* c : ctxs) c->vb_n = 0;
  if (rc != C_KZG_OK) return rc;
  DeviceGuard dg(c0->device);
  return phase3_on(c0, ok, partials.data(), false, g);
}

static C_KZG_RET verify_blob_batch(bool* ok, const Blob* blobs, const Bytes48* commitments_bytes, const Bytes48* proofs_bytes, size_t n,
                                   const KZGSettings* s, bool dev_inputs) {
  if (!ok) return C_KZG_ERROR;
  *ok = false;  // lib.rs:533-535
  if (n == 0) {
    // lib.rs:538-543: the reference rejects an empty batch; c-kzg (MODE_CKZG_LE) accepts it
    Ctx* c0 = ctx_of(s);
    if (c0 && c0->lagrange()) *ok = true;
    return C_KZG_OK;
  }
  if (n == 1) return verify_blob_single(ok, blobs, commitments_bytes, proofs_bytes, s, dev_inputs);  // lib.rs:544
  Ctx* c = ctx_of(s);
  if (!c) return C_KZG_ERROR;
  if (!dev_inputs) {
    std::vector<Ctx*> ctxs = ctxs_for(c, n);
    if (ctxs.size() > 1) return verify_blob_batch_multi(ok, blobs, commitments_bytes, proofs_bytes, n, ctxs);
  }
  CtxLock L(c);
  static const bool trace = getenv("LWKZG_VERIFY_TRACE") != nullptr;
  auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t0 = now();
  if (C_KZG_RET rc = phase1_on(c, blobs, commitments_bytes, proofs_bytes, n, dev_inputs, true, nullptr, false)) return rc;   // leaves r in vb_r
  const double t1 = now();
  if (!phase2_on(c, 0, n, nullptr, false) || phase3_on(c, ok, c->vb_partial.p, true, 1) != C_KZG_OK) {
    set_err("CUDA failure in batch verification");
    return C_KZG_ERROR;
  }
  c->vb_n = 0;
  if (trace) fprintf(stderr, "[lwkzg] verify batch n=%zu: prepare + status %.2f ms, partials+pairing %.2f ms\n", n, t1 - t0, now() - t1);
  return C_KZG_OK;
}

C_KZG_RET verify_blob_kzg_proof(bool* ok, const Blob* blob, const Bytes48* commitment_bytes, const Bytes48* proof_bytes, const KZGSettings* s) {
  return verify_blob_single(ok, blob, commitment_bytes, proof_bytes, s, false);
}

C_KZG_RET verify_blob_kzg_proof_batch(bool* ok, const Blob* blobs, const Bytes48* commitments_bytes, const Bytes48* proofs_bytes, size_t n,
                                      const KZGSettings* s) {
  return verify_blob_batch(ok, blobs, commitments_bytes, proofs_bytes, n, s, false);
}

// the same check with blobs, commitments and proofs already in device memory (the boolean still comes back to the host)
C_KZG_RET lwkzg_verify_blob_kzg_proof_batch_device(bool* ok, const void* d_blobs, const void* d_commitments, const void* d_proofs, size_t n,
                                                   const KZGSettings* s) {
  return verify_blob_batch(ok, (const Blob*)d_blobs, (const Bytes48*)d_commitments, (const Bytes48*)d_proofs, n, s, true);
}

// ---- multi-GPU batched verification phases (one process per GPU; the caller runs the two all-gathers)
static C_KZG_RET phase1_impl(uint8_t* tuples_out, bool out_on_device, const Blob* blobs, const Bytes48* commitments, const Bytes48* proofs,
                             size_t n_local, bool inputs_on_device, const KZGSettings* s) {
  Ctx* c = ctx_of(s);
  if (!c) return C_KZG_ERROR;
  CtxLock L(c);
  c->vb_n = 0;
  if (n_local == 0) return C_KZG_OK;
  return phase1_on(c, blobs, commitments, proofs, n_local, inputs_on_device, false, tuples_out, out_on_device);
}
C_KZG_RET lwkzg_verify_batch_phase1(uint8_t* tuples160, const Blob* blobs, const Bytes48* commitments, const Bytes48* proofs, size_t n_local,
                                    const KZGSettings* s) {
  return phase1_impl(tuples160, false, blobs, commitments, proofs, n_local, false, s);
}
C_KZG_RET lwkzg_verify_batch_phase1_device(void* d_tuples160, const void* blobs, const void* commitments, const void* proofs, size_t n_local,
                                           int inputs_on_device, const KZGSettings* s) {
  return phase1_impl((uint8_t*)d_tuples160, true, (const Blob*)blobs, (const Bytes48*)commitments, (const Bytes48*)proofs, n_local,
                     inputs_on_device != 0, s);
}

static C_KZG_RET phase2_impl(uint8_t* partial288, const uint8_t* all_tuples160, bool on_device, size_t n_total, size_t first, size_t n_local,
                             const KZGSettings* s) {
  Ctx* c = ctx_of(s);
  if (!c) return C_KZG_ERROR;
  CtxLock L(c);
  if (c->vb_n != n_local || first + n_local > n_total) { set_err("phase2 does not match the preceding phase1"); return C_KZG_BADARGS; }
  cudaStream_t s0 = c->slot[0].st;
  DevBuf staged;   // all tuples, when they come from host memory
  if (!on_device && !staged.ensure(std::max<size_t>(n_total, 1) * 160)) { set_err("cudaMalloc failed"); return C_KZG_MALLOC; }
  bool good = [&]() -> bool {
    if (!on_device) CU_TRY(cudaMemcpyAsync(staged.p, all_tuples160, n_total * 160, cudaMemcpyHostToDevice, s0));
    if (!c->vb_r.ensure(32)) return false;
    launch_batch_challenge(c->vb_r.p, on_device ? (const void*)all_tuples160 : staged.p, n_total, s0, c->mode);
    return phase2_on(c, first, n_local, partial288, on_device);
  }();
  return good ? C_KZG_OK : C_KZG_ERROR;
}
C_KZG_RET lwkzg_verify_batch_phase2(uint8_t* partial288, const uint8_t* all_tuples160, size_t n_total, size_t first, size_t n_local,
                                    const KZGSettings* s) {
  return phase2_impl(partial288, all_tuples160, false, n_total, first, n_local, s);
}
C_KZG_RET lwkzg_verify_batch_phase2_device(void* d_partial288, const void* d_all_tuples160, size_t n_total, size_t first, size_t n_local,
                                           const KZGSettings* s) {
  return phase2_impl((uint8_t*)d_partial288, (const uint8_t*)d_all_tuples160, true, n_total, first, n_local, s);
}

static C_KZG_RET phase3_impl(bool* ok, const uint8_t* partials288, bool on_device, size_t n_ranks, const KZGSettings* s) {
  if (!ok) return C_KZG_ERROR;
  *ok = false;
  Ctx* c = ctx_of(s);
  if (!c) return C_KZG_ERROR;
  CtxLock L(c);
  if (!c->srs_valid || !c->g2_valid) { set_err("SRS re-hydration failed"); return C_KZG_ERROR; }
  return phase3_on(c, ok, partials288, on_device, n_ranks);
}
C_KZG_RET lwkzg_verify_batch_phase3(bool* ok, const uint8_t* partials288, size_t n_ranks, const KZGSettings* s) {
  return phase3_impl(ok, partials288, false, n_ranks, s);
}
C_KZG_RET lwkzg_verify_batch_phase3_device(bool* ok, const void* d_partials288, size_t n_ranks, const KZGSettings* s) {
  return phase3_impl(ok, (const uint8_t*)d_partials288, true, n_ranks, s);
}

// ---- devices: after lwkzg_set_devices(ids, n) the host-buffer batch calls (commit / proof / commit+proof batches,
// verify_blob_kzg_proof_batch) shard their items over the listed GPUs from this one process
int lwkzg_set_devices(const int* ids, int n) {
  int have = 0;
  if (n < 0 || (n > 0 && !ids) || cudaGetDeviceCount(&have) != cudaSuccess) return 1;
  std::vector<int> v;
  for (int i = 0; i < n; i++) {
    if (ids[i] < 0 || ids[i] >= have) return 1;
    for (int d : v)
      if (d == ids[i]) return 1;
    v.push_back(ids[i]);
  }
  std::lock_guard<std::mutex> lk(g_mu);
  device_list() = v;
  return 0;
}
int lwkzg_get_devices(int* ids, int cap) {
  std::lock_guard<std::mutex> lk(g_mu);
  const int n = (int)device_list().size();
  for (int i = 0; i < n && i < cap; i++) ids[i] = device_list()[i];
  return n;
}

// ---- measurement hook: the dominant kernel alone, timed with CUDA events on
// the stream it is launched on (bench.py's roofline leg)
double lwkzg_bench_msm_kernel(const void* d_blobs, size_t n, int blocks_per_blob, int iters, const KZGSettings* s) {
  Ctx* c = ctx_of(s);
  if (!c || !c->srs_valid || n == 0 || iters <= 0) return -1.0;
  CtxLock L(c);
  Slot& sl = c->slot[0];
  int bpb = blocks_per_blob > 0 ? blocks_per_blob : auto_bpb((int)n);
  cudaStreamSynchronize(sl.st);
  if (!reserve(slot_buffers(sl, (int)n, bpb, false))) return -1.0;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  auto run = [&]() {
    if (blocks_per_blob > 0) launch_msm_gather(sl.partials.p, c->d_table, c->c, d_blobs, true, (int)n, bpb, sl.st);   // explicit: the XYZZ kernel
    else run_msm(sl, c, d_blobs, true, (int)n, bpb, sl.st);
  };
  run();  // warm-up
  cudaEventRecord(e0, sl.st);
  for (int i = 0; i < iters; i++) run();
  cudaEventRecord(e1, sl.st);
  cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (cudaGetLastError() != cudaSuccess) return -1.0;
  return (double)ms / iters;
}
// measurement hook: the last step of a batched verification alone (fold of the partial sums + 2-pairing check) on
// the partial sums the previous batched verification on these settings left in the workspace
double lwkzg_bench_pairing(int iters, const KZGSettings* s) {
  Ctx* c = ctx_of(s);
  if (!c || !c->srs_valid || !c->g2_valid || iters <= 0 || !c->vb_partial.p || !c->vb_ok.p) return -1.0;
  CtxLock L(c);
  cudaStream_t s0 = c->slot[0].st;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  launch_batch_final((int*)c->vb_ok.p, c->vb_partial.p, 1, c->d_prep0, c->d_prep1, s0);
  cudaEventRecord(e0, s0);
  for (int i = 0; i < iters; i++) launch_batch_final((int*)c->vb_ok.p, c->vb_partial.p, 1, c->d_prep0, c->d_prep1, s0);
  cudaEventRecord(e1, s0);
  cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (cudaGetLastError() != cudaSuccess) return -1.0;
  return (double)ms / iters;
}
// test hook: the batch challenge r (canonical, 8 little-endian u32) left in the workspace by the last batched
// verification / phase 2 on these settings
C_KZG_RET lwkzg_debug_batch_challenge(uint8_t* out32, const KZGSettings* s) {
  Ctx* c = ctx_of(s);
  if (!c || !out32 || !c->vb_r.p) return C_KZG_ERROR;
  CtxLock L(c);
  if (cudaMemcpy(out32, c->vb_r.p, 32, cudaMemcpyDeviceToHost) != cudaSuccess) { set_err("D2H failed"); return C_KZG_ERROR; }
  return C_KZG_OK;
}
int lwkzg_window_bits(const KZGSettings* s) {
  Ctx* c = ctx_of(s);
  return c ? c->c : -1;
}
void lwkzg_debug_stage_copy(void* dst, const void* src, size_t bytes) { HostStager::get().copy(dst, src, bytes); }
int lwkzg_table_share(const KZGSettings* s) {
  Ctx* c = ctx_of(s);
  return c ? c->table_share : -1;
}

// ---- measurement hook for BASELINE config 5 (variable-base MSM size sweep):
// n synthetic points (pseudo-randomly chosen fixed-base table entries, so their
// discrete logs are known to the tests) x n synthetic scalars, all generated and
// kept on the device; the MSM pipeline alone is timed with CUDA events.
double lwkzg_bench_var_msm(Bytes48* out, size_t n, int iters, uint64_t seed, const KZGSettings* s) {
  Ctx* c = ctx_of(s);
  if (!c || !c->srs_valid || !out || n == 0 || iters <= 0) return -1.0;
  CtxLock L(c);
  cudaStream_t st = c->slot[0].st;
  void *d_pts = nullptr, *d_sc = nullptr, *d_scratch = nullptr, *d_out = nullptr;
  double ms_per = -1.0;
  bool good = [&]() -> bool {
    CU_TRY(cudaMalloc(&d_pts, n * 96));
    CU_TRY(cudaMalloc(&d_sc, n * 32));
    CU_TRY(cudaMalloc(&d_scratch, var_msm_scratch_bytes(n)));
    CU_TRY(cudaMalloc(&d_out, 48));
    unsigned long long entries = table_entries(c->c, N_POINTS);
    launch_var_msm_synth(d_pts, d_sc, c->d_table, entries, seed, n, st);
    // the synthetic points are entries of the fixed-base table, i.e. multiples of validated SRS points: in G1
    launch_var_msm(d_out, d_pts, d_sc, n, d_scratch, st, true);  // warm-up
    cudaEvent_t e0, e1;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    CU_TRY(cudaEventRecord(e0, st));
    for (int i = 0; i < iters; i++) launch_var_msm(d_out, d_pts, d_sc, n, d_scratch, st, true);
    CU_TRY(cudaEventRecord(e1, st));
    CU_TRY(cudaEventSynchronize(e1));
    float ms = 0;
    CU_TRY(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpy(out, d_out, 48, cudaMemcpyDeviceToHost));
    ms_per = (double)ms / iters;
    return true;
  }();
  cudaFree(d_pts); cudaFree(d_sc); cudaFree(d_scratch); cudaFree(d_out);
  return good ? ms_per : -1.0;
}

// ---- generic linear combination (g1_lincomb, lib.rs:241-243)
// The call has no KZGSettings to hang a context on: the device buffers (inputs, MSM scratch, result) and the stream
// live in a per-device workspace that grows to the largest n seen and is reused -- no cudaMalloc / cudaFree and no
// device-wide synchronisation per call.
namespace {
struct LincombWs {
  DevBuf pts, sc, scratch, out;
  cudaStream_t st = nullptr;
  void* h_out = nullptr;   // pinned: 48 result bytes + the bad-point flag
};
std::mutex g_lincomb_mu;
std::map<int, LincombWs>& lincomb_ws() {
  static auto* m = new std::map<int, LincombWs>();   // never destroyed: no cudaFree during static destruction at exit
  return *m;
}
}  // namespace

C_KZG_RET lwkzg_g1_lincomb(Bytes48* out, const uint8_t* points_xy_be, const uint8_t* scalars_be, size_t n) {
  if (!out || (n && (!points_xy_be || !scalars_be))) return C_KZG_ERROR;
  bool in_g1;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    in_g1 = opts().lincomb_points_in_g1 != 0;
  }
  std::lock_guard<std::mutex> lk(g_lincomb_mu);
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { set_err("no CUDA device"); return C_KZG_ERROR; }
  LincombWs& w = lincomb_ws()[dev];
  int bad = 0;
  bool good = [&]() -> bool {
    const size_t nn = std::max<size_t>(n, 1);
    if (!w.st) CU_TRY(cudaStreamCreateWithFlags(&w.st, cudaStreamNonBlocking));
    if (!w.h_out) CU_TRY(cudaMallocHost(&w.h_out, 64));
    if (!w.pts.ensure(nn * 96) || !w.sc.ensure(nn * 32) || !w.scratch.ensure(var_msm_scratch_bytes(nn)) || !w.out.ensure(48)) return false;
    if (n) {
      CU_TRY(cudaMemcpyAsync(w.pts.p, points_xy_be, n * 96, cudaMemcpyHostToDevice, w.st));
      CU_TRY(cudaMemcpyAsync(w.sc.p, scalars_be, n * 32, cudaMemcpyHostToDevice, w.st));
    }
    launch_var_msm(w.out.p, w.pts.p, w.sc.p, n, w.scratch.p, w.st, in_g1);
    CU_TRY(cudaMemcpyAsync(w.h_out, w.out.p, 48, cudaMemcpyDeviceToHost, w.st));
    CU_TRY(cudaMemcpyAsync((uint8_t*)w.h_out + 48, (uint8_t*)w.scratch.p + var_msm_bad_flag_offset(nn, in_g1), sizeof(int), cudaMemcpyDeviceToHost, w.st));
    CU_TRY(cudaStreamSynchronize(w.st));
    CU_TRY(cudaGetLastError());
    memcpy(&bad, (uint8_t*)w.h_out + 48, sizeof(int));
    return true;
  }();
  if (!good) return C_KZG_ERROR;
  if (bad) { set_err("point not on the curve"); return C_KZG_BADARGS; }
  memcpy(out, w.h_out, 48);
  return C_KZG_OK;
}

#include "cells_api.inl"

}  // extern "C"
