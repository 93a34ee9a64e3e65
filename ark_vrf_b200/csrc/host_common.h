// Host-side plumbing shared by the entry points of libavrf_gpu.so: error reporting, per-device state,
// device / pinned buffers, and the background hasher that absorbs a batch's (c_j, s_j) stream
// (reference src/thin.rs:273-279) while the caller keeps pushing.  Included by avrf_gpu.cu only.
#pragma once
#include <cuda_runtime.h>
#include <openssl/evp.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <initializer_list>
#include <mutex>
#include <string>
#include <thread>

#include "../../include/avrf.h"
#include "mbsha512.h"

namespace avrf {

static thread_local std::string g_err;

static int fail(int code, const char* what, const char* detail = "") {
  g_err = std::string(what) + (detail[0] ? ": " : "") + detail;
  return code;
}

#define CK(call)                                                                         \
  do {                                                                                   \
    cudaError_t e__ = (call);                                                            \
    if (e__ != cudaSuccess) {                                                            \
      char buf__[256];                                                                   \
      snprintf(buf__, sizeof buf__, "%s at %s:%d", cudaGetErrorString(e__), __FILE__, __LINE__); \
      return fail(e__ == cudaErrorMemoryAllocation ? AVRF_ERR_NOMEM : AVRF_ERR_CUDA, #call, buf__); \
    }                                                                                    \
  } while (0)

// ---- devices ------------------------------------------------------------------------------
// One process may drive several GPUs (avrf_init_multi).  Every device has the two streams of the
// handle-less entry points; every batch handle remembers its device and owns its own streams.
constexpr int AVRF_MAX_DEV = 16;
struct DevState {
  bool ready = false;
  cudaStream_t stream = nullptr;      // hash-to-curve, outputs, proving, ingest, combine, microbenchmarks
  cudaStream_t copy = nullptr;        // overlapped D2H inside avrf_thin_seed_dev
  int prio_hi = 0;
};
static DevState g_devs[AVRF_MAX_DEV];
static std::atomic<int> g_device{-1};      // default device (avrf_init / first of avrf_init_multi)
static std::atomic<int> g_ndev{0};         // devices initialised
static int g_dev_list[AVRF_MAX_DEV];
static std::mutex g_init_mu;

// The CUDA "current device" is per host thread: cache it so that binding costs nothing when unchanged.
static thread_local int t_bound = -1;
static int bind_device(int dev) {
  if (t_bound != dev) {
    CK(cudaSetDevice(dev));
    t_bound = dev;
  }
  return 0;
}

static int dev_setup(int device) {          // g_init_mu held
  DevState& d = g_devs[device];
  if (d.ready) return 0;
  CK(cudaSetDevice(device));
  t_bound = device;
  CK(cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&d.copy, cudaStreamNonBlocking));
  int lo = 0;
  CK(cudaDeviceGetStreamPriorityRange(&lo, &d.prio_hi));
  d.ready = true;
  g_dev_list[g_ndev++] = device;
  return 0;
}

static int ensure_init() {
  int dev = g_device.load();
  if (dev < 0) {
    int rc = avrf_init(0);
    if (rc) return rc;
    dev = g_device.load();
  }
  return bind_device(dev);
}
static inline cudaStream_t gs() { return g_devs[g_device.load()].stream; }
static inline cudaStream_t gc() { return g_devs[g_device.load()].copy; }

#define NEED_DEVICE()                                                                    \
  do {                                                                                   \
    int rc__ = ensure_init();                                                            \
    if (rc__) return rc__;                                                               \
  } while (0)

// ---- buffers ------------------------------------------------------------------------------
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }       // temporaries in the entry points free their memory on every return path
  // Grow to at least `bytes`; keep the first `keep` bytes (copied on `st`).  The caller guarantees that no
  // other stream still uses the old allocation (quiesce() for batch handles).
  int reserve(size_t bytes, size_t keep = 0, cudaStream_t st = nullptr) {
    if (bytes <= cap) return 0;
    if (!st) st = gs();
    size_t ncap = cap ? cap : 256;
    while (ncap < bytes) ncap += ncap + 256;
    void* q = nullptr;
    CK(cudaMalloc(&q, ncap));
    if (keep && p) CK(cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, st));
    if (p) {
      CK(cudaStreamSynchronize(st));
      cudaFree(p);
    }
    p = q;
    cap = ncap;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  PinBuf() = default;
  PinBuf(const PinBuf&) = delete;
  PinBuf& operator=(const PinBuf&) = delete;
  ~PinBuf() { release(); }
  int reserve(size_t bytes, size_t keep = 0) {
    if (bytes <= cap) return 0;
    void* q = nullptr;
    CK(cudaHostAlloc(&q, bytes, cudaHostAllocPortable));     // portable: usable from every device of the process
    if (keep && p) memcpy(q, p, keep);
    if (p) cudaFreeHost(p);
    p = q;
    cap = bytes;
    return 0;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Events created inside one call and destroyed on every return path.
struct EventPool {
  std::deque<cudaEvent_t> evs;
  ~EventPool() { for (cudaEvent_t e : evs) cudaEventDestroy(e); }
  cudaEvent_t make(unsigned flags = cudaEventDisableTiming) {
    cudaEvent_t e = nullptr;
    if (cudaEventCreateWithFlags(&e, flags) != cudaSuccess) return nullptr;
    evs.push_back(e);
    return e;
  }
};

static inline uint32_t cdiv(size_t a, size_t b) { return (uint32_t)((a + b - 1) / b); }

// ---- SHA-512 on the calling thread --------------------------------------------------------
struct ByteRange {
  const void* p;
  size_t n;
};
// A SHA-512 context that has absorbed `parts`; nullptr (with the error set) when it cannot be allocated.
static EVP_MD_CTX* sha512_begin(std::initializer_list<ByteRange> parts) {
  EVP_MD_CTX* ctx = EVP_MD_CTX_new();
  if (!ctx) { fail(AVRF_ERR_NOMEM, "EVP_MD_CTX_new"); return nullptr; }
  EVP_DigestInit_ex(ctx, EVP_sha512(), nullptr);
  for (const ByteRange& r : parts) if (r.n) EVP_DigestUpdate(ctx, r.p, r.n);
  return ctx;
}
static void sha512_end(EVP_MD_CTX* ctx, uint8_t out[64]) {
  unsigned int outl = 64;
  EVP_DigestFinal_ex(ctx, out, &outl);
  EVP_MD_CTX_free(ctx);
}
static int sha512(std::initializer_list<ByteRange> parts, uint8_t out[64]) {
  EVP_MD_CTX* ctx = sha512_begin(parts);
  if (!ctx) return AVRF_ERR_NOMEM;
  sha512_end(ctx, out);
  return 0;
}

// ---- hasher -------------------------------------------------------------------------------
// The batch seed is ONE serial SHA-512 over SUITE_ID || 0x50 || (c_j, s_j)... (src/thin.rs:273-279).  A Hasher
// owns that running hash, a pinned staging area the device->host copies of the stream land in, and a thread
// that absorbs the staged chunks, in the order they were queued, as soon as their copies complete - so the
// pushing thread never waits for the hash.  One Hasher per batch handle, or one for all the shards of a
// multi-GPU batch (the chunks are then queued in global proof order).
class Hasher {
 public:
  explicit Hasher(int device) : device_(device) {}
  ~Hasher() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      stop_ = true;
    }
    cv_.notify_all();
    if (th_.joinable()) th_.join();
    if (ctx_) EVP_MD_CTX_free(ctx_);
    if (mb_ && lane_ >= 0) mb_->release(lane_);
  }
  // Hand the hashing to a shared multi-buffer thread (batch server); call before the first begin().
  void use_multibuffer(MbSha512* mb) {
    int lane = mb->acquire();
    if (lane >= 0) { mb_ = mb; lane_ = lane; }
  }
  // Start a new stream: waits for queued work, resets the hash and absorbs `prefix`.
  int begin(const unsigned char* prefix, size_t n) {
    drain();
    head_ = 0;
    queued_bytes_ = 0;
    hash_ms_ = 0;
    if (mb_) {
      mb_->reset(lane_);
      memcpy(prefix_, prefix, n);          // must stay valid until absorbed
      mb_->update(lane_, prefix_, n);
    } else {
      if (!ctx_) ctx_ = EVP_MD_CTX_new();
      if (!ctx_) return fail(AVRF_ERR_NOMEM, "EVP_MD_CTX_new");
      EVP_DigestInit_ex(ctx_, EVP_sha512(), nullptr);
      EVP_DigestUpdate(ctx_, prefix, n);
    }
    return 0;
  }
  // `len` bytes of pinned staging for the next chunk (nullptr on allocation failure).  The area is a bump
  // allocator over one pinned block: when it wraps or grows, queued chunks are absorbed first.
  uint8_t* stage(size_t len) {
    if (head_ + len > pin_.cap) {
      drain();
      if (len > pin_.cap && pin_.reserve(len + (len >> 2) + 4096)) return nullptr;
      head_ = 0;
    }
    uint8_t* p = pin_.as<uint8_t>() + head_;
    head_ += (len + 63) & ~(size_t)63;
    return p;
  }
  int reserve_stage(size_t bytes) {
    if (bytes <= pin_.cap) return 0;
    drain();
    head_ = 0;
    return pin_.reserve(bytes);
  }
  // Absorb `len` bytes at `p` (staging memory) once `ev` has completed.  Takes ownership of `ev` (may be null).
  void enqueue(cudaEvent_t ev, const uint8_t* p, size_t len) {
    {
      std::lock_guard<std::mutex> lk(mu_);
      if (!th_.joinable()) th_ = std::thread(&Hasher::run, this);
      q_.push_back(Job{ev, p, len});
      queued_bytes_ += len;
    }
    cv_.notify_one();
  }
  void drain() {
    std::unique_lock<std::mutex> lk(mu_);
    idle_.wait(lk, [&] { return q_.empty() && !busy_; });
    lk.unlock();
    if (mb_) mb_->sync(lane_);
  }
  // SHA-512 of everything absorbed so far; the stream can continue afterwards (verify is repeatable).
  int digest(uint8_t out[64]) {
    drain();
    if (err_) return fail(AVRF_ERR_CUDA, "hasher thread", cudaGetErrorString(err_));
    if (mb_) {
      mb_->digest(lane_, out);
      return 0;
    }
    if (!ctx_) return fail(AVRF_ERR_STATE, "no hash in progress");
    EVP_MD_CTX* fin = EVP_MD_CTX_new();
    if (!fin) return fail(AVRF_ERR_NOMEM, "EVP_MD_CTX_new");
    unsigned int outl = 64;
    EVP_MD_CTX_copy_ex(fin, ctx_);
    EVP_DigestFinal_ex(fin, out, &outl);
    EVP_MD_CTX_free(fin);
    return 0;
  }
  uint64_t queued_bytes() const { return queued_bytes_; }
  float hash_ms() {
    std::lock_guard<std::mutex> lk(mu_);
    return hash_ms_;
  }
  bool active() const { return ctx_ != nullptr || mb_ != nullptr; }

 private:
  struct Job { cudaEvent_t ev; const uint8_t* p; size_t len; };
  void run() {
    cudaSetDevice(device_);
    for (;;) {
      Job j;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return stop_ || !q_.empty(); });
        if (q_.empty()) return;
        j = q_.front();
        q_.pop_front();
        busy_ = true;
      }
      if (j.ev) {
        cudaError_t e = cudaEventSynchronize(j.ev);
        if (e != cudaSuccess && !err_) err_ = e;
        cudaEventDestroy(j.ev);
      }
      auto t0 = std::chrono::steady_clock::now();
      if (mb_) mb_->update(lane_, j.p, j.len);
      else EVP_DigestUpdate(ctx_, j.p, j.len);
      float ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
      {
        std::lock_guard<std::mutex> lk(mu_);
        busy_ = false;
        hash_ms_ += ms;
      }
      idle_.notify_all();
    }
  }
  int device_;
  EVP_MD_CTX* ctx_ = nullptr;
  MbSha512* mb_ = nullptr;
  int lane_ = -1;
  uint8_t prefix_[64] = {};
  PinBuf pin_;
  size_t head_ = 0;
  uint64_t queued_bytes_ = 0;
  float hash_ms_ = 0;
  cudaError_t err_ = cudaSuccess;
  std::mutex mu_;
  std::condition_variable cv_, idle_;
  std::deque<Job> q_;
  bool busy_ = false, stop_ = false;
  std::thread th_;
};

}  // namespace avrf
