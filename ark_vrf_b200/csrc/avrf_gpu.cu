// libavrf_gpu.so - host pipeline and C ABI (include/avrf.h) of the B200-native Thin-VRF
// batch verifier.  Single translation unit: all kernels are instantiated here for sm_100a
// (msm.cuh: Pippenger; prepare.cuh: per-proof transcripts; feeders.cuh: hash-to-curve, outputs,
// proving, ingest, per-proof verdicts; verify_one.cuh: the single-proof verifier; microbench.cuh: roofline probes).
//
// Path implemented (reference file:line):
//   push / prepare     src/thin.rs:209-243      -> k_prepare   (transcripts, z_i, c, point prep)
//   verify             src/thin.rs:257-325      -> host seed (serial SHA-512) + k_scalars + MSM kernels
//   Verifier::verify   src/thin.rs:131-165      -> k_verify_one (the exact equation, no batch weight)
//   Input::new         src/lib.rs:500-502       -> k_h2c
//   Secret::output     src/lib.rs:391-393       -> k_scalar_mul
//   Prover::prove      src/thin.rs:111-129      -> k_prove      (synthetic-input generator)
//   pedersen::Prover::prove      src/pedersen.rs:136-186 -> k_prove_ped
//   pedersen::Verifier::verify   src/pedersen.rs:188-253 -> k_verify_one_ped, k_verify_each_ped (per-proof verdicts)
//   pedersen Proof::deserialize_compressed (wire push) -> k_ped_wire_unpack, k_dec_prep/k_dec_finish, k_ped_proof_ok
// There is no CPU fallback: without a CUDA device every compute entry point fails.
#include <array>
#include <cstdlib>
#include <functional>
#include <map>
#include <memory>
#include <new>
#include <vector>

#include "host_common.h"
#include "hostutil.h"
#include "feeders.cuh"      // -> prepare.cuh -> msm.cuh -> thin.cuh, curve.cuh, fp.cuh, sha512.cuh
#include "verify_one.cuh"
#include "microbench.cuh"

using namespace avrf;

// =========================================================================================
// Batch handle
// =========================================================================================
// proofs per k_prepare launch: one full wave of the 126-register kernel (148 SMs x 4 blocks x 128 threads; a 65536-proof
// chunk filled only 86 % of the block slots); 4.6 MiB of (c,s) stream per chunk
constexpr size_t PREP_CHUNK = 148 * 4 * 128;
// proofs per shipment of staged single pushes: half a chunk, so that at most 2.4 MiB of the (c,s) stream (3 ms of
// SHA-512) remains to be hashed when the caller's push loop ends and verify is called
constexpr size_t STAGE_CHUNK = PREP_CHUNK / 2;

// Pinned SoA staging of single pushes (avrf_thin_batch_push, avrf_pedersen_batch_push): one buffer per input column of
// the handle's scheme (Scheme::col), filled by the caller's thread, shipped to the device one chunk at a time while the
// other buffer fills.
struct PushStage {
  PinBuf col[5], ios, ad, io_off, ad_off;
  size_t n = 0, nio = 0, nad = 0, cap_io = 0, cap_ad = 0;
  cudaEvent_t free_ev = nullptr;        // recorded once the device has consumed the buffer
  bool inflight = false;
};

struct avrf_batch {
  int device = 0;
  uint32_t suite = 0, fmt = 0, weights_mode = AVRF_WEIGHTS_REFERENCE;
  uint32_t scheme = 0;                  // 0 = Thin VRF, 1 = Pedersen VRF (src/pedersen.rs)
  uint64_t n = 0, n_ios = 0, ad_bytes = 0;
  bool prepared = false;
  bool have_seed = false;
  bool want_taps = false;
  uint8_t seed[64];
  uint64_t first_index = 0;             // global index of this handle's first proof in the last MSM run
  std::vector<uint64_t> segs;           // shards of a multi-GPU batch: (local start, global first) runs, see msm.cuh
  bool segs_dirty = false;
  // inputs on the device
  DevBuf pk, r, s, ios, io_off, ad_off, ad;
  DevBuf ok, sb;                        // Pedersen only (pk holds the key commitments)
  // decode buffers of the wire-format pushes (feed_api.inl, WireChunk): allocated by the first such push, so that
  // pushes on different handles hold no lock shared with other handles or the handle-less entry points
  DevBuf w_in, w_y, w_den, w_scr, w_fl, w_out, w_ok, w_sc, w_po, w_off, w_rec;
  // single-push staging on the host: pinned double buffer (eager handles), plain vectors otherwise
  PushStage stage[2];
  int cur = 0;
  std::vector<uint8_t> h_col[5], h_ios, h_ad;   // h_col: one vector per input column of the scheme (Scheme::col)
  std::vector<uint32_t> h_io_off{0}, h_ad_off{0};
  // derived
  DevBuf dig_w, rank_w;                 // window-major copies of the digits / ranks (k_sort_transpose)
  DevBuf pts, cs, z, renc, digits, hist, cursor, offs, toff, btot, totals, entries, tasks, task_out, chunk_out, wsum,
      partial, gpart, flags, w_tap, scalars_tap, segs_dev;
  PinBuf h_cs, h_small;
  std::vector<cudaEvent_t> prep_ev;     // one per PREP_CHUNK proofs: cs chunk i is ready
  size_t prep_ev_chunks = 0;            // chunks of the CURRENT batch covered by prep_ev (0: use a plain stream order)
  // eager path: push = H2D + prepare + D2H + incremental SHA-512 of the batch transcript, pipelined; the hash runs
  // on the hasher's own thread (host_common.h), so neither push nor the caller's loop waits for it
  bool eager = true;
  std::unique_ptr<Hasher> hasher;
  Hasher* ext_hasher = nullptr;         // shards of a multi-GPU batch feed their parent's hasher instead
  MbSha512* mb = nullptr;               // batch-server handles: hashing delegated to a shared multi-buffer thread
  bool blocking = false;                // host waits sleep instead of spinning (many worker threads per core)
  cudaEvent_t sync_ev = nullptr;
  uint64_t hashed = 0;                  // proofs whose (c,s) are absorbed or queued in the hasher
  uint64_t push_launches = 0;           // k_prepare launches of the push pipeline for the current batch
  // the handle's own streams: compute + ordered copies; overlapped D2H of the (c,s) stream; chunked H2D of
  // pushed proofs; k_prepare of the eager push pipeline (high priority: it feeds the host hash)
  cudaStream_t st = nullptr, st_copy = nullptr, st_h2d = nullptr, st_prep = nullptr;
  ShardSlot* remote_slot = nullptr;     // peer-mapped slot on the combining device (multi-GPU batches)
  // asynchronous verify: MSM enqueued on st, verdict read back at wait
  bool inflight = false;
  bool inflight_did_prepare = false;
  int32_t early_status = -1;            // >= 0: verdict known without waiting (empty batch)
  cudaEvent_t done_ev = nullptr;
  cudaEvent_t gate_ev = nullptr;        // this handle's entry in the device's MSM gate
  cudaEvent_t h2d_gate_ev = nullptr;    // ... and in its host-to-device copy gate
  std::chrono::steady_clock::time_point t_verify0;
  cudaEvent_t ev[10] = {};
  avrf_timings tm = {};
};

// Wait for a stream of the handle: spinning (lowest latency) by default, sleeping for batch-server handles.
static cudaError_t hsync(avrf_batch* b, cudaStream_t st) {
  if (!b->blocking) return cudaStreamSynchronize(st);
  cudaError_t e;
  if (!b->sync_ev && (e = cudaEventCreateWithFlags(&b->sync_ev, cudaEventDisableTiming | cudaEventBlockingSync)) != cudaSuccess) return e;
  if ((e = cudaEventRecord(b->sync_ev, st)) != cudaSuccess) return e;
  return cudaEventSynchronize(b->sync_ev);
}

// What a proof scheme stores in a batch handle, indexed by avrf_batch::scheme.
struct Column {
  DevBuf avrf_batch::*buf;
  size_t bytes;                         // per proof
};
struct Scheme {
  uint32_t ncol;
  Column col[5];                        // the per-proof device inputs, in the order push_many_impl takes them
  size_t cs_stride;                     // bytes per proof of the (c,s) stream that the batch seed hashes
  size_t w_tap;                         // bytes per proof of AVRF_TAP_W
  size_t pts_proof, pts_pair, pts_fixed;  // MSM terms: per proof, per I/O pair, and the fixed bases added at MSM time
  uint32_t scal_per_thread;             // proofs per k_scalars / k_scalars_ped thread
  const char* prepare;                  // k_prepare<S> / k_prepare_ped<S>
  size_t proof_points(uint64_t n, uint64_t n_ios) const { return pts_proof * n + pts_pair * n_ios; }
  size_t points(uint64_t n, uint64_t n_ios) const { return proof_points(n, n_ios) + pts_fixed; }
};
static constexpr Scheme SCHEMES[2] = {
    // Thin VRF (src/thin.rs): pk | r | s; bases R, pk, (O_i, I_i) per proof and the generator
    {3, {{&avrf_batch::pk, 64}, {&avrf_batch::r, 64}, {&avrf_batch::s, 32}}, 64, 16, 2, 2, 1, SCAL_PER_THREAD, "k_prepare"},
    // Pedersen VRF (src/pedersen.rs): pk holds the key commitments; five bases per proof, then G and B
    {5, {{&avrf_batch::pk, 64}, {&avrf_batch::r, 64}, {&avrf_batch::s, 32}, {&avrf_batch::ok, 64}, {&avrf_batch::sb, 32}},
     96, 32, 5, 0, 2, 1, "k_prepare_ped"},
};
static const Scheme& scheme_of(const avrf_batch* b) { return SCHEMES[b->scheme]; }
using Columns = std::array<const uint8_t*, 5>;     // one array per input column of a push, in table order

static uint64_t pending_of(const avrf_batch* b) { return b->stage[0].n + b->stage[1].n + (b->h_io_off.size() - 1); }

#define DISPATCH(suite, STMT)                      \
  switch (suite) {                                 \
    case 0: { constexpr int S = 0; STMT; } break;  \
    case 1: { constexpr int S = 1; STMT; } break;  \
    case 2: { constexpr int S = 2; STMT; } break;  \
    default: return fail(AVRF_ERR_ARG, "unknown suite"); \
  }

static int launch_check(const char* name) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(AVRF_ERR_CUDA, name, cudaGetErrorString(e));
  return 0;
}
#define LAUNCHED(name) do { int rc__ = launch_check(name); if (rc__) return rc__; } while (0)

// SUITE_ID || 0x50: the start of every batch-seed hash (src/thin.rs:273-279).  Returns its length.
static size_t batch_prefix(uint32_t suite, unsigned char buf[40]) {
  size_t sl = CC_HOST[suite].sid_len;
  memcpy(buf, CC_HOST[suite].suite_id, sl);
  buf[sl] = DOM_BATCH;
  return sl + 1;
}

// SHA512(SUITE_ID || 0x50 || stream) of a host-resident batch-seed stream of n_items records of `stride` bytes (the
// Scheme::cs_stride of the proofs' scheme): avrf_thin_seed, avrf_pedersen_seed.
static int seed_of_stream(uint32_t suite, const uint8_t* stream, uint64_t n_items, size_t stride, uint8_t seed[64]) {
  if (suite > 2 || !seed || (n_items && !stream)) return fail(AVRF_ERR_ARG, "bad argument");
  unsigned char prefix[40];
  return sha512({{prefix, batch_prefix(suite, prefix)}, {stream, stride * n_items}}, seed);
}

// Orders `waiter` after the work enqueued so far on `st`.
static int stream_after(cudaStream_t waiter, cudaStream_t st) {
  cudaEvent_t e;
  CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  cudaEventRecord(e, st);
  cudaStreamWaitEvent(waiter, e, 0);
  cudaEventDestroy(e);
  return 0;
}

static int finish_inflight(avrf_batch* b);

// Every entry point that takes a handle starts here: bind the calling thread to the handle's device and complete
// a verify that is still in flight (include/avrf.h: "any other call on the handle completes it first").
static int enter(avrf_batch* b) {
  if (!b) return fail(AVRF_ERR_ARG, "null batch");
  int rc = bind_device(b->device);
  if (rc) return rc;
  return b->inflight ? finish_inflight(b) : 0;
}
#define ENTER(b) do { int rc__ = enter(b); if (rc__) return rc__; } while (0)

// All the streams of the handle are idle: required before a device buffer that they use is reallocated.
static int quiesce(avrf_batch* b) {
  for (cudaStream_t q : {b->st_h2d, b->st_prep, b->st_copy, b->st}) CK(hsync(b, q));
  return 0;
}
static int grow(avrf_batch* b, DevBuf& buf, size_t bytes, size_t keep) {
  if (bytes <= buf.cap) return 0;
  int rc = quiesce(b);
  return rc ? rc : buf.reserve(bytes, keep, b->st);
}
// Room for n proofs with n_ios pairs and ad_bytes of additional data in the input buffers, keeping the handle's proofs.
static int grow_inputs(avrf_batch* b, uint64_t n, uint64_t n_ios, uint64_t ad_bytes) {
  const Scheme& sc = scheme_of(b);
  int rc;
  for (uint32_t k = 0; k < sc.ncol; k++)
    if ((rc = grow(b, b->*sc.col[k].buf, sc.col[k].bytes * n, sc.col[k].bytes * b->n))) return rc;
  if ((rc = grow(b, b->ios, 128 * n_ios + 128, 128 * b->n_ios)) || (rc = grow(b, b->ad, ad_bytes + 16, b->ad_bytes)) ||
      (rc = grow(b, b->io_off, 4 * (n + 1), 4 * (b->n + 1))) || (rc = grow(b, b->ad_off, 4 * (n + 1), 4 * (b->n + 1))))
    return rc;
  return 0;
}
// ... and in the buffers k_prepare fills, keeping what it derived for the handle's proofs when they are prepared
static int grow_derived(avrf_batch* b, uint64_t n, uint64_t n_ios) {
  const Scheme& sc = scheme_of(b);
  const bool keep = b->prepared;
  size_t np = sc.points(n, n_ios), np_old = b->n ? sc.proof_points(b->n, b->n_ios) : 0;
  int rc;
  if ((rc = grow(b, b->pts, sizeof(BaseRec) * np, keep ? sizeof(BaseRec) * np_old : 0)) ||
      (rc = grow(b, b->cs, sc.cs_stride * n + 64, keep ? sc.cs_stride * b->n : 0)) ||
      (rc = grow(b, b->z, 16 * n_ios + 16, keep ? 16 * b->n_ios : 0)) ||
      (rc = grow(b, b->renc, 32 * n + 32, keep ? 32 * b->n : 0)))
    return rc;
  return 0;
}

static Hasher* hasher_of(avrf_batch* b) {
  if (b->ext_hasher) return b->ext_hasher;
  if (!b->hasher) {
    b->hasher.reset(new (std::nothrow) Hasher(b->device));
    if (b->hasher && b->mb) b->hasher->use_multibuffer(b->mb);
  }
  return b->hasher.get();
}

// Device buffers of the handle-less entry points (hash-to-curve, outputs, proving, ingest), kept between calls: a
// cudaMalloc / cudaFree pair per buffer per call costs more than the kernels of a small call.  One pool per device;
// the calls share that device's stream, so they are serialised by the pool's mutex anyway.
struct H2cScratch { DevBuf u01, den, scr; };
struct FeedPool {
  std::mutex mu;
  DevBuf b[12];
  H2cScratch w;
};
static FeedPool g_feed[AVRF_MAX_DEV];
static void feed_pool_release(int dev) {
  FeedPool& fp = g_feed[dev];
  std::lock_guard<std::mutex> lk(fp.mu);
  for (DevBuf& d : fp.b) d.release();
  fp.w.u01.release(); fp.w.den.release(); fp.w.scr.release();
}

// One call over a device's feed pool: holds the pool for the duration of the call, hands out its buffers in order and
// stages the call's copies on `st`.  The first error is kept in `rc` and turns every later buffer or copy into a no-op,
// so a caller checks `rc` once before it launches.
struct FeedFrame {
  FeedPool& fp;
  std::lock_guard<std::mutex> lock;
  cudaStream_t st;
  int rc = 0;
  FeedFrame(int device, cudaStream_t s) : fp(g_feed[device]), lock(fp.mu), st(s) {}
  H2cScratch& scratch() { return fp.w; }
  // the next pool buffer, grown to at least `bytes` (an empty buffer once an error is kept)
  DevBuf& take(size_t bytes) {
    if (!rc && used == std::size(fp.b)) rc = fail(AVRF_ERR_STATE, "feed pool exhausted");
    if (rc) return none;
    DevBuf& d = fp.b[used++];
    rc = d.reserve(bytes);
    return d;
  }
  // the next pool buffer, grown to `bytes + slack`, with `bytes` of host memory copied in
  DevBuf& in(const void* h, size_t bytes, size_t slack = 0) {
    DevBuf& d = take(bytes + slack);
    if (!rc && bytes) rc = copy(d.p, h, bytes, cudaMemcpyHostToDevice);
    return d;
  }
  // `bytes` of device memory back to `h`; nothing when `h` is null (an output the caller did not ask for).  Returns
  // the kept error, for a caller that launches more work after the copy.
  int out(void* h, const void* d, size_t bytes) {
    if (!rc && h) rc = copy(h, d, bytes, cudaMemcpyDeviceToHost);
    return rc;
  }
  // the end of the call: waits for the stream, so that every output has landed
  int sync() {
    if (!rc) rc = wait();
    return rc;
  }

 private:
  size_t used = 0;
  DevBuf none;
  int copy(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) { CK(cudaMemcpyAsync(dst, src, bytes, kind, st)); return 0; }
  int wait() { CK(cudaStreamSynchronize(st)); return 0; }
};

// MSM gate: the heavy part of the MSMs of different handles on one device (scalars, sort, bucket accumulation) runs
// one batch after the other, in submission order.  Left to themselves the streams of T handles interleave kernel by
// kernel, all T MSMs finish together after T x 10 ms, and no handle can start hashing its next batch before that;
// in FIFO order handle i has its verdict after (i + 1) x 10 ms and its next hash overlaps the MSMs of the others.
// The latency-bound tail (combine, bucket reduction, fold: ~1.4 ms on a handful of SMs) is outside the gate and
// overlaps the next batch's accumulation.
struct MsmGate {
  std::mutex mu;
  cudaEvent_t tail = nullptr;       // recorded after the k_accumulate of the MSM submitted last (owned by its handle)
};
static MsmGate g_gate[AVRF_MAX_DEV];
static int sm_count(int device) {
  static int cached[AVRF_MAX_DEV] = {};
  if (device < 0 || device >= AVRF_MAX_DEV) return 148;
  if (!cached[device]) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || v <= 0) v = 148;
    cached[device] = v;
  }
  return cached[device];
}
// The same for the host-to-device copies of the push pipeline: pushes that arrive together would share PCIe evenly and
// all of their data would land at the end; in FIFO order push i has its data after (i + 1) x 6 ms, its transcripts and
// its batch-seed hash start then, and the first verdicts are ready while the later pushes are still copying.
static MsmGate g_h2d_gate[AVRF_MAX_DEV];

extern "C" {

// =========================================================================================
// Library / devices
// =========================================================================================
const char* avrf_last_error(void) { return g_err.c_str(); }
const char* avrf_version(void) { return "ark-vrf_b200 0.2 (sm_100a)"; }

int avrf_init(int device) {
  int ids[1] = {device};
  std::lock_guard<std::mutex> lock(g_init_mu);
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(AVRF_ERR_NO_DEVICE, "no CUDA device (this library has no CPU fallback)", cudaGetErrorString(e));
  if (device < 0 || device >= count || device >= AVRF_MAX_DEV) return fail(AVRF_ERR_ARG, "device index out of range");
  if (g_device >= 0 && g_device != device) return fail(AVRF_ERR_STATE, "already initialised on another device");
  int rc = dev_setup(ids[0]);
  if (rc) return rc;
  g_device = device;
  return bind_device(device);              // binds the calling thread too
}

int avrf_init_multi(int n_dev, const int* dev_ids) {
  std::lock_guard<std::mutex> lock(g_init_mu);
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(AVRF_ERR_NO_DEVICE, "no CUDA device (this library has no CPU fallback)", cudaGetErrorString(e));
  if (n_dev <= 0) n_dev = count;
  if (n_dev > count || n_dev > AVRF_MAX_DEV) return fail(AVRF_ERR_ARG, "more devices requested than present");
  int first = dev_ids ? dev_ids[0] : 0;
  if (g_device >= 0 && g_device != first) return fail(AVRF_ERR_STATE, "already initialised with another default device");
  for (int i = 0; i < n_dev; i++) {
    int d = dev_ids ? dev_ids[i] : i;
    if (d < 0 || d >= count || d >= AVRF_MAX_DEV) return fail(AVRF_ERR_ARG, "device index out of range");
    int rc = dev_setup(d);
    if (rc) return rc;
  }
  // peer access between every pair (NVLink / NVSwitch): shards store their partial sums straight into the
  // combining device's memory.  Pairs without peer access fall back to cudaMemcpyPeerAsync.
  int nd = g_ndev.load();
  for (int i = 0; i < nd; i++)
    for (int j = 0; j < nd; j++) {
      if (i == j) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, g_dev_list[i], g_dev_list[j]);
      if (!can) continue;
      cudaSetDevice(g_dev_list[i]);
      cudaError_t pe = cudaDeviceEnablePeerAccess(g_dev_list[j], 0);
      if (pe != cudaSuccess) (void)cudaGetLastError();      // already enabled
    }
  t_bound = -1;
  g_device = first;
  return bind_device(first);
}

int avrf_device_count(void) { return g_ndev.load(); }

int avrf_shutdown(void) {
  std::lock_guard<std::mutex> lock(g_init_mu);
  for (int i = 0; i < AVRF_MAX_DEV; i++) {
    DevState& d = g_devs[i];
    if (!d.ready) continue;
    cudaSetDevice(i);
    feed_pool_release(i);
    if (d.stream) cudaStreamDestroy(d.stream);
    if (d.copy) cudaStreamDestroy(d.copy);
    d = DevState{};
  }
  g_ndev = 0;
  g_device = -1;
  t_bound = -1;
  return 0;
}

// =========================================================================================
// Handle life cycle
// =========================================================================================
avrf_batch* avrf_thin_batch_new_on(int device, uint32_t suite, uint32_t fmt) {
  if (suite > 2 || fmt > 1) { fail(AVRF_ERR_ARG, "bad suite/fmt"); return nullptr; }
  if (ensure_init()) return nullptr;
  if (device < 0) device = g_device.load();
  if (device >= AVRF_MAX_DEV || !g_devs[device].ready) { fail(AVRF_ERR_ARG, "device not initialised (avrf_init / avrf_init_multi)"); return nullptr; }
  if (bind_device(device)) return nullptr;
  avrf_batch* b = new (std::nothrow) avrf_batch();
  if (!b) { fail(AVRF_ERR_NOMEM, "host allocation"); return nullptr; }
  b->device = device;
  b->suite = suite;
  b->fmt = fmt;
  for (auto& e : b->ev) cudaEventCreate(&e);
  if (cudaStreamCreateWithFlags(&b->st, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&b->st_copy, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&b->st_h2d, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithPriority(&b->st_prep, cudaStreamNonBlocking, g_devs[device].prio_hi) != cudaSuccess) {
    fail(AVRF_ERR_CUDA, "cudaStreamCreate", cudaGetErrorString(cudaGetLastError()));
    avrf_thin_batch_free(b);
    return nullptr;
  }
  return b;
}

avrf_batch* avrf_thin_batch_new(uint32_t suite, uint32_t fmt) { return avrf_thin_batch_new_on(-1, suite, fmt); }

void avrf_thin_batch_free(avrf_batch* b) {
  if (!b) return;
  bind_device(b->device);
  if (b->inflight) finish_inflight(b);
  b->hasher.reset();                      // joins the hashing thread
  if (b->done_ev) cudaEventDestroy(b->done_ev);
  if (b->gate_ev) {
    MsmGate& g = g_gate[b->device];
    std::lock_guard<std::mutex> lk(g.mu);
    if (g.tail == b->gate_ev) g.tail = nullptr;
    cudaStreamSynchronize(b->st);
    cudaEventDestroy(b->gate_ev);
  }
  if (b->h2d_gate_ev) {
    MsmGate& g = g_h2d_gate[b->device];
    std::lock_guard<std::mutex> lk(g.mu);
    if (g.tail == b->h2d_gate_ev) g.tail = nullptr;
    cudaStreamSynchronize(b->st_h2d);
    cudaEventDestroy(b->h2d_gate_ev);
  }
  for (cudaStream_t q : {b->st, b->st_copy, b->st_h2d, b->st_prep}) if (q) cudaStreamSynchronize(q);
  const Scheme& sc = scheme_of(b);
  for (uint32_t k = 0; k < sc.ncol; k++) (b->*sc.col[k].buf).release();
  DevBuf* bufs[] = {&b->ios, &b->io_off, &b->ad_off, &b->ad, &b->pts, &b->cs, &b->z, &b->renc,
                    &b->dig_w, &b->rank_w, &b->digits, &b->hist, &b->cursor, &b->offs, &b->toff, &b->btot, &b->totals, &b->entries, &b->tasks,
                    &b->task_out, &b->chunk_out, &b->wsum, &b->partial, &b->gpart, &b->flags, &b->w_tap, &b->scalars_tap,
                    &b->segs_dev, &b->w_in, &b->w_y, &b->w_den, &b->w_scr, &b->w_fl, &b->w_out, &b->w_ok, &b->w_sc,
                    &b->w_po, &b->w_off, &b->w_rec};
  for (DevBuf* d : bufs) d->release();
  for (auto& e : b->ev) if (e) cudaEventDestroy(e);
  for (auto& e : b->prep_ev) cudaEventDestroy(e);
  for (auto& sg : b->stage) if (sg.free_ev) cudaEventDestroy(sg.free_ev);
  if (b->sync_ev) cudaEventDestroy(b->sync_ev);
  for (cudaStream_t q : {b->st, b->st_copy, b->st_h2d, b->st_prep}) if (q) cudaStreamDestroy(q);
  delete b;
}

int avrf_thin_batch_clear(avrf_batch* b) {
  ENTER(b);
  if (b->hasher) b->hasher->drain();
  // staged single pushes that were never flushed are dropped; buffers still owned by an H2D copy are waited for
  for (auto& sg : b->stage) {
    if (sg.inflight) { CK(cudaEventSynchronize(sg.free_ev)); sg.inflight = false; }
    sg.n = sg.nio = sg.nad = 0;
  }
  b->n = b->n_ios = b->ad_bytes = 0;
  b->prepared = b->have_seed = false;
  b->hashed = 0;
  b->push_launches = 0;
  b->prep_ev_chunks = 0;
  b->segs.clear();
  b->segs_dirty = true;
  for (auto& v : b->h_col) v.clear();
  b->h_ios.clear(); b->h_ad.clear();
  b->h_io_off.assign(1, 0);
  b->h_ad_off.assign(1, 0);
  return 0;
}

int avrf_thin_batch_invalidate(avrf_batch* b) {
  ENTER(b);
  if (b->hasher) b->hasher->drain();
  { int rc__ = quiesce(b); if (rc__) return rc__; }   // the next prepare runs on the compute stream: nothing of the push pipeline may be pending
  b->prepared = b->have_seed = false;
  b->hashed = 0;
  b->push_launches = 0;
  b->prep_ev_chunks = 0;
  return 0;
}

int avrf_thin_batch_set_eager(avrf_batch* b, int eager) {
  ENTER(b);
  if (pending_of(b)) return fail(AVRF_ERR_STATE, "set_eager with staged single pushes pending: call it on an empty handle");
  b->eager = eager != 0;
  return 0;
}

// Host waits of this handle sleep (blocking-sync events) instead of spinning.  Spinning gives the lowest latency for one
// handle; with several handles driven from as many threads it burns the cores the other batches' hashes need.
int avrf_thin_batch_set_blocking(avrf_batch* b, int blocking) {
  ENTER(b);
  b->blocking = blocking != 0;
  if (b->done_ev) { cudaEventDestroy(b->done_ev); b->done_ev = nullptr; }     // recreated with the right flags
  return 0;
}

// ---- shared multi-buffer hashing threads -------------------------------------------------------------------------
struct avrf_hash_pool {
  std::vector<std::unique_ptr<MbSha512>> hashers;
  std::atomic<uint32_t> next{0};
};

avrf_hash_pool* avrf_hash_pool_new(uint32_t n_threads) {
  if (n_threads == 0 || n_threads > 64) { fail(AVRF_ERR_ARG, "bad thread count"); return nullptr; }
  avrf_hash_pool* hp = new (std::nothrow) avrf_hash_pool();
  if (!hp) { fail(AVRF_ERR_NOMEM, "host allocation"); return nullptr; }
  try {
    for (uint32_t i = 0; i < n_threads; i++) hp->hashers.emplace_back(new MbSha512());
  } catch (...) {
    delete hp;
    fail(AVRF_ERR_NOMEM, "cannot start hashing threads");
    return nullptr;
  }
  return hp;
}

void avrf_hash_pool_free(avrf_hash_pool* hp) { delete hp; }

int avrf_thin_batch_set_hash_pool(avrf_batch* b, avrf_hash_pool* hp) {
  ENTER(b);
  if (b->ext_hasher) return fail(AVRF_ERR_STATE, "the shards of a multi-GPU batch hash through their parent");
  if (b->hasher) { b->hasher->drain(); b->hasher.reset(); }          // releases its lane, if any
  b->mb = hp && !hp->hashers.empty() ? hp->hashers[hp->next++ % hp->hashers.size()].get() : nullptr;
  b->hashed = 0;                          // what was absorbed so far is gone with the old hasher
  b->have_seed = false;
  return 0;
}

void* avrf_stream(void) { return g_device.load() >= 0 ? (void*)gs() : nullptr; }
void* avrf_thin_batch_stream(avrf_batch* b) { return b ? (void*)b->st : nullptr; }
int avrf_thin_batch_device(const avrf_batch* b) { return b ? b->device : -1; }

int64_t avrf_thin_batch_len(const avrf_batch* b) { return b ? (int64_t)(b->n + pending_of(b)) : -1; }

int avrf_thin_batch_set_weights_mode(avrf_batch* b, uint32_t mode) {
  if (mode > AVRF_WEIGHTS_TREE) return fail(AVRF_ERR_ARG, "bad weights mode");
  ENTER(b);
  // the tree leaves hash the 64-byte thin (c,s) records; the Pedersen stream is (c,s,sb), 96 bytes per proof
  if (mode == AVRF_WEIGHTS_TREE && b->scheme != 0) return fail(AVRF_ERR_ARG, "AVRF_WEIGHTS_TREE is defined for Thin-VRF batches only");
  b->weights_mode = mode;
  b->have_seed = false;
  return 0;
}

// Room for n proofs, n_ios pairs and ad_bytes of additional data (like Vec::with_capacity): pushes up to that
// size never reallocate device memory.
int avrf_thin_batch_reserve(avrf_batch* b, uint64_t n, uint64_t n_ios, uint64_t ad_bytes) {
  ENTER(b);
  if (n >= (1ull << 30) || n_ios >= (1ull << 30) || ad_bytes >= (1ull << 32)) return fail(AVRF_ERR_ARG, "batch too large");
  int rc = grow_inputs(b, n, n_ios, ad_bytes);
  return rc ? rc : grow_derived(b, n, n_ios);
}

// Leaf digests (64 B each) of this handle's (c,s) stream; first_index = global index of its first proof
// (must be a multiple of 32 unless it is 0).
int avrf_thin_batch_tree_leaves(avrf_batch* b, uint64_t first_index, uint8_t* out, uint64_t* n_leaves) {
  if (!b || !out || !n_leaves || (first_index % TREE_LEAF)) return fail(AVRF_ERR_ARG, "bad argument");
  if (b->scheme != 0) return fail(AVRF_ERR_ARG, "tree leaves are defined for Thin-VRF batches only");
  int rc = avrf_thin_batch_prepare(b, nullptr);
  if (rc) return rc;
  uint32_t nl = (uint32_t)((b->n + TREE_LEAF - 1) / TREE_LEAF);
  *n_leaves = nl;
  if (!nl) return 0;
  if ((rc = b->gpart.reserve(64 * (size_t)nl + 64))) return rc;
  k_tree_leaves<<<cdiv(nl, 64), 64, 0, b->st>>>(b->cs.as<uint32_t>(), (uint32_t)b->n, first_index / TREE_LEAF,
                                                   b->gpart.as<uint64_t>());
  LAUNCHED("k_tree_leaves");
  CK(cudaMemcpyAsync(out, b->gpart.p, 64 * (size_t)nl, cudaMemcpyDeviceToHost, b->st));
  CK(hsync(b, b->st));
  return 0;
}

// seed = SHA512(SUITE_ID || 0x50 || 0x01 || LE64(n_total) || leaf_0 || leaf_1 || ...)
int avrf_thin_seed_tree(uint32_t suite, uint64_t n_total, const uint8_t* leaves, uint64_t n_leaves, uint8_t seed[64]) {
  if (suite > 2 || !seed || (n_leaves && !leaves)) return fail(AVRF_ERR_ARG, "bad argument");
  unsigned char head[49];
  size_t hl = batch_prefix(suite, head);
  head[hl++] = 0x01;
  for (int i = 0; i < 8; i++) head[hl++] = (unsigned char)(n_total >> (8 * i));
  return sha512({{head, hl}, {leaves, 64 * n_leaves}}, seed);
}

// =========================================================================================
// Push
// =========================================================================================
// The offsets of a push of n proofs start at 0, and a blob that the offsets say is not empty is present.
static int check_offsets(uint64_t n, const uint32_t* io_offsets, const uint32_t* ad_offsets, const uint8_t* ios,
                         const uint8_t* ad_blob) {
  if (io_offsets[0] != 0 || ad_offsets[0] != 0) return fail(AVRF_ERR_ARG, "offsets must start at 0");
  if ((io_offsets[n] && !ios) || (ad_offsets[n] && !ad_blob)) return fail(AVRF_ERR_ARG, "null argument");
  return 0;
}

// k_prepare<S> (Thin) / k_prepare_ped<S> (Pedersen) over the resident proofs [first, last) of the handle, on `st`.
static int launch_prepare(avrf_batch* b, size_t first, size_t last, cudaStream_t st) {
  const uint32_t grid = cdiv(last - first, 128);
  if (b->scheme == 1) {
    PedPrepArgs a;
    a.pkcom = b->pk.as<Affine>(); a.r = b->r.as<Affine>(); a.ok = b->ok.as<Affine>(); a.s = b->s.as<Fe>();
    a.sb = b->sb.as<Fe>(); a.ios = b->ios.as<Affine>(); a.io_off = b->io_off.as<uint32_t>();
    a.ad_off = b->ad_off.as<uint32_t>(); a.ad = b->ad.as<uint8_t>(); a.pts = b->pts.as<BaseRec>();
    a.cs = b->cs.as<uint32_t>(); a.flags = b->flags.as<int>();
    a.first = (uint32_t)first; a.n = (uint32_t)last; a.canonical = b->fmt == AVRF_FMT_CANONICAL;
    DISPATCH(b->suite, (k_prepare_ped<S><<<grid, 128, 0, st>>>(a)));
  } else {
    PrepArgs a;
    a.pk = b->pk.as<Affine>(); a.r = b->r.as<Affine>(); a.s = b->s.as<Fe>(); a.ios = b->ios.as<Affine>();
    a.io_off = b->io_off.as<uint32_t>(); a.ad_off = b->ad_off.as<uint32_t>(); a.ad = b->ad.as<uint8_t>();
    a.pts = b->pts.as<BaseRec>(); a.cs = b->cs.as<uint32_t>(); a.z = b->z.as<uint32_t>();
    a.renc = b->renc.as<uint32_t>(); a.flags = b->flags.as<int>();
    a.first = (uint32_t)first; a.n = (uint32_t)last; a.canonical = b->fmt == AVRF_FMT_CANONICAL;
    DISPATCH(b->suite, (k_prepare<S><<<grid, 128, 0, st>>>(a)));
  }
  LAUNCHED(scheme_of(b).prepare);
  return 0;
}

// n proofs from host arrays into the handle: `cols` holds one array per input column of the handle's scheme, in table
// order.  With the eager pipeline the (c,s) chunks are handed to the hasher thread and the call returns without waiting
// for the hash; `consumed` (optional) is recorded once the device no longer reads the host arrays.
static int push_many_impl(avrf_batch* b, uint64_t n, const Columns& cols, const uint8_t* ios, const uint32_t* io_offsets,
                          const uint8_t* ad_blob, const uint32_t* ad_offsets, cudaEvent_t consumed = nullptr,
                          size_t stage_chunks = 0) {
  const Scheme& sc = scheme_of(b);
  const size_t stride = sc.cs_stride;
  if (n == 0) return 0;
  // offsets may start anywhere (a slice of a larger push): `ios` / `ad_blob` point at the slice's first pair / byte
  const uint32_t iob = io_offsets[0], adb = ad_offsets[0];
  uint64_t add_ios = io_offsets[n] - iob, add_ad = ad_offsets[n] - adb;
  uint64_t n0 = b->n, i0 = b->n_ios, a0 = b->ad_bytes;
  if (n0 + n >= (1ull << 30) || i0 + add_ios >= (1ull << 30) || a0 + add_ad >= (1ull << 32))
    return fail(AVRF_ERR_ARG, "batch too large");
  int rc;
  bool pipeline = b->eager && (b->prepared || n0 == 0) && b->hashed == n0;
  if ((rc = grow_inputs(b, n0 + n, i0 + add_ios, a0 + add_ad))) return rc;
  // offsets first (small), rebased on the device
  cudaStream_t ost = pipeline ? b->st_prep : b->st;
  CK(cudaMemcpyAsync(b->io_off.as<uint32_t>() + n0, io_offsets, 4 * (n + 1), cudaMemcpyHostToDevice, ost));
  CK(cudaMemcpyAsync(b->ad_off.as<uint32_t>() + n0, ad_offsets, 4 * (n + 1), cudaMemcpyHostToDevice, ost));
  if (i0 != iob) { k_rebase<<<cdiv(n + 1, 256), 256, 0, ost>>>(b->io_off.as<uint32_t>() + n0, n + 1, (uint32_t)i0 - iob); LAUNCHED("k_rebase"); }
  if (a0 != adb) { k_rebase<<<cdiv(n + 1, 256), 256, 0, ost>>>(b->ad_off.as<uint32_t>() + n0, n + 1, (uint32_t)a0 - adb); LAUNCHED("k_rebase"); }
  if (!pipeline) {
    for (uint32_t k = 0; k < sc.ncol; k++) {
      const Column& c = sc.col[k];
      CK(cudaMemcpyAsync((b->*c.buf).as<uint8_t>() + c.bytes * n0, cols[k], c.bytes * n, cudaMemcpyDefault, b->st));
    }
    if (add_ios) CK(cudaMemcpyAsync(b->ios.as<uint8_t>() + 128 * i0, ios, 128 * add_ios, cudaMemcpyDefault, b->st));
    if (add_ad) CK(cudaMemcpyAsync(b->ad.as<uint8_t>() + a0, ad_blob, add_ad, cudaMemcpyDefault, b->st));
    if (consumed) CK(cudaEventRecord(consumed, b->st));
    b->n += n;
    b->n_ios += add_ios;
    b->ad_bytes += add_ad;
    b->prepared = b->have_seed = false;
    b->hashed = 0;
    b->prep_ev_chunks = 0;
    return 0;
  }
  // ---- eager pipeline: per chunk  H2D (st_h2d) -> k_prepare (st_prep) -> D2H of (c,s) (st_copy) -> hasher thread ----
  Hasher* hs = hasher_of(b);
  if (!hs) return fail(AVRF_ERR_NOMEM, "hasher");
  if ((rc = b->flags.reserve(64))) return rc;
  if ((rc = b->h_small.reserve(4096))) return rc;
  if ((rc = grow_derived(b, n0 + n, i0 + add_ios))) return rc;       // (the pipeline runs on prepared or empty handles)
  if (n0 == 0) {
    if (!b->ext_hasher) {                 // a shard's parent starts the stream of the whole batch itself
      unsigned char prefix[40];
      if ((rc = hs->begin(prefix, batch_prefix(b->suite, prefix)))) return rc;
    }
    CK(cudaMemsetAsync(b->flags.p, 0, 64, b->st_prep));
  }
  // pinned staging of the (c,s) chunks: room for the whole call (capped at 16 chunks), or for `stage_chunks`
  // chunks when the caller ships one chunk at a time (single pushes) - the area is reused as the hasher drains it
  if ((rc = hs->reserve_stage(std::max(stride * std::min<size_t>(n, 16 * PREP_CHUNK) + 64, stage_chunks * (stride * PREP_CHUNK + 64))))) return rc;
  size_t nch = (n + PREP_CHUNK - 1) / PREP_CHUNK;
  EventPool evs;
  cudaEvent_t off_ev = evs.make();
  if (!off_ev) return fail(AVRF_ERR_CUDA, "cudaEventCreate");
  CK(cudaEventRecord(off_ev, b->st_prep));
  CK(cudaStreamWaitEvent(b->st_h2d, off_ev, 0));         // also orders after any device-side realloc copies
  if (!b->h2d_gate_ev) CK(cudaEventCreateWithFlags(&b->h2d_gate_ev, cudaEventDisableTiming));
  MsmGate& hgate = g_h2d_gate[b->device];
  std::unique_lock<std::mutex> hgate_lock(hgate.mu);
  if (hgate.tail && hgate.tail != b->h2d_gate_ev) CK(cudaStreamWaitEvent(b->st_h2d, hgate.tail, 0));
  for (size_t c = 0; c < nch; c++) {
    size_t c0 = c * PREP_CHUNK, c1 = std::min((size_t)n, c0 + PREP_CHUNK), cnt = c1 - c0;
    size_t q0 = io_offsets[c0] - iob, q1 = io_offsets[c1] - iob, d0 = ad_offsets[c0] - adb, d1 = ad_offsets[c1] - adb;
    cudaEvent_t h2d_ev = evs.make(), prep_ev = evs.make();
    cudaEvent_t d2h_ev = nullptr;                          // owned by the hasher once queued
    if (!h2d_ev || !prep_ev) return fail(AVRF_ERR_CUDA, "cudaEventCreate");
    for (uint32_t k = 0; k < sc.ncol; k++) {
      const Column& col = sc.col[k];
      CK(cudaMemcpyAsync((b->*col.buf).as<uint8_t>() + col.bytes * (n0 + c0), cols[k] + col.bytes * c0, col.bytes * cnt,
                         cudaMemcpyDefault, b->st_h2d));
    }
    if (q1 > q0) CK(cudaMemcpyAsync(b->ios.as<uint8_t>() + 128 * (i0 + q0), ios + 128 * q0, 128 * (q1 - q0), cudaMemcpyDefault, b->st_h2d));
    if (d1 > d0) CK(cudaMemcpyAsync(b->ad.as<uint8_t>() + a0 + d0, ad_blob + d0, d1 - d0, cudaMemcpyDefault, b->st_h2d));
    CK(cudaEventRecord(h2d_ev, b->st_h2d));
    CK(cudaStreamWaitEvent(b->st_prep, h2d_ev, 0));
    if ((rc = launch_prepare(b, n0 + c0, n0 + c1, b->st_prep))) return rc;
    CK(cudaEventRecord(prep_ev, b->st_prep));
    CK(cudaStreamWaitEvent(b->st_copy, prep_ev, 0));
    uint8_t* dst = hs->stage(stride * cnt);
    if (!dst) return fail(AVRF_ERR_NOMEM, "pinned staging");
    CK(cudaMemcpyAsync(dst, b->cs.as<uint8_t>() + stride * (n0 + c0), stride * cnt, cudaMemcpyDeviceToHost, b->st_copy));
    CK(cudaEventCreateWithFlags(&d2h_ev, cudaEventDisableTiming | cudaEventBlockingSync));
    CK(cudaEventRecord(d2h_ev, b->st_copy));
    hs->enqueue(d2h_ev, dst, stride * cnt);
  }
  CK(cudaEventRecord(b->h2d_gate_ev, b->st_h2d));
  hgate.tail = b->h2d_gate_ev;
  hgate_lock.unlock();
  if (consumed) CK(cudaEventRecord(consumed, b->st_prep));   // after the last k_prepare: covers the H2D copies as well
  b->n += n;
  b->n_ios += add_ios;
  b->ad_bytes += add_ad;
  b->hashed = b->n;
  b->prepared = true;
  b->have_seed = false;
  b->prep_ev_chunks = 0;
  b->push_launches += nch;
  return 0;
}

static int stage_reserve(const Scheme& sc, PushStage& sg, size_t cap_io, size_t cap_ad) {
  int rc;
  for (uint32_t k = 0; k < sc.ncol; k++)
    if ((rc = sg.col[k].reserve(sc.col[k].bytes * PREP_CHUNK))) return rc;
  if ((rc = sg.io_off.reserve(4 * (PREP_CHUNK + 1))) || (rc = sg.ad_off.reserve(4 * (PREP_CHUNK + 1)))) return rc;
  if (cap_io > sg.cap_io) { if ((rc = sg.ios.reserve(128 * cap_io, 128 * sg.nio))) return rc; sg.cap_io = cap_io; }
  if (cap_ad > sg.cap_ad) { if ((rc = sg.ad.reserve(cap_ad, sg.nad))) return rc; sg.cap_ad = cap_ad; }
  if (!sg.free_ev) CK(cudaEventCreateWithFlags(&sg.free_ev, cudaEventDisableTiming));
  return 0;
}

// Ship the staged single pushes: the eager pipeline takes them as one chunk; the caller goes on filling the
// other buffer.
static int flush_stage(avrf_batch* b) {
  PushStage& sg = b->stage[b->cur];
  if (sg.n == 0) return 0;
  { int rc0 = bind_device(b->device); if (rc0) return rc0; }
  stage_fence();
  const Scheme& sc = scheme_of(b);
  Columns cols{};
  for (uint32_t k = 0; k < sc.ncol; k++) cols[k] = sg.col[k].as<uint8_t>();
  int rc = push_many_impl(b, sg.n, cols, sg.ios.as<uint8_t>(), sg.io_off.as<uint32_t>(), sg.ad.as<uint8_t>(),
                          sg.ad_off.as<uint32_t>(), sg.free_ev, sg.n == STAGE_CHUNK ? 4 : 0);
  if (rc) return rc;
  sg.n = sg.nio = sg.nad = 0;
  sg.inflight = true;
  b->cur ^= 1;
  PushStage& nx = b->stage[b->cur];
  if (nx.inflight) { CK(cudaEventSynchronize(nx.free_ev)); nx.inflight = false; }
  return 0;
}

static int flush_pending(avrf_batch* b) {
  int rc = flush_stage(b);
  if (rc) return rc;
  uint64_t pend = b->h_io_off.size() - 1;
  if (!pend) return 0;
  const Scheme& sc = scheme_of(b);
  Columns cols{};
  for (uint32_t k = 0; k < sc.ncol; k++) cols[k] = b->h_col[k].data();
  rc = push_many_impl(b, pend, cols, b->h_ios.data(), b->h_io_off.data(), b->h_ad.data(), b->h_ad_off.data());
  if (rc) return rc;
  if ((rc = quiesce(b))) return rc;        // host vectors are about to be cleared
  for (auto& v : b->h_col) v.clear();
  b->h_ios.clear(); b->h_ad.clear();
  b->h_io_off.assign(1, 0);
  b->h_ad_off.assign(1, 0);
  return 0;
}

// One proof of a single push (avrf_thin_batch_push, avrf_pedersen_batch_push): `cols` holds one field per input column
// of the handle's scheme, in table order.  Eager handles stage it in the pinned double buffer, shipped when it holds
// STAGE_CHUNK proofs, when its I/O or ad room runs out, or when a later call reads or extends the handle (flush_pending).
static int push_one(avrf_batch* b, const Columns& cols, const uint8_t* ios, uint32_t n_ios, const uint8_t* ad,
                    uint32_t ad_len) {
  if (b->inflight) ENTER(b);             // (the device is bound where CUDA is called: flush_stage)
  const Scheme& sc = scheme_of(b);
  if (!b->eager) {
    // shards of a multi-process batch: plain host vectors, shipped at prepare
    for (uint32_t k = 0; k < sc.ncol; k++) b->h_col[k].insert(b->h_col[k].end(), cols[k], cols[k] + sc.col[k].bytes);
    if (n_ios) b->h_ios.insert(b->h_ios.end(), ios, ios + 128 * (size_t)n_ios);
    if (ad_len) b->h_ad.insert(b->h_ad.end(), ad, ad + ad_len);
    b->h_io_off.push_back(b->h_io_off.back() + n_ios);
    b->h_ad_off.push_back(b->h_ad_off.back() + ad_len);
    return 0;
  }
  PushStage* sg = &b->stage[b->cur];
  if (sg->n == STAGE_CHUNK || sg->nio + n_ios > sg->cap_io || sg->nad + ad_len > sg->cap_ad || !sg->free_ev) {
    int rc;
    if (sg->n == STAGE_CHUNK || (sg->n && (sg->nio + n_ios > 4 * PREP_CHUNK || sg->nad + ad_len > 64 * PREP_CHUNK))) {
      if ((rc = flush_stage(b))) return rc;
      sg = &b->stage[b->cur];
    }
    // first use, or a proof with more pairs / additional data than the buffer was sized for
    size_t want_io = std::max<size_t>(sg->cap_io, 2 * PREP_CHUNK), want_ad = std::max<size_t>(sg->cap_ad, 16 * PREP_CHUNK);
    while (want_io < sg->nio + n_ios) want_io *= 2;
    while (want_ad < sg->nad + ad_len) want_ad *= 2;
    if ((rc = bind_device(b->device)) || (rc = stage_reserve(sc, *sg, want_io, want_ad))) return rc;
  }
  size_t j = sg->n;
  StageField f[5];
  for (uint32_t k = 0; k < sc.ncol; k++) f[k] = {sg->col[k].as<uint8_t>() + sc.col[k].bytes * j, cols[k], sc.col[k].bytes};
  stage_proof(f, sc.ncol, sg->ios.as<uint8_t>() + 128 * sg->nio, ios, 128 * (size_t)n_ios);
  if (ad_len) memcpy(sg->ad.as<uint8_t>() + sg->nad, ad, ad_len);
  if (j == 0) { sg->io_off.as<uint32_t>()[0] = 0; sg->ad_off.as<uint32_t>()[0] = 0; }
  sg->nio += n_ios;
  sg->nad += ad_len;
  sg->io_off.as<uint32_t>()[j + 1] = (uint32_t)sg->nio;
  sg->ad_off.as<uint32_t>()[j + 1] = (uint32_t)sg->nad;
  sg->n = j + 1;
  return 0;
}

int avrf_thin_batch_push(avrf_batch* b, const uint8_t pk[64], const uint8_t* ios, uint32_t n_ios, const uint8_t* ad,
                         uint32_t ad_len, const uint8_t r[64], const uint8_t s[32]) {
  if (!b || !pk || !r || !s || (n_ios && !ios) || (ad_len && !ad)) return fail(AVRF_ERR_ARG, "null argument");
  if (b->scheme != 0) return fail(AVRF_ERR_ARG, "not a Thin-VRF batch");
  return push_one(b, {pk, r, s}, ios, n_ios, ad, ad_len);
}

// push_many of arrays that the caller only lends for the duration of the call (thin.rs:218-225): returns once the
// device has consumed them - not the hash, which proceeds on the hasher thread.
static int push_borrowed(avrf_batch* b, uint64_t n, const Columns& cols, const uint8_t* ios, const uint32_t* io_offsets,
                         const uint8_t* ad_blob, const uint32_t* ad_offsets) {
  int rc = check_offsets(n, io_offsets, ad_offsets, ios, ad_blob);
  if (rc) return rc;
  ENTER(b);
  if ((rc = flush_pending(b))) return rc;
  if ((rc = push_many_impl(b, n, cols, ios, io_offsets, ad_blob, ad_offsets))) return rc;
  CK(hsync(b, b->st_h2d));
  CK(hsync(b, b->prepared ? b->st_prep : b->st));
  return 0;
}

int avrf_thin_batch_push_many(avrf_batch* b, uint64_t n, const uint8_t* pk, const uint8_t* ios,
                              const uint32_t* io_offsets, const uint8_t* ad_blob, const uint32_t* ad_offsets,
                              const uint8_t* r, const uint8_t* s) {
  if (!b) return fail(AVRF_ERR_ARG, "null batch");
  if (b->scheme != 0) return fail(AVRF_ERR_ARG, "not a Thin-VRF batch");
  if (n == 0) return 0;
  if (!pk || !io_offsets || !ad_offsets || !r || !s) return fail(AVRF_ERR_ARG, "null argument");
  return push_borrowed(b, n, {pk, r, s}, ios, io_offsets, ad_blob, ad_offsets);
}

// =========================================================================================
// Prepare, seed
// =========================================================================================
int avrf_thin_batch_prepare(avrf_batch* b, int32_t* invalid) {
  ENTER(b);
  int rc = flush_pending(b);
  if (rc) return rc;
  if ((rc = b->flags.reserve(64))) return rc;
  if ((rc = b->h_small.reserve(4096))) return rc;
  if (!b->prepared) {
    if ((rc = grow_derived(b, b->n, b->n_ios))) return rc;
    CK(cudaMemsetAsync(b->flags.p, 0, 64, b->st));
    size_t nch = (b->n + PREP_CHUNK - 1) / PREP_CHUNK;
    while (b->prep_ev.size() < nch) {
      cudaEvent_t e;
      CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      b->prep_ev.push_back(e);
    }
    // one launch per chunk, an event after each: the D2H + host hash of chunk i start while chunk i+1 runs.  The
    // launches go to the handle's high-priority stream: with several handles sharing the GPU the transcripts of this
    // batch (2 ms, and the 82 ms host hash that waits for them) must not queue behind another batch's 8 ms MSM.
    cudaStream_t ps = b->st_prep;
    if ((rc = stream_after(ps, b->st))) return rc;     // inputs and the flag reset are ordered on the compute stream
    if (nch) cudaEventRecord(b->ev[0], ps);
    for (size_t c = 0; c < nch; c++) {
      if ((rc = launch_prepare(b, c * PREP_CHUNK, std::min<size_t>(b->n, (c + 1) * PREP_CHUNK), ps))) return rc;
      CK(cudaEventRecord(b->prep_ev[c], ps));
    }
    if (nch) {
      cudaEventRecord(b->ev[1], ps);
      cudaStreamWaitEvent(b->st, b->ev[1], 0);         // the MSM follows on the compute stream
      b->tm.kernel_launches = nch;
    }
    b->prep_ev_chunks = nch;            // events of THIS batch, all chunks: seed_from_device may overlap on them
    b->prepared = true;
    b->have_seed = false;
  } else {
    // prepared by the push pipeline on st_prep: order the compute stream after it
    if ((rc = stream_after(b->st, b->st_prep))) return rc;
  }
  if (invalid) {
    CK(cudaMemcpyAsync(b->h_small.p, b->flags.p, 8, cudaMemcpyDeviceToHost, b->st));
    CK(hsync(b, b->st));
    int fl = reinterpret_cast<int*>(b->h_small.p)[0];
    if (fl & 2) return fail(AVRF_ERR_ARG, "an input coordinate or scalar is not below its modulus (not a field element)");
    *invalid = fl & 1;
  }
  return 0;
}

int avrf_thin_batch_cs_stream(avrf_batch* b, uint8_t* out) {
  if (!b || !out) return fail(AVRF_ERR_ARG, "null argument");
  int rc = avrf_thin_batch_prepare(b, nullptr);
  if (rc) return rc;
  if (b->n) CK(cudaMemcpyAsync(out, b->cs.p, scheme_of(b).cs_stride * b->n, cudaMemcpyDeviceToHost, b->st));
  CK(hsync(b, b->st));
  return 0;
}

void* avrf_thin_batch_cs_dev(avrf_batch* b) {
  if (!b) { fail(AVRF_ERR_ARG, "null batch"); return nullptr; }
  if (avrf_thin_batch_prepare(b, nullptr)) return nullptr;
  if (hsync(b, b->st) != cudaSuccess) return nullptr;
  return b->cs.p;
}

int avrf_thin_seed(uint32_t suite, const uint8_t* cs_stream, uint64_t n_items, uint8_t seed[64]) {
  return seed_of_stream(suite, cs_stream, n_items, SCHEMES[0].cs_stride, seed);
}

int avrf_pedersen_seed(uint32_t suite, const uint8_t* stream, uint64_t n_items, uint8_t seed[64]) {
  return seed_of_stream(suite, stream, n_items, SCHEMES[1].cs_stride, seed);
}

}  // extern "C"

// Device->host copy of a (c,s) stream in chunks on the copy stream, each chunk hashed on the host
// as soon as it lands: the serial SHA-512 of thin.rs:273-279 (SURVEY.md H1).
static int seed_of_device_stream(cudaStream_t st, cudaStream_t st_copy, uint32_t suite, const uint8_t* cs_dev,
                                 size_t total, PinBuf& pin, uint8_t seed[64]) {
  int rc;
  if ((rc = pin.reserve(total + 64))) return rc;
  const size_t CH = 64 * PREP_CHUNK;      // one k_prepare chunk: 4.6 MiB
  size_t nch = (total + CH - 1) / CH;
  EventPool pool;
  std::vector<cudaEvent_t> evs(nch);
  cudaEvent_t ready = pool.make();
  if (!ready) return fail(AVRF_ERR_CUDA, "cudaEventCreate");
  CK(cudaEventRecord(ready, st));
  CK(cudaStreamWaitEvent(st_copy, ready, 0));
  for (size_t i = 0; i < nch; i++) {
    size_t off = i * CH, len = std::min(CH, total - off);
    CK(cudaMemcpyAsync((uint8_t*)pin.p + off, cs_dev + off, len, cudaMemcpyDeviceToHost, st_copy));
    if (!(evs[i] = pool.make())) return fail(AVRF_ERR_CUDA, "cudaEventCreate");
    CK(cudaEventRecord(evs[i], st_copy));
  }
  unsigned char prefix[40];
  EVP_MD_CTX* ctx = sha512_begin({{prefix, batch_prefix(suite, prefix)}});
  if (!ctx) return AVRF_ERR_NOMEM;
  cudaError_t ce = cudaSuccess;
  for (size_t i = 0; i < nch && ce == cudaSuccess; i++) {
    size_t off = i * CH, len = std::min(CH, total - off);
    ce = cudaEventSynchronize(evs[i]);
    EVP_DigestUpdate(ctx, (uint8_t*)pin.p + off, len);
  }
  sha512_end(ctx, seed);
  if (ce != cudaSuccess) return fail(AVRF_ERR_CUDA, "cudaEventSynchronize", cudaGetErrorString(ce));
  return 0;
}

// The seed of a batch whose (c,s) stream is on the device and was not absorbed at push time (verify after invalidate, a
// handle with eager seeding off): the same hasher thread as the push pipeline - chunked D2H into its pinned staging,
// every chunk absorbed as soon as it lands (and as soon as the k_prepare launch that produces it has finished) - so a
// handle that hashes in a shared multi-buffer pool does so here as well.
static int seed_from_device(avrf_batch* b) {
  Hasher* hs = hasher_of(b);
  if (!hs || b->ext_hasher) return fail(AVRF_ERR_STATE, "no hasher for this handle");
  int rc;
  unsigned char prefix[40];
  if ((rc = hs->begin(prefix, batch_prefix(b->suite, prefix)))) return rc;
  const size_t stride = scheme_of(b).cs_stride, total = stride * b->n, CH = stride * PREP_CHUNK;
  const size_t nch = (total + CH - 1) / CH;
  if ((rc = hs->reserve_stage(std::min(total, 16 * CH) + 64 * (nch + 1)))) return rc;
  const bool per_chunk = b->prep_ev_chunks >= nch && b->prep_ev.size() >= nch;      // this batch's own chunk events
  if (!per_chunk && (rc = stream_after(b->st_copy, b->st))) return rc;
  auto t0 = std::chrono::steady_clock::now();
  for (size_t i = 0; i < nch; i++) {
    size_t off = i * CH, len = std::min(CH, total - off);
    if (per_chunk) CK(cudaStreamWaitEvent(b->st_copy, b->prep_ev[i], 0));
    uint8_t* dst = hs->stage(len);
    if (!dst) return fail(AVRF_ERR_NOMEM, "pinned staging");
    CK(cudaMemcpyAsync(dst, b->cs.as<uint8_t>() + off, len, cudaMemcpyDeviceToHost, b->st_copy));
    cudaEvent_t ev;
    CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming | cudaEventBlockingSync));
    CK(cudaEventRecord(ev, b->st_copy));
    hs->enqueue(ev, dst, len);
  }
  if ((rc = hs->digest(b->seed))) return rc;
  b->tm.host_hash_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  b->have_seed = true;
  return 0;
}

static PinBuf g_pin_stream[AVRF_MAX_DEV];
static std::mutex g_pin_mu;               // guards g_pin_stream (avrf_thin_seed_dev, avrf_pedersen_seed_dev)

// The same seed of a device-resident stream (avrf_thin_seed_dev, avrf_pedersen_seed_dev), on the default device.
static int seed_of_dev_stream(uint32_t suite, const void* stream_dev, uint64_t n_items, size_t stride, uint8_t seed[64]) {
  if (suite > 2 || !seed || (n_items && !stream_dev)) return fail(AVRF_ERR_ARG, "bad argument");
  NEED_DEVICE();
  std::lock_guard<std::mutex> lock(g_pin_mu);
  return seed_of_device_stream(gs(), gc(), suite, (const uint8_t*)stream_dev, stride * n_items, g_pin_stream[g_device.load()],
                               seed);
}

static void seed_to_words(Seed64& sd, const uint8_t seed[64]) {
  for (int i = 0; i < 8; i++) {
    uint64_t w = 0;
    for (int k = 0; k < 8; k++) w = (w << 8) | seed[8 * i + k];
    sd.w[i] = w;
  }
}

// =========================================================================================
// MSM
// =========================================================================================
// Everything after the seed: scalars, sort, accumulate, reduce.  Leaves the partial point in
// b->partial and flags[1] (and in b->remote_slot for the shards of a multi-GPU batch).
static int run_msm(avrf_batch* b, const uint8_t seed[64], uint64_t first_index) {
  int rc;
  const Scheme& sc = scheme_of(b);
  size_t np = sc.points(b->n, b->n_ios);
  if (np >= (1ull << 28)) return fail(AVRF_ERR_ARG, "batch too large for one handle (2^28 MSM terms): shard it");
  size_t max_entries = np * MSM_NWIN;
  uint32_t nblk = cdiv(b->n, 128 * sc.scal_per_thread);
  // accumulation grid: four waves of resident blocks (lazy-reduction additions: 120-126 registers, 4 blocks of 128 threads
  // per SM; Ed25519 5), every thread an equal share of the sorted entries
  // (measured at 2^20 proofs: 1 wave 7.38 ms - the slowest SM sets the time -, 2 waves 7.14, 4 waves 6.99, 8 waves 6.92 with
  // a longer tail of partial sums; the 3616 fixed 128-entry segments of before: 7.07)
  const bool acc_lazy = b->suite != 1;         // Bandersnatch, Baby-JubJub: lazy-reduction addition, 4 blocks per SM
  const uint32_t acc_blocks = (uint32_t)sm_count(b->device) * (acc_lazy ? 4u : 5u) * 4u;
  const uint32_t acc_nthr = acc_blocks * 128u;
  size_t max_slots = (size_t)acc_nthr + MSM_NBINS + 1;
  if ((rc = b->digits.reserve(32 * np))) return rc;
  if ((rc = b->hist.reserve(4 * MSM_NBINS))) return rc;
  if ((rc = b->cursor.reserve(64 * np))) return rc;                  // ranks: 16 x u32 per point
  const size_t np_pad = (np + SORT_TP - 1) / SORT_TP * SORT_TP;
  if ((rc = b->dig_w.reserve(2 * MSM_NWIN * np_pad)) || (rc = b->rank_w.reserve(4 * MSM_NWIN * np_pad))) return rc;
  if ((rc = b->offs.reserve(4 * (MSM_NBINS + 1)))) return rc;
  if ((rc = b->toff.reserve(4 * (MSM_NBINS + 1)))) return rc;       // nzr: rank among non-empty bins
  if ((rc = b->btot.reserve(4 * 1024))) return rc;
  if ((rc = b->totals.reserve(64))) return rc;
  if ((rc = b->entries.reserve(4 * max_entries))) return rc;
  if ((rc = b->tasks.reserve(4 * (size_t)MSM_NBINS))) return rc;    // list of bins with many partial sums
  if ((rc = b->task_out.reserve(sizeof(Ext) * max_slots))) return rc;
  if ((rc = b->chunk_out.reserve(sizeof(Ext) * MSM_NWIN * MSM_NCHUNK))) return rc;
  if ((rc = b->wsum.reserve(sizeof(Ext) * MSM_NWIN))) return rc;
  if ((rc = b->partial.reserve(sizeof(Ext)))) return rc;
  if ((rc = b->gpart.reserve(80 * (size_t)nblk + 80))) return rc;
  if (b->want_taps) {
    if ((rc = b->w_tap.reserve(32 * b->n + 32))) return rc;
    if ((rc = b->scalars_tap.reserve(32 * np))) return rc;
  }
  cudaStream_t st = b->st;
  if (!b->gate_ev) CK(cudaEventCreateWithFlags(&b->gate_ev, cudaEventDisableTiming));
  if (b->segs.size() > 2 && b->segs_dirty) {
    if ((rc = b->segs_dev.reserve(8 * b->segs.size()))) return rc;
    CK(cudaMemcpyAsync(b->segs_dev.p, b->segs.data(), 8 * b->segs.size(), cudaMemcpyHostToDevice, st));
    CK(hsync(b, st));                    // the vector may be modified by the next push
    b->segs_dirty = false;
  }
  MsmGate& gate = g_gate[b->device];
  std::unique_lock<std::mutex> gate_lock(gate.mu);
  if (gate.tail && gate.tail != b->gate_ev) CK(cudaStreamWaitEvent(st, gate.tail, 0));
  CK(cudaMemsetAsync(b->hist.p, 0, 4 * MSM_NBINS, st));

  ScalArgs a;
  a.cs = b->cs.as<uint32_t>(); a.z = b->z.as<uint32_t>(); a.io_off = b->io_off.as<uint32_t>();
  a.digits = b->digits.as<uint4>(); a.hist = b->hist.as<uint32_t>(); a.gpart = b->gpart.as<uint32_t>();
  a.ranks = b->cursor.as<uint4>();
  a.w_tap = b->want_taps ? b->w_tap.as<uint32_t>() : nullptr;
  a.scalars_tap = b->want_taps ? b->scalars_tap.as<Fe>() : nullptr;
  seed_to_words(a.seed, seed);
  a.first_index = b->segs.size() == 2 ? b->segs[1] : first_index;
  a.segs = b->segs.size() > 2 ? b->segs_dev.as<uint64_t>() : nullptr;
  a.nseg = (uint32_t)(b->segs.size() / 2);
  b->first_index = first_index;
  a.n = (uint32_t)b->n;
  uint32_t* hist = b->hist.as<uint32_t>();
  uint32_t* offs = b->offs.as<uint32_t>();
  uint32_t* nzr = b->toff.as<uint32_t>();
  uint32_t* totals = b->totals.as<uint32_t>();
  Ext* slots = b->task_out.as<Ext>();
  cudaEventRecord(b->ev[2], st);
  if (b->scheme == 1) {
    PedScalArgs pa;
    pa.cs = a.cs; pa.digits = a.digits; pa.ranks = a.ranks; pa.hist = a.hist; pa.gpart = a.gpart;
    pa.w_tap = b->want_taps ? b->w_tap.as<uint32_t>() : nullptr;
    pa.scalars_tap = a.scalars_tap; pa.seed = a.seed; pa.first_index = a.first_index; pa.segs = a.segs; pa.nseg = a.nseg;
    pa.n = a.n;
    DISPATCH(b->suite, (k_scalars_ped<S><<<nblk, 128, 0, st>>>(pa)));
    LAUNCHED("k_scalars_ped");
    DISPATCH(b->suite, (k_gscalar_ped<S><<<1, 32, 0, st>>>(a.gpart, nblk, a.digits, a.ranks, a.hist, a.scalars_tap,
                                                            b->pts.as<BaseRec>(), np - 2)));
    LAUNCHED("k_gscalar_ped");
  } else {
    DISPATCH(b->suite, (k_scalars<S><<<nblk, 128, 0, st>>>(a)));
    LAUNCHED("k_scalars");
    DISPATCH(b->suite, (k_gscalar<S><<<1, 256, 0, st>>>(a.gpart, nblk, a.digits, a.ranks, a.hist, a.scalars_tap,
                                                         b->pts.as<BaseRec>(), np - 1)));
    LAUNCHED("k_gscalar");
  }
  cudaEventRecord(b->ev[3], st);
  k_scan_local<<<MSM_NBINS / 1024, 1024, 0, st>>>(hist, offs, nzr, b->btot.as<uint32_t>());
  LAUNCHED("k_scan_local");
  k_scan_totals<<<1, 512, 0, st>>>(b->btot.as<uint32_t>(), totals, offs);
  LAUNCHED("k_scan_totals");
  k_scan_add<<<MSM_NBINS / 1024, 1024, 0, st>>>(offs, nzr, b->btot.as<uint32_t>());
  LAUNCHED("k_scan_add");
  // large batches: window by window with the bin offsets in shared memory (0.85 -> 0.71 ms at 2^20 proofs; what is left is
  // the 59 M partial-sector stores); small ones: one thread per point (the 592 x 128 KiB offset fills would dominate)
  if (np >= (1u << 18)) {
    static std::once_flag smem_once[AVRF_MAX_DEV];
    std::call_once(smem_once[b->device], [] {
      cudaFuncSetAttribute(k_scatter_window, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * MSM_NBUCKET);
    });
    k_sort_transpose<<<cdiv(np, SORT_TP), SORT_TP, 0, st>>>(b->digits.as<uint4>(), b->cursor.as<uint4>(), np, np_pad,
                                                            b->dig_w.as<uint16_t>(), b->rank_w.as<uint32_t>());
    LAUNCHED("k_sort_transpose");
    k_scatter_window<<<dim3(37, MSM_NWIN), 1024, 4 * MSM_NBUCKET, st>>>(b->dig_w.as<uint16_t>(), b->rank_w.as<uint32_t>(), np, np_pad,
                                                                         offs, b->entries.as<uint32_t>());
    LAUNCHED("k_scatter_window");
  } else {
    k_scatter<<<cdiv(np, 256), 256, 0, st>>>(b->digits.as<uint4>(), b->cursor.as<uint4>(), offs,
                                             b->entries.as<uint32_t>(), np);
    LAUNCHED("k_scatter");
  }
  cudaEventRecord(b->ev[4], st);
  AccArgs ac;
  ac.entries = b->entries.as<uint32_t>(); ac.offs = offs; ac.hist = hist; ac.nzr = nzr; ac.totals = totals;
  ac.pts = b->pts.as<BaseRec>(); ac.slots = slots; ac.nthr = acc_nthr;
  // Bandersnatch, Baby-JubJub: the lazy-reduction addition holds three wide products at once: 120-126 registers
  if (b->suite == 0) k_accumulate<0, 4><<<acc_blocks, 128, 0, st>>>(ac);
  else if (b->suite == 2) k_accumulate<2, 4><<<acc_blocks, 128, 0, st>>>(ac);
  else k_accumulate<1, 5><<<acc_blocks, 128, 0, st>>>(ac);
  LAUNCHED("k_accumulate");
  cudaEventRecord(b->ev[5], st);
  CK(cudaEventRecord(b->gate_ev, st));
  gate.tail = b->gate_ev;
  gate_lock.unlock();
  DISPATCH(b->suite, (k_combine<S><<<MSM_NBINS / 128, 128, 0, st>>>(hist, offs, nzr, slots, acc_nthr, totals,
                                                                    b->tasks.as<uint32_t>())));
  LAUNCHED("k_combine");
  DISPATCH(b->suite, (k_combine_big<S><<<64, 256, 0, st>>>(hist, offs, nzr, slots, acc_nthr, totals,
                                                           b->tasks.as<uint32_t>())));
  LAUNCHED("k_combine_big");
  DISPATCH(b->suite, (k_bucket_reduce<S><<<MSM_NWIN * MSM_NCHUNK / 128, 128, 0, st>>>(hist, offs, nzr, acc_nthr, totals, slots,
                                                                                      b->chunk_out.as<Ext>())));
  LAUNCHED("k_bucket_reduce");
  DISPATCH(b->suite, (k_window_sum<S><<<MSM_NWIN, 256, 0, st>>>(b->chunk_out.as<Ext>(), b->wsum.as<Ext>())));
  LAUNCHED("k_window_sum");
  DISPATCH(b->suite, (k_fold<S><<<1, 32, 0, st>>>(b->wsum.as<Ext>(), b->partial.as<Ext>(), b->flags.as<int>(), b->remote_slot)));
  LAUNCHED("k_fold");
  cudaEventRecord(b->ev[6], st);
  b->tm.kernel_launches += 12;
  b->tm.n_points = np;
  return 0;
}

static void collect_timings(avrf_batch* b, bool with_prepare) {
  float ms = 0;
  if (with_prepare && cudaEventElapsedTime(&ms, b->ev[0], b->ev[1]) == cudaSuccess) b->tm.prepare_ms = ms;
  if (cudaEventElapsedTime(&ms, b->ev[2], b->ev[3]) == cudaSuccess) b->tm.scalars_ms = ms;
  if (cudaEventElapsedTime(&ms, b->ev[3], b->ev[4]) == cudaSuccess) b->tm.sort_ms = ms;
  if (cudaEventElapsedTime(&ms, b->ev[4], b->ev[5]) == cudaSuccess) b->tm.accumulate_ms = ms;
  if (cudaEventElapsedTime(&ms, b->ev[5], b->ev[6]) == cudaSuccess) b->tm.reduce_ms = ms;
  (void)cudaGetLastError();   // an event pair that was never recorded (prepare done at push time) is not an error
}

extern "C" {

int avrf_thin_seed_dev(uint32_t suite, const void* cs_stream_dev, uint64_t n_items, uint8_t seed[64]) {
  return seed_of_dev_stream(suite, cs_stream_dev, n_items, SCHEMES[0].cs_stride, seed);
}

int avrf_pedersen_seed_dev(uint32_t suite, const void* stream_dev, uint64_t n_items, uint8_t seed[64]) {
  return seed_of_dev_stream(suite, stream_dev, n_items, SCHEMES[1].cs_stride, seed);
}

int avrf_thin_batch_partial(avrf_batch* b, const uint8_t seed[64], uint64_t first_index, uint8_t partial[128]) {
  if (!b || !seed || !partial) return fail(AVRF_ERR_ARG, "null argument");
  int rc = avrf_thin_batch_prepare(b, nullptr);
  if (rc) return rc;
  memcpy(b->seed, seed, 64);
  b->have_seed = true;
  if ((rc = run_msm(b, seed, first_index))) return rc;
  CK(cudaMemcpyAsync(b->h_small.p, b->partial.p, 128, cudaMemcpyDeviceToHost, b->st));
  CK(cudaMemcpyAsync((uint8_t*)b->h_small.p + 128, b->totals.p, 8, cudaMemcpyDeviceToHost, b->st));
  CK(hsync(b, b->st));
  memcpy(partial, b->h_small.p, 128);
  b->tm.n_entries = reinterpret_cast<uint32_t*>((uint8_t*)b->h_small.p + 128)[0];
  b->tm.n_tasks = reinterpret_cast<uint32_t*>((uint8_t*)b->h_small.p + 128)[1];
  collect_timings(b, true);
  return 0;
}

int avrf_thin_combine_partials(uint32_t suite, const uint8_t* partials, uint32_t n, int32_t* status) {
  if (suite > 2 || !partials || !status || n == 0) return fail(AVRF_ERR_ARG, "bad argument");
  NEED_DEVICE();
  FeedFrame f(g_device.load(), gs());
  DevBuf& in = f.in(partials, 128 * (size_t)n);
  DevBuf& out = f.take(128);
  DevBuf& flags = f.take(64);
  if (f.rc) return f.rc;
  DISPATCH(suite, (k_combine_partials<S><<<1, 32, 0, f.st>>>(in.as<Ext>(), n, out.as<Ext>(), flags.as<int>())));
  LAUNCHED("k_combine_partials");
  int h[2] = {0, 0};
  f.out(h, flags.p, 8);
  int rc = f.sync();
  if (rc) return rc;
  *status = h[1] ? AVRF_OK : AVRF_VERIFICATION_FAILURE;
  return 0;
}

// verify = verify_async + verify_wait.  verify_async enqueues everything up to the device->host copy of the
// verdict words and returns.
int avrf_thin_batch_verify_async(avrf_batch* b) {
  ENTER(b);
  int rc;
  b->t_verify0 = std::chrono::steady_clock::now();
  if ((rc = flush_pending(b))) return rc;
  b->early_status = -1;
  if (b->n == 0) { b->early_status = AVRF_OK; b->inflight = true; return 0; }   // thin.rs:262-264
  bool did_prepare = !b->prepared;
  b->tm = avrf_timings{};
  if (!did_prepare) b->tm.kernel_launches = b->push_launches;
  if ((rc = avrf_thin_batch_prepare(b, nullptr))) return rc;
  if (b->weights_mode == AVRF_WEIGHTS_TREE) {
    uint64_t nl = 0;
    if ((rc = b->h_cs.reserve(64 * ((b->n + TREE_LEAF - 1) / TREE_LEAF) + 64))) return rc;
    auto th = std::chrono::steady_clock::now();
    if ((rc = avrf_thin_batch_tree_leaves(b, 0, (uint8_t*)b->h_cs.p, &nl))) return rc;
    if ((rc = avrf_thin_seed_tree(b->suite, b->n, (const uint8_t*)b->h_cs.p, nl, b->seed))) return rc;
    b->tm.host_hash_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - th).count();
    b->have_seed = true;
  } else if (b->eager && b->hasher && b->hasher->active() && b->hashed == b->n && !did_prepare) {
    // every (c_j, s_j) was queued at push time: wait for the hasher thread, finalise a copy of the running state
    auto th = std::chrono::steady_clock::now();
    if ((rc = b->hasher->digest(b->seed))) return rc;
    b->tm.host_hash_ms = b->hasher->hash_ms();
    b->tm.d2h_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - th).count();   // time verify waited for the hash
    b->have_seed = true;
  } else if ((rc = seed_from_device(b))) return rc;                // also orders after k_prepare
  // The identity gate (thin.rs:266-271) is decided at wait time from flags[0]; it takes precedence over
  // the MSM verdict, so running the MSM regardless does not change any result.
  if ((rc = run_msm(b, b->seed, 0))) return rc;
  CK(cudaMemcpyAsync(b->h_small.p, b->flags.p, 8, cudaMemcpyDeviceToHost, b->st));
  CK(cudaMemcpyAsync((uint8_t*)b->h_small.p + 128, b->totals.p, 8, cudaMemcpyDeviceToHost, b->st));
  if (!b->done_ev) CK(cudaEventCreateWithFlags(&b->done_ev, cudaEventDisableTiming | (b->blocking ? cudaEventBlockingSync : 0)));
  CK(cudaEventRecord(b->done_ev, b->st));
  b->inflight = true;
  b->inflight_did_prepare = did_prepare;
  return 0;
}

int avrf_thin_batch_verify_wait(avrf_batch* b, int32_t* status) {
  if (!b || !status) return fail(AVRF_ERR_ARG, "null argument");
  if (!b->inflight) return fail(AVRF_ERR_STATE, "no verify in flight");
  int rc = bind_device(b->device);
  if (rc) return rc;
  b->inflight = false;
  if (b->early_status >= 0) { *status = b->early_status; return 0; }
  CK(cudaEventSynchronize(b->done_ev));
  const int* fl = reinterpret_cast<const int*>(b->h_small.p);
  if (fl[0] & 2) return fail(AVRF_ERR_ARG, "an input coordinate or scalar is not below its modulus (not a field element)");
  if (fl[0] & 1) *status = AVRF_INVALID_DATA;                                  // thin.rs:266-271
  else *status = fl[1] ? AVRF_OK : AVRF_VERIFICATION_FAILURE;                  // thin.rs:320-324
  b->tm.n_entries = reinterpret_cast<uint32_t*>((uint8_t*)b->h_small.p + 128)[0];
  b->tm.n_tasks = reinterpret_cast<uint32_t*>((uint8_t*)b->h_small.p + 128)[1];
  collect_timings(b, b->inflight_did_prepare);
  b->tm.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - b->t_verify0).count();
  return 0;
}

}  // extern "C"

static int finish_inflight(avrf_batch* b) {
  if (!b->inflight) return 0;
  int32_t st;
  return avrf_thin_batch_verify_wait(b, &st);
}

extern "C" {

int avrf_thin_batch_verify(avrf_batch* b, int32_t* status) {
  if (!b || !status) return fail(AVRF_ERR_ARG, "null argument");
  int rc = avrf_thin_batch_verify_async(b);
  if (rc) return rc;
  return avrf_thin_batch_verify_wait(b, status);
}

// ---- Pedersen VRF batch verifier on the same engine (reference src/pedersen.rs:255-427) -------
avrf_batch* avrf_pedersen_batch_new_on(int device, uint32_t suite, uint32_t fmt) {
  avrf_batch* b = avrf_thin_batch_new_on(device, suite, fmt);
  if (b) b->scheme = 1;      // eager seeding like the thin verifier: push pipelines H2D, k_prepare_ped, D2H and the host SHA-512
  return b;
}

avrf_batch* avrf_pedersen_batch_new(uint32_t suite, uint32_t fmt) { return avrf_pedersen_batch_new_on(-1, suite, fmt); }

int avrf_pedersen_batch_push_many(avrf_batch* b, uint64_t n, const uint8_t* ios, const uint32_t* io_offsets,
                                  const uint8_t* ad_blob, const uint32_t* ad_offsets, const uint8_t* pk_com,
                                  const uint8_t* r, const uint8_t* ok, const uint8_t* s, const uint8_t* sb) {
  if (!b || b->scheme != 1) return fail(AVRF_ERR_ARG, "not a Pedersen batch");
  if (n == 0) return 0;
  if (!io_offsets || !ad_offsets || !pk_com || !r || !ok || !s || !sb) return fail(AVRF_ERR_ARG, "null argument");
  // same pipeline as the thin verifier: chunked H2D -> k_prepare_ped -> D2H of (c, s, sb) -> incremental SHA-512
  return push_borrowed(b, n, {pk_com, r, s, ok, sb}, ios, io_offsets, ad_blob, ad_offsets);
}

// pedersen::BatchVerifier::push (src/pedersen.rs:322-427): one proof, staged exactly as avrf_thin_batch_push stages one.
int avrf_pedersen_batch_push(avrf_batch* b, const uint8_t* ios, uint32_t n_ios, const uint8_t* ad, uint32_t ad_len,
                             const uint8_t pk_com[64], const uint8_t r[64], const uint8_t ok[64], const uint8_t s[32],
                             const uint8_t sb[32]) {
  if (!b || !pk_com || !r || !ok || !s || !sb || (n_ios && !ios) || (ad_len && !ad)) return fail(AVRF_ERR_ARG, "null argument");
  if (b->scheme != 1) return fail(AVRF_ERR_ARG, "not a Pedersen batch");
  return push_one(b, {pk_com, r, s, ok, sb}, ios, n_ios, ad, ad_len);
}

int avrf_pedersen_batch_verify(avrf_batch* b, int32_t* status) {
  if (!b || b->scheme != 1) return fail(AVRF_ERR_ARG, "not a Pedersen batch");
  return avrf_thin_batch_verify(b, status);
}

// ---- the exact single-proof verifiers ---------------------------------------------------------------------------
// One small context per host thread and device: a pinned + a device buffer and a stream, reused across calls.
struct OneCtx {
  int device = -1;
  cudaStream_t st = nullptr;
  PinBuf pin;
  DevBuf dev;
};

// One proof through a single-proof verifier kernel.  Its input on the device: the proof's fixed-size fields (`proof`),
// n_ios (u32), ad_len (u32), 8 zero bytes, the I/O pairs and ad; then `scratch` bytes at the next 256-byte boundary, and
// the two status words after them.  `launch` starts the kernel on the given stream with (input, scratch, status).
using OneLaunch = std::function<int(cudaStream_t, const uint8_t*, uint8_t*, int32_t*)>;
static int run_one(std::initializer_list<ByteRange> proof, const uint8_t* ios, uint32_t n_ios, const uint8_t* ad,
                   uint32_t ad_len, size_t scratch, const OneLaunch& launch, int32_t* status) {
  static thread_local OneCtx ctx;
  int rc, dev = g_device.load();
  if (ctx.device != dev) {
    if (!ctx.st) CK(cudaStreamCreateWithFlags(&ctx.st, cudaStreamNonBlocking));
    ctx.device = dev;
  }
  size_t head = 16;
  for (const ByteRange& f : proof) head += f.n;
  size_t in_bytes = head + 128 * (size_t)n_ios + ad_len;
  size_t scr_off = (in_bytes + 255) & ~(size_t)255, st_off = scr_off + scratch, total = st_off + 64;
  if ((rc = ctx.pin.reserve(total)) || (rc = ctx.dev.reserve(total, 0, ctx.st))) return rc;
  uint8_t* h = ctx.pin.as<uint8_t>();
  for (const ByteRange& f : proof) { memcpy(h, f.p, f.n); h += f.n; }
  memcpy(h, &n_ios, 4);
  memcpy(h + 4, &ad_len, 4);
  memset(h + 8, 0, 8);
  if (n_ios) memcpy(h + 16, ios, 128 * (size_t)n_ios);
  if (ad_len) memcpy(h + 16 + 128 * (size_t)n_ios, ad, ad_len);
  h = ctx.pin.as<uint8_t>();
  uint8_t* d = ctx.dev.as<uint8_t>();
  CK(cudaMemcpyAsync(d, h, in_bytes, cudaMemcpyHostToDevice, ctx.st));
  if ((rc = launch(ctx.st, d, d + scr_off, reinterpret_cast<int32_t*>(d + st_off)))) return rc;
  CK(cudaMemcpyAsync(h + st_off, d + st_off, 8, cudaMemcpyDeviceToHost, ctx.st));
  CK(cudaStreamSynchronize(ctx.st));
  const int32_t* out = reinterpret_cast<const int32_t*>(h + st_off);
  if (out[1] & 2) return fail(AVRF_ERR_ARG, "an input coordinate or scalar is not below its modulus (not a field element)");
  *status = out[0];
  return 0;
}

// thin::Verifier::verify (src/thin.rs:131-165): the exact single-proof equation; 16 bytes of z scratch per pair
int avrf_thin_verify_one(uint32_t suite, uint32_t fmt, const uint8_t pk[64], const uint8_t* ios, uint32_t n_ios,
                         const uint8_t* ad, uint32_t ad_len, const uint8_t r[64], const uint8_t s[32], int32_t* status) {
  if (suite > 2 || fmt > 1) return fail(AVRF_ERR_ARG, "bad suite/fmt");
  if (!pk || !r || !s || !status || (n_ios && !ios) || (ad_len && !ad)) return fail(AVRF_ERR_ARG, "null argument");
  if (n_ios >= (1u << 20)) return fail(AVRF_ERR_ARG, "too many I/O pairs");
  NEED_DEVICE();
  return run_one({{pk, 64}, {r, 64}, {s, 32}}, ios, n_ios, ad, ad_len, 16 * (size_t)n_ios + 16,
                 [&](cudaStream_t st, const uint8_t* in, uint8_t* z, int32_t* out) {
                   OneArgs a;
                   a.in = in;
                   a.z = reinterpret_cast<uint32_t*>(z);
                   a.status = out;
                   a.canonical = fmt == AVRF_FMT_CANONICAL;
                   DISPATCH(suite, (k_verify_one<S><<<1, 32, 0, st>>>(a)));
                   LAUNCHED("k_verify_one");
                   return 0;
                 }, status);
}

// pedersen::Verifier::verify (src/pedersen.rs:188-253): both equations, exact, one thread
int avrf_pedersen_verify_one(uint32_t suite, uint32_t fmt, const uint8_t* ios, uint32_t n_ios, const uint8_t* ad,
                             uint32_t ad_len, const uint8_t pk_com[64], const uint8_t r[64], const uint8_t ok[64],
                             const uint8_t s[32], const uint8_t sb[32], int32_t* status) {
  if (suite > 2 || fmt > 1) return fail(AVRF_ERR_ARG, "bad suite/fmt");
  if (!pk_com || !r || !ok || !s || !sb || !status || (n_ios && !ios) || (ad_len && !ad))
    return fail(AVRF_ERR_ARG, "null argument");
  if (n_ios >= (1u << 20)) return fail(AVRF_ERR_ARG, "too many I/O pairs");
  NEED_DEVICE();
  return run_one({{pk_com, 64}, {r, 64}, {ok, 64}, {s, 32}, {sb, 32}}, ios, n_ios, ad, ad_len, 0,
                 [&](cudaStream_t st, const uint8_t* in, uint8_t*, int32_t* out) {
                   PedOneArgs a;
                   a.in = in;
                   a.status = out;
                   a.canonical = fmt == AVRF_FMT_CANONICAL;
                   DISPATCH(suite, (k_verify_one_ped<S><<<1, 32, 0, st>>>(a)));
                   LAUNCHED("k_verify_one_ped");
                   return 0;
                 }, status);
}

int avrf_thin_batch_timings(const avrf_batch* b, avrf_timings* out) {
  if (!b || !out) return fail(AVRF_ERR_ARG, "null argument");
  *out = b->tm;
  return 0;
}

int avrf_thin_batch_tap(avrf_batch* b, uint32_t what, void* out, size_t out_bytes) {
  if (!b || !out) return fail(AVRF_ERR_ARG, "null argument");
  ENTER(b);
  int rc;
  auto d2h = [&](const void* src, size_t bytes) -> int {
    if (out_bytes < bytes) return fail(AVRF_ERR_ARG, "tap buffer too small");
    if (bytes) CK(cudaMemcpyAsync(out, src, bytes, cudaMemcpyDeviceToHost, b->st));
    CK(hsync(b, b->st));
    return 0;
  };
  switch (what) {
    case AVRF_TAP_C: {
      if ((rc = avrf_thin_batch_prepare(b, nullptr))) return rc;
      if (out_bytes < 16 * b->n) return fail(AVRF_ERR_ARG, "tap buffer too small");
      if (b->n) CK(cudaMemcpy2DAsync(out, 16, b->cs.p, scheme_of(b).cs_stride, 16, b->n, cudaMemcpyDeviceToHost, b->st));
      CK(hsync(b, b->st));
      return 0;
    }
    case AVRF_TAP_Z:
      if ((rc = avrf_thin_batch_prepare(b, nullptr))) return rc;
      return d2h(b->z.p, 16 * b->n_ios);
    case AVRF_TAP_R_COMPRESSED:
      if ((rc = avrf_thin_batch_prepare(b, nullptr))) return rc;
      return d2h(b->renc.p, 32 * b->n);
    case AVRF_TAP_SEED:
      if (!b->have_seed) return fail(AVRF_ERR_STATE, "no seed yet: call verify or partial first");
      if (out_bytes < 64) return fail(AVRF_ERR_ARG, "tap buffer too small");
      memcpy(out, b->seed, 64);
      return 0;
    case AVRF_TAP_W:
    case AVRF_TAP_SCALARS: {
      if (!b->have_seed) return fail(AVRF_ERR_STATE, "no seed yet: call verify or partial first");
      if (b->n == 0) return 0;
      if ((rc = avrf_thin_batch_prepare(b, nullptr))) return rc;
      b->want_taps = true;
      rc = run_msm(b, b->seed, b->first_index);
      b->want_taps = false;
      if (rc) return rc;
      const Scheme& sc = scheme_of(b);
      return what == AVRF_TAP_W ? d2h(b->w_tap.p, sc.w_tap * b->n) : d2h(b->scalars_tap.p, 32 * sc.points(b->n, b->n_ios));
    }
    case AVRF_TAP_PARTIAL:
      if (!b->have_seed || !b->partial.p) return fail(AVRF_ERR_STATE, "no partial yet");
      return d2h(b->partial.p, 128);
    default:
      return fail(AVRF_ERR_ARG, "unknown tap");
  }
}

// Per-proof verdicts of a prepared batch: `launch` writes one status word per proof on b->st, copied back to `statuses`.
static int verdicts(avrf_batch* b, int32_t* statuses, const std::function<int(int32_t*)>& launch) {
  if (b->n == 0) return 0;
  DevBuf dst;
  int rc;
  if ((rc = dst.reserve(4 * b->n, 0, b->st))) return rc;
  if ((rc = launch(dst.as<int32_t>()))) return rc;
  CK(cudaMemcpyAsync(statuses, dst.p, 4 * b->n, cudaMemcpyDeviceToHost, b->st));
  CK(hsync(b, b->st));
  return 0;
}

int avrf_thin_batch_verify_each(avrf_batch* b, int32_t* statuses) {
  if (!b || !statuses) return fail(AVRF_ERR_ARG, "null argument");
  if (b->scheme != 0) return fail(AVRF_ERR_ARG, "not a Thin-VRF batch");
  int rc = avrf_thin_batch_prepare(b, nullptr);
  if (rc) return rc;
  return verdicts(b, statuses, [&](int32_t* out) {
    EachArgs a;
    a.pk = b->pk.as<Affine>(); a.r = b->r.as<Affine>(); a.ios = b->ios.as<Affine>();
    a.canonical = b->fmt == AVRF_FMT_CANONICAL;
    a.cs = b->cs.as<uint32_t>(); a.z = b->z.as<uint32_t>();
    a.io_off = b->io_off.as<uint32_t>(); a.status = out; a.n = (uint32_t)b->n;
    DISPATCH(b->suite, (k_verify_each<S><<<cdiv(b->n, 128), 128, 0, b->st>>>(a)));
    LAUNCHED("k_verify_each");
    return 0;
  });
}

int avrf_pedersen_batch_verify_each(avrf_batch* b, int32_t* statuses) {
  if (!b || !statuses) return fail(AVRF_ERR_ARG, "null argument");
  if (b->scheme != 1) return fail(AVRF_ERR_ARG, "not a Pedersen batch");
  int32_t invalid = 0;                  // (per-proof verdicts below; this call only surfaces out-of-range inputs)
  int rc = avrf_thin_batch_prepare(b, &invalid);
  if (rc) return rc;
  return verdicts(b, statuses, [&](int32_t* out) {
    PedEachArgs a;
    a.pkcom = b->pk.as<Affine>(); a.ios = b->ios.as<Affine>(); a.io_off = b->io_off.as<uint32_t>();
    a.canonical = b->fmt == AVRF_FMT_CANONICAL;
    a.pts = b->pts.as<BaseRec>(); a.cs = b->cs.as<uint32_t>(); a.status = out; a.n = (uint32_t)b->n;
    DISPATCH(b->suite, (k_verify_each_ped<S><<<cdiv(b->n, 128), 128, 0, b->st>>>(a)));
    LAUNCHED("k_verify_each_ped");
    return 0;
  });
}

#include "feed_api.inl"     // hash-to-curve, outputs, proving, ingest, compression, microbenchmarks

}  // extern "C"

#include "server.inl"       // avrf_server_*: worker pool + shared multi-buffer SHA-512 threads, avrf_mb_sha512
#include "sharded.inl"      // avrf_thin_sharded_*: one batch over several GPUs of this process
