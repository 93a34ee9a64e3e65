/* avrf.h - C ABI of the B200-native Thin-VRF batch-verification engine (libavrf_gpu.so).
 *
 * The reference (davxy/ark-vrf 0.5.3) is a pure-Rust library with no FFI of its own; this
 * ABI is what a Rust `gpu` module (ark_vrf_b200/rust/gpu.rs, see INTEGRATION.md) binds to
 * keep `thin::BatchVerifier::{new, push, push_prepared, verify}` and `thin::Verifier`
 * unchanged for callers.  Each entry point cites the reference item it stands in for
 * (paths relative to the reference repository root).
 *
 * Conventions
 *  - All pointers are HOST pointers unless a name ends in `_dev`.  Inputs are borrowed for
 *    the duration of the call and copied (reference: src/thin.rs:218-225).
 *  - Field elements are 32-byte little-endian integers.  `fmt` selects how they are to be
 *    read: AVRF_FMT_MONTGOMERY = the arkworks in-memory image (4x u64 limbs, value * 2^256
 *    mod p), so `Affine{x,y}` / `Fr` structs can be passed as they lie in memory;
 *    AVRF_FMT_CANONICAL = plain integers < p.  A point is x (32 B) then y (32 B).
 *    An I/O pair is input point (64 B) then output point (64 B) (src/lib.rs:615-619).
 *    Every coordinate must be < p and every scalar < r in either format (arkworks' field types cannot hold
 *    anything else): verify / prepare return AVRF_ERR_ARG for a batch that contains a larger value.  Whether a
 *    point is on the curve or in the prime subgroup is NOT checked here, exactly as in the reference
 *    (src/thin.rs:78-88); avrf_points_deserialize is the validating entry.
 *  - Return value: 0 on success, < 0 on a system error (CUDA, memory, bad argument) - never
 *    a verification verdict.  Verdicts come back through `status`.
 *  - One process drives one GPU (avrf_init(device)) or several (avrf_init_multi).  Every batch handle lives on one
 *    device and owns its CUDA streams
 *    and buffers: one host thread at a time per handle, different handles may be driven from
 *    different threads concurrently (as the reference's BatchVerifier values may); the
 *    handle-less entry points share one stream and are safe to call from any thread.
 *    avrf_server_* is a ready-made worker pool on top of that (the throughput mode).
 *  - There is no CPU fallback: every entry point that computes fails with
 *    AVRF_ERR_NO_DEVICE when no CUDA device is usable.
 */
#ifndef AVRF_H
#define AVRF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Suites (src/suites/bandersnatch.rs:56-70, ed25519.rs:44-54, baby_jubjub.rs:50-60). */
enum {
  AVRF_SUITE_BANDERSNATCH_SHA512_ELL2 = 0,
  AVRF_SUITE_ED25519_SHA512_TAI = 1,
  AVRF_SUITE_BABYJUBJUB_SHA512_TAI = 2
};

enum { AVRF_FMT_MONTGOMERY = 0, AVRF_FMT_CANONICAL = 1 };

/* Verdicts: the reachable subset of `Error` (src/lib.rs:136-147). */
enum { AVRF_OK = 0, AVRF_VERIFICATION_FAILURE = 1, AVRF_INVALID_DATA = 2 };

/* System errors. */
enum { AVRF_ERR_CUDA = -1, AVRF_ERR_ARG = -2, AVRF_ERR_NOMEM = -3, AVRF_ERR_NO_DEVICE = -4, AVRF_ERR_STATE = -5 };

/* Weight derivation for the random linear combination.
 * AVRF_WEIGHTS_REFERENCE: w_j exactly as src/thin.rs:273-289 (one serial SHA-512 over all
 *   (c_j, s_j); computed on the host, the only step of the path that does not shard).
 * AVRF_WEIGHTS_TREE: seed = SHA512(SUITE_ID || 0x50 || 0x01 || LE64(n) || leaf digests), the
 *   leaf digests (32 proofs each) computed on the GPU.  Same accept/reject (weights are internal:
 *   any collision-resistant hash of all (c_j, s_j) gives sound weights), but not the reference's
 *   transcript bytes, so w_j differ from the reference's; opt-in. */
enum { AVRF_WEIGHTS_REFERENCE = 0, AVRF_WEIGHTS_TREE = 1 };

/* Parity taps (device intermediates copied to the host). */
enum {
  AVRF_TAP_C = 0,           /* 16 B per proof: challenge c_j          (src/utils/common.rs:270-280) */
  AVRF_TAP_Z = 1,           /* 16 B per I/O pair: z_1..z_M per proof  (src/utils/common.rs:335-369) */
  AVRF_TAP_W = 2,           /* 16 B per proof: batch weight w_j       (src/thin.rs:289)             */
  AVRF_TAP_SEED = 3,        /* 64 B: SHA-512 of the batch transcript  (src/thin.rs:273-279)         */
  AVRF_TAP_R_COMPRESSED = 4,/* 32 B per proof: enc(R_j)               (ark-serialize compressed)    */
  AVRF_TAP_PARTIAL = 5,     /* 128 B: this GPU's partial MSM sum, extended coords (X,Y,Z,T), Montgomery */
  AVRF_TAP_SCALARS = 6      /* 32 B per MSM term, canonical, order of src/thin.rs:291-312 then G   */
};

typedef struct avrf_batch avrf_batch;

/* Select the CUDA device of this process and create its streams.  Idempotent. */
int avrf_init(int device);
/* Several GPUs in ONE process: initialise n_dev devices (dev_ids == NULL: 0 .. n_dev-1; n_dev <= 0: all), enable
 * peer access between them (NVLink / NVSwitch) and make the first one the default device of the handle-less
 * entry points and of avrf_thin_batch_new.  avrf_thin_sharded_* then spreads one batch over all of them;
 * avrf_thin_batch_new_on places an ordinary handle on a chosen device. */
int avrf_init_multi(int n_dev, const int* dev_ids);
int avrf_device_count(void);
int avrf_shutdown(void);
const char* avrf_last_error(void);
const char* avrf_version(void);

/* thin::BatchVerifier::new (src/thin.rs:200-202) / Drop. */
avrf_batch* avrf_thin_batch_new(uint32_t suite, uint32_t fmt);
avrf_batch* avrf_thin_batch_new_on(int device, uint32_t suite, uint32_t fmt);   /* device < 0: the default device */
int avrf_thin_batch_device(const avrf_batch* b);
void avrf_thin_batch_free(avrf_batch* b);
/* Room for n proofs, n_ios I/O pairs and ad_bytes of additional data, like Vec::with_capacity: pushes up to that
 * size never reallocate device memory. */
int avrf_thin_batch_reserve(avrf_batch* b, uint64_t n, uint64_t n_ios, uint64_t ad_bytes);
/* Forget all pushed proofs, keep allocations. */
int avrf_thin_batch_clear(avrf_batch* b);
int64_t avrf_thin_batch_len(const avrf_batch* b);
/* Drop the derived state (c_j, z_ij, prepared bases) but keep the pushed inputs in device
 * memory: the next verify re-runs the whole path, prepare included, on resident inputs. */
int avrf_thin_batch_invalidate(avrf_batch* b);
/* Eager seeding (default on): push = H2D + per-proof transcripts + D2H of (c_j, s_j) + incremental host
 * SHA-512 of the batch transcript (src/thin.rs:273-279), pipelined in 75776-proof chunks (one full wave of the
 * transcript kernel).  The hash runs on a thread owned by the handle, so neither push_many nor a loop of single
 * pushes waits for it; verify waits for that thread, finalises the hash and runs the MSM.  Single pushes
 * (avrf_thin_batch_push) are staged in pinned host memory and shipped one chunk at a time while the caller goes
 * on pushing.  Turn off for the shards of a multi-PROCESS batch (the seed there comes from the gathered global
 * stream); must be called on an empty handle. */
int avrf_thin_batch_set_eager(avrf_batch* b, int eager);
/* Streams and threads.  Every batch handle owns its CUDA streams; avrf_thin_batch_stream returns the
 * one (cudaStream_t) its kernels run on, so that callers can bracket calls with events recorded on it.
 * avrf_stream is the stream of the handle-less entry points (hash-to-curve, outputs, proving, ingest).
 * One host thread at a time per handle; DIFFERENT handles may be driven from different host threads
 * concurrently (src/thin.rs: BatchVerifier is plain owned data, Send + Sync) - their host SHA-512s then
 * run in parallel and their kernels share the GPU.  avrf_last_error is per thread. */
void* avrf_stream(void);
void* avrf_thin_batch_stream(avrf_batch* b);
/* Host waits of this handle sleep instead of spinning (default: spin, lowest latency for one handle).  Turn on when
 * several handles are driven from as many threads: the waiting threads then leave the cores to the batch-seed hashes
 * of the other handles (the batch server does this for its workers). */
int avrf_thin_batch_set_blocking(avrf_batch* b, int blocking);
/* Shared multi-buffer hashing: a pool of n_threads host threads, each advancing up to EIGHT batches' SHA-512 chains
 * (src/thin.rs:273-279) in lockstep in the 64-bit lanes of AVX-512 registers - one chain is then ~3x slower than on a
 * core of its own, eight together ~2.5x faster.  For hosts with fewer free cores than batches in flight (e.g. 8 GPUs
 * on 32 cores).  avrf_thin_batch_set_hash_pool moves a handle's batch-seed hash into a lane of the pool (NULL: back
 * to its own thread); call it on an empty handle or follow it with _invalidate.  Digests, hence weights and
 * verdicts, are identical.  The pool must outlive the handles that use it. */
typedef struct avrf_hash_pool avrf_hash_pool;
avrf_hash_pool* avrf_hash_pool_new(uint32_t n_threads);
void avrf_hash_pool_free(avrf_hash_pool* hp);
int avrf_thin_batch_set_hash_pool(avrf_batch* b, avrf_hash_pool* hp);
int avrf_thin_batch_set_weights_mode(avrf_batch* b, uint32_t mode);

/* thin::BatchVerifier::push (src/thin.rs:234-243): one proof.  `ios` = n_ios pairs (128 B each). */
int avrf_thin_batch_push(avrf_batch* b, const uint8_t pk[64], const uint8_t* ios, uint32_t n_ios,
                         const uint8_t* ad, uint32_t ad_len, const uint8_t r[64], const uint8_t s[32]);

/* Bulk push of n proofs.  io_offsets / ad_offsets have n+1 entries (first is 0): proof j owns
 * pairs [io_offsets[j], io_offsets[j+1]) of `ios` and bytes [ad_offsets[j], ad_offsets[j+1])
 * of `ad_blob`.  Data goes straight to device memory (use pinned host buffers for speed). */
int avrf_thin_batch_push_many(avrf_batch* b, uint64_t n, const uint8_t* pk, const uint8_t* ios,
                              const uint32_t* io_offsets, const uint8_t* ad_blob, const uint32_t* ad_offsets,
                              const uint8_t* r, const uint8_t* s);

/* The same for proofs still in WIRE format - what the reference's callers hold before `Proof::deserialize_compressed`
 * (src/thin.rs:42) and the `Public` / `Input` / `Output` deserialisers (src/lib.rs:410-433,471-494,552-575): pk32 and r32
 * are n x 32-byte compressed points, ios32 is 64 bytes per pair (input, output), s is n x 32 bytes canonical
 * little-endian.  The points are decoded and validated on the device (on-curve, prime-order subgroup; identity
 * rejected for pk / I / O, allowed for R) and enter the push pipeline without a round trip: 160 instead of 296 bytes
 * per proof cross PCIe at M = 1.  All or nothing, as in the reference where a proof that fails to deserialize never
 * reaches push: when any proof does not decode, *n_bad is their number, ok[j] (optional, n bytes) is 0 for them, and
 * NOTHING is pushed.  Works with handles of either format. */
int avrf_thin_batch_push_compressed(avrf_batch* b, uint64_t n, const uint8_t* pk32, const uint8_t* ios32,
                                    const uint32_t* io_offsets, const uint8_t* ad_blob, const uint32_t* ad_offsets,
                                    const uint8_t* r32, const uint8_t* s, uint8_t* ok, uint64_t* n_bad);

/* thin::BatchVerifier::verify (src/thin.rs:257-325).  Repeatable, does not consume items. */
int avrf_thin_batch_verify(avrf_batch* b, int32_t* status);

/* The same verify split in two for pipelined serving: _async enqueues the MSM on the GPU and returns,
 * _wait blocks for the verdict.  With eager seeding the host is free between the two calls, so the next
 * batch's push (its SHA-512 and its own prepare kernels on a high-priority stream) overlaps this batch's MSM.
 * Any other call on the handle completes a verify that is still in flight first. */
int avrf_thin_batch_verify_async(avrf_batch* b);
int avrf_thin_batch_verify_wait(avrf_batch* b, int32_t* status);

/* thin::Verifier::verify (src/thin.rs:131-165): the exact equation s*I_m - c*O_m == R of the reference, with no
 * batch weight (a small-order component on R can never cancel, whatever (c, s) are) and none of the batch
 * machinery - one single-warp kernel, a per-thread context reused across calls.  Exact on every curve point, in
 * the prime-order subgroup or not (csrc/verify_one.cuh).  A single proof is a chain of ~256 dependent point
 * doublings: latency-bound on a GPU (use a batch for throughput). */
int avrf_thin_verify_one(uint32_t suite, uint32_t fmt, const uint8_t pk[64], const uint8_t* ios, uint32_t n_ios,
                         const uint8_t* ad, uint32_t ad_len, const uint8_t r[64], const uint8_t s[32],
                         int32_t* status);

/* Per-proof verdicts (the reference only reports "some proof is bad"): thin::Verifier::verify
 * (src/thin.rs:131-165) for every pushed proof, statuses[j] in {AVRF_OK, AVRF_VERIFICATION_FAILURE,
 * AVRF_INVALID_DATA}.  Use after a failed batch to name the offenders. */
int avrf_thin_batch_verify_each(avrf_batch* b, int32_t* statuses);

/* ---- Sharded verification (one batch over several GPUs / processes) --------------------
 * rank-local:  avrf_thin_batch_prepare -> avrf_thin_batch_cs_stream  (gather streams, in
 * global proof order, on every rank) -> avrf_thin_seed -> avrf_thin_batch_partial
 * (first_index = global index of this shard's first proof) -> gather the 128-byte partials
 * -> avrf_thin_combine_partials on any rank. */

/* BatchVerifier::prepare for every pushed proof (src/thin.rs:209-226) on the GPU.
 * `invalid` (may be NULL) receives 1 if any pk / I / O is the identity (src/thin.rs:266-271). */
int avrf_thin_batch_prepare(avrf_batch* b, int32_t* invalid);
/* 64 bytes per proof: LE32(c_j) || LE32(s_j), the bytes src/thin.rs:276-279 absorbs. */
int avrf_thin_batch_cs_stream(avrf_batch* b, uint8_t* out);
/* Device address of the same stream (valid until the next push / clear), for a device-side
 * all-gather; avrf_thin_seed_dev hashes a device-resident stream (chunked D2H overlapped with the
 * host SHA-512). */
void* avrf_thin_batch_cs_dev(avrf_batch* b);
int avrf_thin_seed_dev(uint32_t suite, const void* cs_stream_dev, uint64_t n_items, uint8_t seed[64]);
/* seed = SHA512(SUITE_ID || 0x50 || stream)  (src/thin.rs:274-279; host, serial). */
int avrf_thin_seed(uint32_t suite, const uint8_t* cs_stream, uint64_t n_items, uint8_t seed[64]);
/* AVRF_WEIGHTS_TREE building blocks: leaf_i = SHA512(0x00 || LE64(i) || (c,s) stream of proofs 32i..32i+31),
 * seed = SHA512(SUITE_ID || 0x50 || 0x01 || LE64(n_total) || leaf_0 || leaf_1 || ...).  first_index % 32 == 0. */
int avrf_thin_batch_tree_leaves(avrf_batch* b, uint64_t first_index, uint8_t* out, uint64_t* n_leaves);
int avrf_thin_seed_tree(uint32_t suite, uint64_t n_total, const uint8_t* leaves, uint64_t n_leaves, uint8_t seed[64]);
/* This shard's share of the MSM of src/thin.rs:282-319 (incl. its share of the G term). */
int avrf_thin_batch_partial(avrf_batch* b, const uint8_t seed[64], uint64_t first_index, uint8_t partial[128]);
/* Sum n partials and test for the identity (src/thin.rs:320-324): *status = OK / VERIFICATION_FAILURE. */
int avrf_thin_combine_partials(uint32_t suite, const uint8_t* partials, uint32_t n, int32_t* status);

int avrf_thin_batch_tap(avrf_batch* b, uint32_t what, void* out, size_t out_bytes);

/* ---- Multi-GPU batches inside the library (one process, several devices; avrf_init_multi first) ------------
 * thin::BatchVerifier (src/thin.rs:198-325) over all initialised devices.  Every push is cut into contiguous
 * parts, one per device; the devices run the per-proof transcripts of their parts while ONE host thread absorbs
 * the (c_j, s_j) chunks of all of them in global proof order (the serial SHA-512 of src/thin.rs:273-279 runs once,
 * on one core).  verify: every device reduces its proofs to one partial point (weights addressed by global index,
 * src/thin.rs:289), the tail of its fold kernel stores the partial and the identity-gate flag into a peer-mapped
 * slot on the first device, which adds the slots and writes the verdict (src/thin.rs:320-324).  Seed, weights and
 * verdict are bit-identical to a single-device handle holding the same proofs in the same order.
 * avrf_thin_sharded_shard returns the ordinary handle of one device (taps, timings; do not push to it). */
typedef struct avrf_sharded avrf_sharded;
typedef struct avrf_sharded_timings {
  float hash_wait_ms;      /* verify waited this long for the hashing thread */
  float host_hash_ms;      /* time that thread spent in SHA-512 for the batch */
  float issue_ms;          /* host time to enqueue the MSM kernels of all devices */
  float device_wait_ms;    /* from the last launch to the verdict on the host */
  float total_ms;
  float shard_msm_ms_max;  /* slowest device: scalars + sort + accumulate + reduce */
} avrf_sharded_timings;
avrf_sharded* avrf_thin_sharded_new(uint32_t suite, uint32_t fmt);
void avrf_thin_sharded_free(avrf_sharded* sh);
int avrf_thin_sharded_devices(const avrf_sharded* sh);
int64_t avrf_thin_sharded_len(const avrf_sharded* sh);
int avrf_thin_sharded_clear(avrf_sharded* sh);
int avrf_thin_sharded_push_many(avrf_sharded* sh, uint64_t n, const uint8_t* pk, const uint8_t* ios,
                                const uint32_t* io_offsets, const uint8_t* ad_blob, const uint32_t* ad_offsets,
                                const uint8_t* r, const uint8_t* s);
int avrf_thin_sharded_verify(avrf_sharded* sh, int32_t* status);
int avrf_thin_sharded_seed(const avrf_sharded* sh, uint8_t seed[64]);
int avrf_thin_sharded_timings(const avrf_sharded* sh, avrf_sharded_timings* out);
avrf_batch* avrf_thin_sharded_shard(avrf_sharded* sh, int index);

/* ---- Pedersen VRF batch verifier (SURVEY 8f-3; reference src/pedersen.rs:255-427) on the same MSM engine ---
 * pedersen::BatchVerifier::new / push (x n) / verify.  The handle is an avrf_batch: _free, _clear, _len,
 * _tap (C, SEED, W = t_i||u_i, SCALARS) apply; proofs are (pk_com 64, r 64, ok 64, s 32, sb 32). */
avrf_batch* avrf_pedersen_batch_new(uint32_t suite, uint32_t fmt);
int avrf_pedersen_batch_push_many(avrf_batch* b, uint64_t n, const uint8_t* ios, const uint32_t* io_offsets,
                                  const uint8_t* ad_blob, const uint32_t* ad_offsets, const uint8_t* pk_com,
                                  const uint8_t* r, const uint8_t* ok, const uint8_t* s, const uint8_t* sb);
int avrf_pedersen_batch_verify(avrf_batch* b, int32_t* status);

/* The same push for proofs in WIRE format: `proofs` is n records of 160 bytes, each exactly
 * pedersen::Proof::serialize_compressed (pk_com 32 | r 32 | ok 32 | s 32 | sb 32, src/pedersen.rs:43-50: compressed
 * points, canonical little-endian scalars), and ios32 is 64 bytes per pair (input, output) as in
 * avrf_thin_batch_push_compressed.  Decoded and validated on the device: pk_com, R and Ok are bare points (on the curve,
 * prime-order subgroup, identity allowed: an identity pk_com decodes and verify then reports InvalidData); I and O are
 * Input / Output (identity refused); s >= r or sb >= r fails the proof's deserialisation.  224 instead of 384 bytes per
 * proof cross PCIe at M = 1.  All or nothing: when any proof does not decode, *n_bad is their number, ok[j] (optional,
 * n bytes) is 0 for them, and NOTHING is pushed - a handle that held proofs keeps exactly those, and their seed.
 * A Thin handle is an argument error.  Works with handles of either format. */
int avrf_pedersen_batch_push_compressed(avrf_batch* b, uint64_t n, const uint8_t* ios32, const uint32_t* io_offsets,
                                        const uint8_t* ad_blob, const uint32_t* ad_offsets, const uint8_t* proofs,
                                        uint8_t* ok, uint64_t* n_bad);

/* pedersen::Verifier::verify (src/pedersen.rs:188-253) for every proof pushed to a Pedersen handle: statuses[j] in
 * {AVRF_OK, AVRF_VERIFICATION_FAILURE, AVRF_INVALID_DATA}, each proof judged on its own as avrf_pedersen_verify_one
 * would.  Use after a failed batch to name the offenders.  Runs on the handle's stream; a Thin handle is an argument
 * error (and avrf_thin_batch_verify_each refuses Pedersen handles). */
int avrf_pedersen_batch_verify_each(avrf_batch* b, int32_t* statuses);

/* pedersen::Verifier::verify (src/pedersen.rs:188-253) for ONE proof, exact: InvalidData when pk_com or an I/O point
 * is the identity (before any equation), otherwise Ok when BOTH s*I_m - c*O_m == Ok and s*G + sb*B - c*pk_com == R
 * hold, each tested with integer scalars and no batch weight (exact on every curve point, in the prime-order subgroup
 * or not).  A coordinate >= p or s / sb >= r is AVRF_ERR_ARG (status untouched).  Uses a per-thread context, as
 * avrf_thin_verify_one does; latency-bound (use a batch for throughput). */
int avrf_pedersen_verify_one(uint32_t suite, uint32_t fmt, const uint8_t* ios, uint32_t n_ios, const uint8_t* ad,
                             uint32_t ad_len, const uint8_t pk_com[64], const uint8_t r[64], const uint8_t ok[64],
                             const uint8_t s[32], const uint8_t sb[32], int32_t* status);

/* ---- Feeder operations (inputs of the hot path; also the synthetic-data generator) ------ */

/* Input::new -> Suite::data_to_point (src/lib.rs:500-502; Elligator2-XMD for Bandersnatch,
 * src/utils/hash_to_curve.rs:66-100; try-and-increment otherwise, :34-57).
 * msgs = blob, offsets n+1 entries.  out_affine (64 B each, in `fmt`) and out_compressed
 * (32 B each) may each be NULL.  ok (may be NULL): 1 per message, 0 where no point was found. */
int avrf_hash_to_curve(uint32_t suite, uint32_t fmt, const uint8_t* msgs, const uint32_t* offsets, uint64_t n,
                       uint8_t* out_affine, uint8_t* out_compressed, uint8_t* ok);

/* Secret::output (src/lib.rs:391-393): out_j = sk_j * input_j.  sk: n scalars (sk_stride = 32)
 * or one shared scalar (sk_stride = 0). */
int avrf_vrf_output(uint32_t suite, uint32_t fmt, const uint8_t* sk, uint32_t sk_stride, const uint8_t* inputs,
                    uint64_t n, uint8_t* outputs);

/* Input::new + Secret::output (+ Output::hash) for n messages in ONE call (BASELINE.json configs[4]): the input points
 * stay on the device between hash-to-curve and the scalar multiplication, every field inversion is batched.
 * out_inputs / out_outputs (64 B each, in `fmt`), out_hashes (32 B each: point_to_hash of the output,
 * src/utils/common.rs:290-305) and ok (1 B each) may each be NULL. */
int avrf_vrf_io_many(uint32_t suite, uint32_t fmt, const uint8_t* msgs, const uint32_t* offsets, uint64_t n, const uint8_t* sk,
                     uint32_t sk_stride, uint8_t* out_inputs, uint8_t* out_outputs, uint8_t* out_hashes, uint8_t* ok);

/* Secret::from_scalar's public key (src/lib.rs:331-334): pk_j = sk_j * G. */
int avrf_public_keys(uint32_t suite, uint32_t fmt, const uint8_t* sk, uint64_t n, uint8_t* pk);

/* thin::Prover::prove (src/thin.rs:111-129) for n proofs; layout as push_many, plus sk (32 B each)
 * and pk (64 B each).  Outputs r (64 B each) and s (32 B each) in `fmt`. */
int avrf_thin_prove_many(uint32_t suite, uint32_t fmt, uint64_t n, const uint8_t* sk, const uint8_t* pk,
                         const uint8_t* ios, const uint32_t* io_offsets, const uint8_t* ad_blob,
                         const uint32_t* ad_offsets, uint8_t* r, uint8_t* s);

/* pedersen::Prover::prove (src/pedersen.rs:136-186) for n proofs; layout as avrf_thin_prove_many (pk = sk*G).
 * Outputs in `fmt`: pk_com, r, ok (64 B each), s, sb (32 B each); blinding (32 B each, may be NULL) = the blinding
 * factor the reference returns beside the proof. */
int avrf_pedersen_prove_many(uint32_t suite, uint32_t fmt, uint64_t n, const uint8_t* sk, const uint8_t* pk,
                             const uint8_t* ios, const uint32_t* io_offsets, const uint8_t* ad_blob,
                             const uint32_t* ad_offsets, uint8_t* pk_com, uint8_t* r, uint8_t* ok, uint8_t* s,
                             uint8_t* sb, uint8_t* blinding);

/* CanonicalSerialize of affine points (ark-serialize compressed; src/utils/transcript.rs:48-50). */
int avrf_point_compress(uint32_t suite, uint32_t fmt, const uint8_t* points, uint64_t n, uint8_t* out32);

/* CanonicalDeserialize (compressed, Validate::Yes) of n 32-byte points: kind 0 = bare AffinePoint
 * (Proof.r, src/thin.rs:42: on-curve + prime-subgroup check, identity allowed), kind 1 = Public / Input /
 * Output (src/lib.rs:410-433,471-494,552-575: identity rejected too).  ok[j] = 1 when valid; invalid
 * entries decode to the identity.  The subgroup test is [r]P == O for the cofactor-8 curves and a 2-descent (two
 * quadratic characters, same verdict, ~5x cheaper) for Bandersnatch. */
int avrf_points_deserialize(uint32_t suite, uint32_t fmt, uint32_t kind, const uint8_t* in32, uint64_t n, uint8_t* out64,
                            uint8_t* ok);

/* Output::hash / point_to_hash (src/utils/common.rs:290-305), 32 bytes per point. */
int avrf_point_to_hash(uint32_t suite, uint32_t fmt, const uint8_t* points, uint64_t n, uint8_t* out32);

/* ---- Measurement helpers -------------------------------------------------------------- */

/* Per-phase device times (ms) of the last verify / partial call on this handle.  With eager seeding host_hash_ms
 * is the time the hashing thread spent in SHA-512 for the batch and d2h_ms the time verify waited for it. */
typedef struct avrf_timings {
  float h2d_ms, prepare_ms, d2h_ms, host_hash_ms, scalars_ms, sort_ms, accumulate_ms, reduce_ms, total_ms;
  uint64_t n_points, n_entries, n_tasks, kernel_launches;
} avrf_timings;
int avrf_thin_batch_timings(const avrf_batch* b, avrf_timings* out);

/* Integer-multiply roofline probe: runs dependency-free multiply streams on every SM and returns
 * operations per second:
 *   kind 0: wide MACs (IMAD.WIDE.U32);
 *   kind 1: Montgomery multiplications;
 *   kind 2: mixed point additions;
 *   kind 3: wide MACs in the carry-chained rows of the field multiplication (IMAD.WIDE.U32.X);
 *   kind 4: 32-bit MACs (IMAD);
 *   kind 6, 7: wide MACs with the carry out only / the carry in only.
 * Any other kind is AVRF_ERR_ARG. */
int avrf_microbench(uint32_t kind, uint32_t iters, double* per_second, float* ms);

/* ---- Batch server: the throughput mode -----------------------------------------------------
 * A pool of n_workers host threads, each owning one batch handle (own CUDA streams).  A submitted
 * batch is a whole thin::BatchVerifier job - new, push of n proofs, verify (src/thin.rs:200-325) -
 * taken by the next free worker; its serial batch-seed SHA-512 (thin.rs:273-279) occupies that
 * worker's core while the kernels of all workers share the GPU.  One caller thread can keep the
 * GPU busy this way: 16 workers verify 2^20-proof batches at 6-7x the one-at-a-time rate.
 * submit takes the arguments of avrf_thin_batch_push_many and returns a ticket (>= 0) or an error
 * (< 0); the buffers are BORROWED until avrf_server_wait returns for that ticket.  wait blocks for
 * the verdict (*status: AVRF_OK / AVRF_VERIFICATION_FAILURE / AVRF_INVALID_DATA); each ticket can be
 * waited on once.  avrf_server_free finishes the queued batches, then stops the workers.
 * submit/wait may be called from any threads. */
typedef struct avrf_server avrf_server;
avrf_server* avrf_server_new(uint32_t suite, uint32_t fmt, uint32_t n_workers);
/* The same pool with n_hashers shared multi-buffer SHA-512 threads (0 = none, as avrf_server_new): worker i hands
 * the (c_j, s_j) stream of its batch to hasher i % n_hashers, which advances up to eight batches' hash chains in
 * lockstep in the 64-bit lanes of AVX-512 registers (4-5x the aggregate rate of one core hashing one stream; plain
 * lane-after-lane hashing on CPUs without AVX-512).  Same digests, hence the same weights and verdicts.  Use it when
 * the box has fewer free cores than batches in flight, e.g. 8 GPUs on 32 cores: n_workers = 8 * n_hashers. */
avrf_server* avrf_server_new_ex(uint32_t suite, uint32_t fmt, uint32_t n_workers, uint32_t n_hashers);
/* Mixed pool: workers 0 .. n_own-1 hash their batches on their own thread (one core each, the lowest latency per
 * batch), the others share the n_hashers multi-buffer threads.  For a burst of more batches than the host has cores.
 * A submitted batch goes to an idle shared-lane worker first and to an own-thread worker only when none is idle: the
 * early arrivals of a burst can afford the slower lanes, the late ones - whose hash ends the burst - get a core. */
avrf_server* avrf_server_new_mixed(uint32_t suite, uint32_t fmt, uint32_t n_workers, uint32_t n_hashers, uint32_t n_own);
void avrf_server_free(avrf_server* sv);
int64_t avrf_server_submit(avrf_server* sv, uint64_t n, const uint8_t* pk, const uint8_t* ios,
                           const uint32_t* io_offsets, const uint8_t* ad_blob, const uint32_t* ad_offsets,
                           const uint8_t* r, const uint8_t* s);
int avrf_server_wait(avrf_server* sv, int64_t ticket, int32_t* status);

/* Host-only utility: SHA-512 of n_streams independent byte streams through the batch server's multi-buffer hasher,
 * fed in interleaved chunk-byte updates; digests = 64 bytes per stream.  *simd (optional) = 1 if the AVX-512 path ran.
 * Needs no GPU (tests and diagnostics). */
int avrf_mb_sha512(uint32_t n_streams, const uint8_t* const* data, const uint64_t* lens, uint64_t chunk,
                   uint8_t* digests, int32_t* simd);

#ifdef __cplusplus
}
#endif
#endif /* AVRF_H */
