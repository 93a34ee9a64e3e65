//! `ark_vrf::gpu` - B200 batch verification of the Thin VRF (and the Pedersen VRF, `gpu::pedersen`) behind the
//! reference's own API.
//!
//! Drop this file in as `src/gpu.rs` of davxy/ark-vrf 0.5.3, add `pub mod gpu;` to `src/lib.rs`
//! behind a `gpu` cargo feature, and link `libavrf_gpu.so` (see INTEGRATION.md).  It keeps the
//! signatures of `thin::BatchVerifier::{new, prepare, push_prepared, push, verify}`
//! (src/thin.rs:198-326) and `thin::Verifier::verify` (src/thin.rs:95-109), forwarding to the C ABI
//! in `include/avrf.h`.  arkworks stores `Fq`/`Fr` as 4x u64 Montgomery limbs (R = 2^256), which is
//! exactly `AVRF_FMT_MONTGOMERY`, so points and scalars are passed as they lie in memory.
//!
//! NOTE: written against the reference sources; there is no Rust toolchain in the build image of
//! ark-vrf_b200, so this module ships uncompiled (the ABI itself is exercised from C++/Python).
#![allow(unsafe_code)] // the crate is #![deny(unsafe_code)] (src/lib.rs:95); FFI needs a scoped allow

use crate::thin::{Proof, ThinSuite};
use crate::{AffinePoint, Error, Public, ScalarField, VrfIo};
use core::marker::PhantomData;

#[repr(C)]
struct AvrfBatch {
    _private: [u8; 0],
}

#[repr(C)]
struct AvrfServer {
    _private: [u8; 0],
}

#[link(name = "avrf_gpu")]
extern "C" {
    fn avrf_init(device: i32) -> i32;
    fn avrf_thin_batch_new(suite: u32, fmt: u32) -> *mut AvrfBatch;
    fn avrf_thin_batch_free(b: *mut AvrfBatch);
    fn avrf_thin_batch_push(
        b: *mut AvrfBatch, pk: *const u8, ios: *const u8, n_ios: u32, ad: *const u8, ad_len: u32,
        r: *const u8, s: *const u8,
    ) -> i32;
    fn avrf_thin_batch_push_many(
        b: *mut AvrfBatch, n: u64, pk: *const u8, ios: *const u8, io_offsets: *const u32,
        ad_blob: *const u8, ad_offsets: *const u32, r: *const u8, s: *const u8,
    ) -> i32;
    fn avrf_thin_batch_push_compressed(
        b: *mut AvrfBatch, n: u64, pk32: *const u8, ios32: *const u8, io_offsets: *const u32,
        ad_blob: *const u8, ad_offsets: *const u32, r32: *const u8, s: *const u8, ok: *mut u8, n_bad: *mut u64,
    ) -> i32;
    fn avrf_thin_batch_verify(b: *mut AvrfBatch, status: *mut i32) -> i32;
    fn avrf_server_new_ex(suite: u32, fmt: u32, n_workers: u32, n_hashers: u32) -> *mut AvrfServer;
    fn avrf_server_free(sv: *mut AvrfServer);
    fn avrf_server_submit(
        sv: *mut AvrfServer, n: u64, pk: *const u8, ios: *const u8, io_offsets: *const u32,
        ad_blob: *const u8, ad_offsets: *const u32, r: *const u8, s: *const u8,
    ) -> i64;
    fn avrf_server_wait(sv: *mut AvrfServer, ticket: i64, status: *mut i32) -> i32;
    fn avrf_server_submit_compressed(
        sv: *mut AvrfServer, n: u64, pk32: *const u8, ios32: *const u8, io_offsets: *const u32,
        ad_blob: *const u8, ad_offsets: *const u32, r32: *const u8, s: *const u8, ok: *mut u8, n_bad: *mut u64,
    ) -> i64;
    fn avrf_pedersen_server_new(suite: u32, fmt: u32, n_workers: u32, n_hashers: u32, n_own: u32) -> *mut AvrfServer;
    fn avrf_pedersen_server_submit(
        sv: *mut AvrfServer, n: u64, ios: *const u8, io_offsets: *const u32, ad_blob: *const u8,
        ad_offsets: *const u32, pk_com: *const u8, r: *const u8, ok: *const u8, s: *const u8, sb: *const u8,
    ) -> i64;
    fn avrf_pedersen_server_submit_compressed(
        sv: *mut AvrfServer, n: u64, ios32: *const u8, io_offsets: *const u32, ad_blob: *const u8,
        ad_offsets: *const u32, proofs: *const u8, ok: *mut u8, n_bad: *mut u64,
    ) -> i64;
    fn avrf_thin_verify_one(
        suite: u32, fmt: u32, pk: *const u8, ios: *const u8, n_ios: u32, ad: *const u8, ad_len: u32,
        r: *const u8, s: *const u8, status: *mut i32,
    ) -> i32;
    fn avrf_thin_batch_reserve(b: *mut AvrfBatch, n: u64, n_ios: u64, ad_bytes: u64) -> i32;
    fn avrf_point_compress(suite: u32, fmt: u32, points: *const u8, n: u64, out32: *mut u8) -> i32;
    fn avrf_init_multi(n_dev: i32, dev_ids: *const i32) -> i32;
    fn avrf_thin_sharded_new(suite: u32, fmt: u32) -> *mut AvrfSharded;
    fn avrf_thin_sharded_free(sh: *mut AvrfSharded);
    fn avrf_thin_sharded_clear(sh: *mut AvrfSharded) -> i32;
    fn avrf_thin_sharded_push_many(
        sh: *mut AvrfSharded, n: u64, pk: *const u8, ios: *const u8, io_offsets: *const u32,
        ad_blob: *const u8, ad_offsets: *const u32, r: *const u8, s: *const u8,
    ) -> i32;
    fn avrf_thin_sharded_verify(sh: *mut AvrfSharded, status: *mut i32) -> i32;
    fn avrf_thin_batch_len(b: *const AvrfBatch) -> i64;
    fn avrf_pedersen_batch_new(suite: u32, fmt: u32) -> *mut AvrfBatch;
    fn avrf_pedersen_batch_push_many(
        b: *mut AvrfBatch, n: u64, ios: *const u8, io_offsets: *const u32, ad_blob: *const u8,
        ad_offsets: *const u32, pk_com: *const u8, r: *const u8, ok: *const u8, s: *const u8, sb: *const u8,
    ) -> i32;
    fn avrf_pedersen_batch_push(
        b: *mut AvrfBatch, ios: *const u8, n_ios: u32, ad: *const u8, ad_len: u32, pk_com: *const u8, r: *const u8,
        ok: *const u8, s: *const u8, sb: *const u8,
    ) -> i32;
    fn avrf_pedersen_batch_push_compressed(
        b: *mut AvrfBatch, n: u64, ios32: *const u8, io_offsets: *const u32, ad_blob: *const u8,
        ad_offsets: *const u32, proofs: *const u8, ok: *mut u8, n_bad: *mut u64,
    ) -> i32;
    fn avrf_pedersen_batch_verify(b: *mut AvrfBatch, status: *mut i32) -> i32;
    fn avrf_pedersen_sharded_new(suite: u32, fmt: u32) -> *mut AvrfSharded;
    fn avrf_pedersen_sharded_push_many(
        sh: *mut AvrfSharded, n: u64, ios: *const u8, io_offsets: *const u32, ad_blob: *const u8,
        ad_offsets: *const u32, pk_com: *const u8, r: *const u8, ok: *const u8, s: *const u8, sb: *const u8,
    ) -> i32;
    fn avrf_pedersen_batch_verify_each(b: *mut AvrfBatch, statuses: *mut i32) -> i32;
    fn avrf_pedersen_verify_one(
        suite: u32, fmt: u32, ios: *const u8, n_ios: u32, ad: *const u8, ad_len: u32, pk_com: *const u8,
        r: *const u8, ok: *const u8, s: *const u8, sb: *const u8, status: *mut i32,
    ) -> i32;
}

#[repr(C)]
struct AvrfSharded {
    _private: [u8; 0],
}

const AVRF_FMT_MONTGOMERY: u32 = 0;

/// Suites the GPU engine implements (SUITE_ID -> `AVRF_SUITE_*`).
pub trait GpuSuite: ThinSuite {
    const AVRF_SUITE: u32;
}
#[cfg(feature = "bandersnatch")]
impl GpuSuite for crate::suites::bandersnatch::BandersnatchSha512Ell2 {
    const AVRF_SUITE: u32 = 0;
}
#[cfg(feature = "ed25519")]
impl GpuSuite for crate::suites::ed25519::Ed25519Sha512Tai {
    const AVRF_SUITE: u32 = 1;
}
#[cfg(feature = "baby-jubjub")]
impl GpuSuite for crate::suites::baby_jubjub::BabyJubJubSha512Tai {
    const AVRF_SUITE: u32 = 2;
}

fn status_to_result(rc: i32, status: i32) -> Result<(), Error> {
    assert!(rc == 0, "libavrf_gpu system error {rc}"); // CUDA / memory: not a verification verdict
    match status {
        0 => Ok(()),
        2 => Err(Error::InvalidData),
        _ => Err(Error::VerificationFailure),
    }
}

/// The shim hands arkworks values to the library as they lie in memory (`AVRF_FMT_MONTGOMERY`).  That relies on
/// three layout facts of arkworks 0.6 that Rust does not promise for `repr(Rust)` types: a twisted-Edwards
/// `Affine` is `{x, y}` = 64 bytes, `Fp` is its four Montgomery limbs = 32 bytes, `VrfIo` is `{input, output}` = 128
/// bytes.  `layout_self_check` turns a violation into a loud failure instead of a wrong verdict: sizes first,
/// then the library's compressed encoding of the generator (computed from the memory image) against arkworks'
/// own `serialize_compressed`.  It runs once per suite, from `BatchVerifier::new`.
pub fn layout_self_check<S: GpuSuite>() {
    use ark_serialize::CanonicalSerialize;
    assert_eq!(core::mem::size_of::<AffinePoint<S>>(), 64, "Affine is not {{x, y}} of 32-byte fields");
    assert_eq!(core::mem::size_of::<ScalarField<S>>(), 32, "Fr is not four 64-bit limbs");
    assert_eq!(core::mem::size_of::<VrfIo<S>>(), 128, "VrfIo is not {{input, output}}");
    assert_eq!(core::mem::size_of::<Proof<S>>(), 96, "thin::Proof is not {{r, s}}");
    let g = S::generator();
    let mut want = [0u8; 32];
    g.serialize_compressed(&mut want[..]).expect("32-byte encoding");
    let mut got = [0u8; 32];
    let rc = unsafe { avrf_point_compress(S::AVRF_SUITE, AVRF_FMT_MONTGOMERY, point_bytes::<S>(&g), 1, got.as_mut_ptr()) };
    assert!(rc == 0, "libavrf_gpu system error {rc}");
    assert_eq!(got, want, "arkworks memory image is not what libavrf_gpu expects (AVRF_FMT_MONTGOMERY)");
}

/// Memory image of a twisted-Edwards `Affine { x, y }` / of `Fr`: 64 / 32 bytes.
fn point_bytes<S: GpuSuite>(p: &AffinePoint<S>) -> *const u8 {
    p as *const AffinePoint<S> as *const u8
}
fn scalar_bytes<S: GpuSuite>(s: &ScalarField<S>) -> *const u8 {
    s as *const ScalarField<S> as *const u8
}

/// Deferred item: like `thin::BatchItem` (src/thin.rs:172-179) but un-hashed - the transcripts are
/// computed on the GPU at `verify`, so `prepare` only copies (it cannot fail, as in the reference).
pub struct BatchItem<S: GpuSuite> {
    pk: Public<S>,
    ios: Vec<VrfIo<S>>,
    ad: Vec<u8>,
    proof: Proof<S>,
}

/// `thin::BatchVerifier` on one B200.
pub struct BatchVerifier<S: GpuSuite> {
    h: *mut AvrfBatch,
    _s: PhantomData<S>,
}

impl<S: GpuSuite> Default for BatchVerifier<S> {
    fn default() -> Self {
        Self::new()
    }
}

impl<S: GpuSuite> BatchVerifier<S> {
    pub fn new() -> Self {
        let h = unsafe {
            avrf_init(0);
            avrf_thin_batch_new(S::AVRF_SUITE, AVRF_FMT_MONTGOMERY)
        };
        assert!(!h.is_null(), "avrf_thin_batch_new failed (no CUDA device?)");
        static CHECKED: std::sync::Once = std::sync::Once::new();     // (one per monomorphisation would be finer still)
        CHECKED.call_once(layout_self_check::<S>);
        Self { h, _s: PhantomData }
    }

    /// Like `Vec::with_capacity`: device memory for `n` proofs up front, so that a loop of `push` never reallocates.
    pub fn with_capacity(n: usize, n_ios: usize, ad_bytes: usize) -> Self {
        let v = Self::new();
        let rc = unsafe { avrf_thin_batch_reserve(v.h, n as u64, n_ios as u64, ad_bytes as u64) };
        assert!(rc == 0, "libavrf_gpu system error {rc}");
        v
    }

    pub fn prepare(
        public: &Public<S>, ios: impl AsRef<[VrfIo<S>]>, ad: impl AsRef<[u8]>, proof: &Proof<S>,
    ) -> BatchItem<S> {
        BatchItem { pk: *public, ios: ios.as_ref().to_vec(), ad: ad.as_ref().to_vec(), proof: proof.clone() }
    }

    pub fn push_prepared(&mut self, e: BatchItem<S>) {
        self.push(&e.pk, &e.ios[..], &e.ad, &e.proof)
    }

    pub fn push(&mut self, public: &Public<S>, ios: impl AsRef<[VrfIo<S>]>, ad: impl AsRef<[u8]>, proof: &Proof<S>) {
        let (ios, ad) = (ios.as_ref(), ad.as_ref());
        // VrfIo<S> is { input: Input(Affine), output: Output(Affine) }: 128 contiguous bytes per pair
        let rc = unsafe {
            avrf_thin_batch_push(
                self.h, point_bytes::<S>(&public.0), ios.as_ptr() as *const u8, ios.len() as u32,
                ad.as_ptr(), ad.len() as u32, point_bytes::<S>(&proof.r), scalar_bytes::<S>(&proof.s),
            )
        };
        assert!(rc == 0, "libavrf_gpu system error {rc}");
    }

    /// Bulk variant for callers that already hold SoA buffers (what the benches use).
    pub fn push_many(
        &mut self, pks: &[AffinePoint<S>], ios: &[VrfIo<S>], io_offsets: &[u32], ad_blob: &[u8],
        ad_offsets: &[u32], rs: &[AffinePoint<S>], ss: &[ScalarField<S>],
    ) {
        let n = pks.len();
        assert!(io_offsets.len() == n + 1 && ad_offsets.len() == n + 1 && rs.len() == n && ss.len() == n);
        let rc = unsafe {
            avrf_thin_batch_push_many(
                self.h, n as u64, pks.as_ptr() as *const u8, ios.as_ptr() as *const u8, io_offsets.as_ptr(),
                ad_blob.as_ptr(), ad_offsets.as_ptr(), rs.as_ptr() as *const u8, ss.as_ptr() as *const u8,
            )
        };
        assert!(rc == 0, "libavrf_gpu system error {rc}");
    }

    /// Proofs still in wire format (`serialize_compressed` bytes: 32 per point, 64 per I/O pair, canonical `s`):
    /// what `Proof::deserialize_compressed` (src/thin.rs:42) and the `Public` / `Input` / `Output` deserialisers
    /// (src/lib.rs:410-433,471-494,552-575) would decode on the CPU is decoded and validated on the GPU.  Returns the
    /// number of proofs that do not deserialize; when it is not zero NOTHING was pushed and `ok[j] == 0` names them.
    pub fn push_compressed(
        &mut self, pk32: &[[u8; 32]], ios32: &[[u8; 64]], io_offsets: &[u32], ad_blob: &[u8],
        ad_offsets: &[u32], r32: &[[u8; 32]], s32: &[[u8; 32]], ok: Option<&mut [u8]>,
    ) -> u64 {
        let n = pk32.len();
        assert!(io_offsets.len() == n + 1 && ad_offsets.len() == n + 1 && r32.len() == n && s32.len() == n);
        let mut bad = 0u64;
        let okp = match ok { Some(v) => { assert!(v.len() >= n); v.as_mut_ptr() } None => core::ptr::null_mut() };
        let rc = unsafe {
            avrf_thin_batch_push_compressed(
                self.h, n as u64, pk32.as_ptr() as *const u8, ios32.as_ptr() as *const u8, io_offsets.as_ptr(),
                ad_blob.as_ptr(), ad_offsets.as_ptr(), r32.as_ptr() as *const u8, s32.as_ptr() as *const u8, okp, &mut bad,
            )
        };
        assert!(rc == 0, "libavrf_gpu system error {rc}");
        bad
    }

    /// Same contract as `thin::BatchVerifier::verify` (src/thin.rs:257-325).
    pub fn verify(&self) -> Result<(), Error> {
        let mut status = -1i32;
        let rc = unsafe { avrf_thin_batch_verify(self.h, &mut status) };
        status_to_result(rc, status)
    }
}

impl<S: GpuSuite> Drop for BatchVerifier<S> {
    fn drop(&mut self) {
        unsafe { avrf_thin_batch_free(self.h) }
    }
}

// A handle owns its device buffers and CUDA streams and the library keeps no mutable global state behind
// it, so a verifier may move to (and be driven from) any thread; different verifiers run concurrently -
// the serial batch-seed SHA-512 of each then occupies its own core.  It is NOT `Sync`: `verify(&self)`
// updates device-side scratch of the handle, one thread at a time per verifier (include/avrf.h).
unsafe impl<S: GpuSuite> Send for BatchVerifier<S> {}

/// `thin::Verifier` on the GPU: the exact equation `s*I_m - c*O_m == R` of src/thin.rs:157-160, no batch weight
/// (csrc/verify_one.cuh).  One proof is ~256 dependent doublings - latency-bound on a GPU; it exists so that the
/// `Verifier` API stays complete and exact, throughput comes from batches.
pub trait Verifier<S: GpuSuite> {
    fn verify_gpu(&self, ios: impl AsRef<[VrfIo<S>]>, ad: impl AsRef<[u8]>, proof: &Proof<S>) -> Result<(), Error>;
}

impl<S: GpuSuite> Verifier<S> for Public<S> {
    fn verify_gpu(&self, ios: impl AsRef<[VrfIo<S>]>, ad: impl AsRef<[u8]>, proof: &Proof<S>) -> Result<(), Error> {
        let (ios, ad) = (ios.as_ref(), ad.as_ref());
        let mut status = -1i32;
        let rc = unsafe {
            avrf_thin_verify_one(
                S::AVRF_SUITE, AVRF_FMT_MONTGOMERY, point_bytes::<S>(&self.0), ios.as_ptr() as *const u8,
                ios.len() as u32, ad.as_ptr(), ad.len() as u32, point_bytes::<S>(&proof.r),
                scalar_bytes::<S>(&proof.s), &mut status,
            )
        };
        status_to_result(rc, status)
    }
}

/// A whole verification job in the flat layout of `avrf_thin_batch_push_many`: what a loop of
/// `BatchVerifier::push` calls (benches/thin.rs:78-81) would have pushed.
pub struct Batch<S: GpuSuite> {
    pk: Vec<AffinePoint<S>>,
    r: Vec<AffinePoint<S>>,
    s: Vec<ScalarField<S>>,
    ios: Vec<VrfIo<S>>,
    io_offsets: Vec<u32>,
    ad: Vec<u8>,
    ad_offsets: Vec<u32>,
}

impl<S: GpuSuite> Default for Batch<S> {
    fn default() -> Self {
        Self { pk: vec![], r: vec![], s: vec![], ios: vec![], io_offsets: vec![0], ad: vec![], ad_offsets: vec![0] }
    }
}

impl<S: GpuSuite> Batch<S> {
    pub fn push(&mut self, public: &Public<S>, ios: impl AsRef<[VrfIo<S>]>, ad: impl AsRef<[u8]>, proof: &Proof<S>) {
        self.pk.push(public.0);
        self.r.push(proof.r);
        self.s.push(proof.s);
        self.ios.extend_from_slice(ios.as_ref());
        self.ad.extend_from_slice(ad.as_ref());
        self.io_offsets.push(self.ios.len() as u32);
        self.ad_offsets.push(self.ad.len() as u32);
    }
}

/// Throughput mode: a native pool of worker threads, one GPU batch verifier each (`avrf_server_*`).
/// Every submitted `Batch` gets the verdict `thin::BatchVerifier::verify` (src/thin.rs:257-325) would
/// return for it; the one serial SHA-512 per batch (thin.rs:273-279) runs on the worker's core while the
/// kernels of all workers share the GPU.
pub struct BatchServer<S: GpuSuite> {
    h: *mut AvrfServer,
    _s: PhantomData<S>,
}

/// A submitted batch; keeps the batch borrowed until the verdict has been read.
pub struct Ticket<'a, S: GpuSuite> {
    id: i64,
    server: &'a BatchServer<S>,
    _batch: PhantomData<&'a Batch<S>>,
}

impl<S: GpuSuite> BatchServer<S> {
    /// `hashers` > 0: that many shared multi-buffer SHA-512 threads (eight batches' hash chains per thread, AVX-512)
    /// instead of one hashing core per worker - for hosts with fewer free cores than batches in flight.
    pub fn new(workers: u32, hashers: u32) -> Self {
        let h = unsafe { avrf_server_new_ex(S::AVRF_SUITE, AVRF_FMT_MONTGOMERY, workers, hashers) };
        assert!(!h.is_null(), "avrf_server_new_ex failed (no CUDA device?)");
        Self { h, _s: PhantomData }
    }

    pub fn submit<'a>(&'a self, b: &'a Batch<S>) -> Ticket<'a, S> {
        let id = unsafe {
            avrf_server_submit(
                self.h, b.pk.len() as u64, b.pk.as_ptr() as *const u8, b.ios.as_ptr() as *const u8,
                b.io_offsets.as_ptr(), b.ad.as_ptr(), b.ad_offsets.as_ptr(), b.r.as_ptr() as *const u8,
                b.s.as_ptr() as *const u8,
            )
        };
        assert!(id >= 0, "libavrf_gpu system error {id}");
        Ticket { id, server: self, _batch: PhantomData }
    }

    /// A batch of proofs in wire format, the arrays of `BatchVerifier::push_compressed`: decoded and validated on the
    /// GPU by the worker.
    pub fn submit_compressed<'a>(
        &'a self, pk32: &'a [[u8; 32]], ios32: &'a [[u8; 64]], io_offsets: &'a [u32], ad_blob: &'a [u8],
        ad_offsets: &'a [u32], r32: &'a [[u8; 32]], s: &'a [[u8; 32]],
    ) -> WireTicket<'a> {
        let n = pk32.len();
        assert!(r32.len() == n && s.len() == n && io_offsets.len() == n + 1 && ad_offsets.len() == n + 1);
        let mut t = WireTicket::new(self.h, n);
        t.id = unsafe {
            avrf_server_submit_compressed(
                self.h, n as u64, pk32.as_ptr() as *const u8, ios32.as_ptr() as *const u8, io_offsets.as_ptr(),
                ad_blob.as_ptr(), ad_offsets.as_ptr(), r32.as_ptr() as *const u8, s.as_ptr() as *const u8,
                t.ok.as_mut_ptr(), &mut *t.n_bad,
            )
        };
        assert!(t.id >= 0, "libavrf_gpu system error {}", t.id);
        t
    }
}

/// A submitted wire-format batch of either scheme: keeps its arrays borrowed and owns the per-proof decode flags the
/// worker fills in.  Dropping it without `wait` still waits, so the worker never writes into freed memory.
pub struct WireTicket<'a> {
    id: i64,
    server: *mut AvrfServer,
    ok: Box<[u8]>,
    n_bad: Box<u64>,
    _borrow: PhantomData<&'a [u8]>,
}

impl<'a> WireTicket<'a> {
    fn new(server: *mut AvrfServer, n: usize) -> Self {
        Self { id: -1, server, ok: vec![0u8; n.max(1)].into_boxed_slice(), n_bad: Box::new(0), _borrow: PhantomData }
    }

    /// Blocks for the verdict and the indices of the proofs that did not deserialize.  When that list is not empty
    /// nothing was verified and the verdict is `Err(Error::InvalidData)`.
    pub fn wait(mut self) -> (Result<(), Error>, Vec<usize>) {
        let mut status = -1i32;
        let rc = unsafe { avrf_server_wait(self.server, self.id, &mut status) };
        self.id = -1;
        let bad = if *self.n_bad > 0 {
            self.ok.iter().enumerate().filter(|(_, &f)| f == 0).map(|(j, _)| j).collect()
        } else {
            Vec::new()
        };
        (status_to_result(rc, status), bad)
    }
}

impl<'a> Drop for WireTicket<'a> {
    fn drop(&mut self) {
        if self.id >= 0 {
            let mut status = -1i32;
            unsafe { avrf_server_wait(self.server, self.id, &mut status) };
        }
    }
}

impl<'a, S: GpuSuite> Ticket<'a, S> {
    /// Blocks for the verdict.
    pub fn wait(self) -> Result<(), Error> {
        let mut status = -1i32;
        let rc = unsafe { avrf_server_wait(self.server.h, self.id, &mut status) };
        status_to_result(rc, status)
    }
}

impl<S: GpuSuite> Drop for BatchServer<S> {
    fn drop(&mut self) {
        unsafe { avrf_server_free(self.h) } // finishes queued batches, joins the workers
    }
}

// submit / wait are internally synchronised (include/avrf.h)
unsafe impl<S: GpuSuite> Send for BatchServer<S> {}
unsafe impl<S: GpuSuite> Sync for BatchServer<S> {}

/// One batch over every GPU of the box, inside this process (`avrf_init_multi` + `avrf_thin_sharded_*`): same seed,
/// weights and verdict as a single-device `BatchVerifier` holding the same proofs in the same order.
pub struct ShardedBatchVerifier<S: GpuSuite> {
    h: *mut AvrfSharded,
    _s: PhantomData<S>,
}

impl<S: GpuSuite> ShardedBatchVerifier<S> {
    /// `n_dev` <= 0: every CUDA device of the box.
    pub fn new(n_dev: i32) -> Self {
        let h = unsafe {
            let rc = avrf_init_multi(n_dev, core::ptr::null());
            assert!(rc == 0, "libavrf_gpu system error {rc}");
            avrf_thin_sharded_new(S::AVRF_SUITE, AVRF_FMT_MONTGOMERY)
        };
        assert!(!h.is_null(), "avrf_thin_sharded_new failed");
        Self { h, _s: PhantomData }
    }
    pub fn push_many(&mut self, b: &Batch<S>) {
        let rc = unsafe {
            avrf_thin_sharded_push_many(
                self.h, b.pk.len() as u64, b.pk.as_ptr() as *const u8, b.ios.as_ptr() as *const u8,
                b.io_offsets.as_ptr(), b.ad.as_ptr(), b.ad_offsets.as_ptr(), b.r.as_ptr() as *const u8,
                b.s.as_ptr() as *const u8,
            )
        };
        assert!(rc == 0, "libavrf_gpu system error {rc}");
    }
    pub fn clear(&mut self) {
        let rc = unsafe { avrf_thin_sharded_clear(self.h) };
        assert!(rc == 0, "libavrf_gpu system error {rc}");
    }
    pub fn verify(&self) -> Result<(), Error> {
        let mut status = -1i32;
        let rc = unsafe { avrf_thin_sharded_verify(self.h, &mut status) };
        status_to_result(rc, status)
    }
}

impl<S: GpuSuite> Drop for ShardedBatchVerifier<S> {
    fn drop(&mut self) {
        unsafe { avrf_thin_sharded_free(self.h) }
    }
}
unsafe impl<S: GpuSuite> Send for ShardedBatchVerifier<S> {}

/// `pedersen::Verifier` and `pedersen::BatchVerifier` (src/pedersen.rs:188-253, 322-427) on the GPU, with per-proof
/// verdicts after a failed batch.  The proof's five fields are passed one by one (each an arkworks memory image, as
/// checked by `layout_self_check`), so `pedersen::Proof`'s own layout does not matter.
pub mod pedersen {
    use super::*;
    use crate::pedersen::{PedersenSuite, Proof};

    /// `pedersen::Verifier::verify` for one proof: exact, both equations (`avrf_pedersen_verify_one`).
    pub fn verify<S: GpuSuite + PedersenSuite>(
        ios: impl AsRef<[VrfIo<S>]>, ad: impl AsRef<[u8]>, proof: &Proof<S>,
    ) -> Result<(), Error> {
        let (ios, ad) = (ios.as_ref(), ad.as_ref());
        let mut status = -1i32;
        let rc = unsafe {
            avrf_pedersen_verify_one(
                S::AVRF_SUITE, AVRF_FMT_MONTGOMERY, ios.as_ptr() as *const u8, ios.len() as u32, ad.as_ptr(),
                ad.len() as u32, point_bytes::<S>(&proof.pk_com), point_bytes::<S>(&proof.r),
                point_bytes::<S>(&proof.ok), scalar_bytes::<S>(&proof.s), scalar_bytes::<S>(&proof.sb), &mut status,
            )
        };
        status_to_result(rc, status)
    }

    /// `pedersen::BatchVerifier` on one B200.
    pub struct BatchVerifier<S: GpuSuite + PedersenSuite> {
        h: *mut AvrfBatch,
        _s: PhantomData<S>,
    }

    impl<S: GpuSuite + PedersenSuite> Default for BatchVerifier<S> {
        fn default() -> Self {
            Self::new()
        }
    }

    impl<S: GpuSuite + PedersenSuite> BatchVerifier<S> {
        pub fn new() -> Self {
            let h = unsafe {
                avrf_init(0);
                avrf_pedersen_batch_new(S::AVRF_SUITE, AVRF_FMT_MONTGOMERY)
            };
            assert!(!h.is_null(), "avrf_pedersen_batch_new failed (no CUDA device?)");
            static CHECKED: std::sync::Once = std::sync::Once::new();
            CHECKED.call_once(layout_self_check::<S>);
            Self { h, _s: PhantomData }
        }

        /// Like `Vec::with_capacity`: device memory for `n` proofs up front, so that a loop of `push` never reallocates.
        pub fn with_capacity(n: usize, n_ios: usize, ad_bytes: usize) -> Self {
            let v = Self::new();
            let rc = unsafe { avrf_thin_batch_reserve(v.h, n as u64, n_ios as u64, ad_bytes as u64) };
            assert!(rc == 0, "libavrf_gpu system error {rc}");
            v
        }

        pub fn push(&mut self, ios: impl AsRef<[VrfIo<S>]>, ad: impl AsRef<[u8]>, proof: &Proof<S>) {
            let (ios, ad) = (ios.as_ref(), ad.as_ref());
            // VrfIo<S> is { input: Input(Affine), output: Output(Affine) }: 128 contiguous bytes per pair
            let rc = unsafe {
                avrf_pedersen_batch_push(
                    self.h, ios.as_ptr() as *const u8, ios.len() as u32, ad.as_ptr(), ad.len() as u32,
                    point_bytes::<S>(&proof.pk_com), point_bytes::<S>(&proof.r), point_bytes::<S>(&proof.ok),
                    scalar_bytes::<S>(&proof.s), scalar_bytes::<S>(&proof.sb),
                )
            };
            assert!(rc == 0, "libavrf_gpu system error {rc}");
        }

        /// Proofs in wire format: `Proof::serialize_compressed` records (pk_com | r | ok | s | sb, 160 bytes) and
        /// compressed (input, output) pairs, decoded and validated on the GPU as `Proof::deserialize_compressed` and the
        /// `Input` / `Output` deserialisers would on the CPU.  Returns the number of proofs that do not deserialize;
        /// when it is not zero NOTHING was pushed and `ok[j] == 0` names them.
        pub fn push_compressed(
            &mut self, ios32: &[[u8; 64]], io_offsets: &[u32], ad_blob: &[u8], ad_offsets: &[u32],
            proofs: &[[u8; 160]], ok: Option<&mut [u8]>,
        ) -> u64 {
            let n = proofs.len();
            assert!(io_offsets.len() == n + 1 && ad_offsets.len() == n + 1);
            let mut bad = 0u64;
            let okp = match ok { Some(v) => { assert!(v.len() >= n); v.as_mut_ptr() } None => core::ptr::null_mut() };
            let rc = unsafe {
                avrf_pedersen_batch_push_compressed(
                    self.h, n as u64, ios32.as_ptr() as *const u8, io_offsets.as_ptr(), ad_blob.as_ptr(),
                    ad_offsets.as_ptr(), proofs.as_ptr() as *const u8, okp, &mut bad,
                )
            };
            assert!(rc == 0, "libavrf_gpu system error {rc}");
            bad
        }

        /// Same contract as `pedersen::BatchVerifier::verify` (src/pedersen.rs:341-426).
        pub fn verify(&self) -> Result<(), Error> {
            let mut status = -1i32;
            let rc = unsafe { avrf_pedersen_batch_verify(self.h, &mut status) };
            status_to_result(rc, status)
        }

        /// `pedersen::Verifier::verify` of every pushed proof, in push order: names the offenders of a failed batch.
        pub fn verify_each(&self) -> Vec<Result<(), Error>> {
            let n = unsafe { avrf_thin_batch_len(self.h) } as usize;
            let mut st = vec![-1i32; n];
            let rc = unsafe { avrf_pedersen_batch_verify_each(self.h, st.as_mut_ptr()) };
            st.into_iter().map(|s| status_to_result(rc, s)).collect()
        }
    }

    impl<S: GpuSuite + PedersenSuite> Drop for BatchVerifier<S> {
        fn drop(&mut self) {
            unsafe { avrf_thin_batch_free(self.h) }
        }
    }
    unsafe impl<S: GpuSuite + PedersenSuite> Send for BatchVerifier<S> {}

    /// The flattened argument list of a whole Pedersen verification, for `BatchServer::submit`.  The proof fields are
    /// kept as their arkworks memory images (`layout_self_check`).
    pub struct Batch<S: GpuSuite + PedersenSuite> {
        pk_com: Vec<[u8; 64]>,
        r: Vec<[u8; 64]>,
        ok: Vec<[u8; 64]>,
        s: Vec<[u8; 32]>,
        sb: Vec<[u8; 32]>,
        ios: Vec<VrfIo<S>>,
        io_offsets: Vec<u32>,
        ad: Vec<u8>,
        ad_offsets: Vec<u32>,
    }

    impl<S: GpuSuite + PedersenSuite> Default for Batch<S> {
        fn default() -> Self {
            Self {
                pk_com: vec![], r: vec![], ok: vec![], s: vec![], sb: vec![], ios: vec![], io_offsets: vec![0], ad: vec![],
                ad_offsets: vec![0],
            }
        }
    }

    impl<S: GpuSuite + PedersenSuite> Batch<S> {
        pub fn push(&mut self, ios: impl AsRef<[VrfIo<S>]>, ad: impl AsRef<[u8]>, proof: &Proof<S>) {
            let pt = |p: &AffinePoint<S>| unsafe { *(point_bytes::<S>(p) as *const [u8; 64]) };
            let sc = |x: &ScalarField<S>| unsafe { *(scalar_bytes::<S>(x) as *const [u8; 32]) };
            self.pk_com.push(pt(&proof.pk_com));
            self.r.push(pt(&proof.r));
            self.ok.push(pt(&proof.ok));
            self.s.push(sc(&proof.s));
            self.sb.push(sc(&proof.sb));
            self.ios.extend_from_slice(ios.as_ref());
            self.ad.extend_from_slice(ad.as_ref());
            self.io_offsets.push(self.ios.len() as u32);
            self.ad_offsets.push(self.ad.len() as u32);
        }
    }

    /// One Pedersen batch over every GPU of the box, inside this process (`avrf_init_multi` +
    /// `avrf_pedersen_sharded_*`, the other `avrf_thin_sharded_*` calls serve both schemes): same seed, weights and
    /// verdict as a single-device `BatchVerifier` holding the same proofs in the same order.
    pub struct ShardedBatchVerifier<S: GpuSuite + PedersenSuite> {
        h: *mut AvrfSharded,
        _s: PhantomData<S>,
    }

    impl<S: GpuSuite + PedersenSuite> ShardedBatchVerifier<S> {
        /// `n_dev` <= 0: every CUDA device of the box.
        pub fn new(n_dev: i32) -> Self {
            let h = unsafe {
                let rc = avrf_init_multi(n_dev, core::ptr::null());
                assert!(rc == 0, "libavrf_gpu system error {rc}");
                avrf_pedersen_sharded_new(S::AVRF_SUITE, AVRF_FMT_MONTGOMERY)
            };
            assert!(!h.is_null(), "avrf_pedersen_sharded_new failed");
            static CHECKED: std::sync::Once = std::sync::Once::new();
            CHECKED.call_once(layout_self_check::<S>);
            Self { h, _s: PhantomData }
        }
        pub fn push_many(&mut self, b: &Batch<S>) {
            let rc = unsafe {
                avrf_pedersen_sharded_push_many(
                    self.h, b.pk_com.len() as u64, b.ios.as_ptr() as *const u8, b.io_offsets.as_ptr(), b.ad.as_ptr(),
                    b.ad_offsets.as_ptr(), b.pk_com.as_ptr() as *const u8, b.r.as_ptr() as *const u8,
                    b.ok.as_ptr() as *const u8, b.s.as_ptr() as *const u8, b.sb.as_ptr() as *const u8,
                )
            };
            assert!(rc == 0, "libavrf_gpu system error {rc}");
        }
        pub fn clear(&mut self) {
            let rc = unsafe { avrf_thin_sharded_clear(self.h) };
            assert!(rc == 0, "libavrf_gpu system error {rc}");
        }
        /// Same contract as `pedersen::BatchVerifier::verify` (src/pedersen.rs:341-426).
        pub fn verify(&self) -> Result<(), Error> {
            let mut status = -1i32;
            let rc = unsafe { avrf_thin_sharded_verify(self.h, &mut status) };
            status_to_result(rc, status)
        }
    }

    impl<S: GpuSuite + PedersenSuite> Drop for ShardedBatchVerifier<S> {
        fn drop(&mut self) {
            unsafe { avrf_thin_sharded_free(self.h) }
        }
    }
    unsafe impl<S: GpuSuite + PedersenSuite> Send for ShardedBatchVerifier<S> {}

    /// Throughput mode for the Pedersen VRF: the worker pool of `gpu::BatchServer`, one Pedersen batch verifier per
    /// worker (`avrf_pedersen_server_new`).  Every submitted batch gets the verdict `pedersen::BatchVerifier::verify`
    /// would return for it.
    pub struct BatchServer<S: GpuSuite + PedersenSuite> {
        h: *mut AvrfServer,
        _s: PhantomData<S>,
    }

    /// A submitted batch; keeps the batch borrowed until the verdict has been read.
    pub struct Ticket<'a, S: GpuSuite + PedersenSuite> {
        id: i64,
        server: &'a BatchServer<S>,
        _batch: PhantomData<&'a Batch<S>>,
    }

    impl<S: GpuSuite + PedersenSuite> BatchServer<S> {
        /// `hashers` > 0: shared multi-buffer SHA-512 threads; `own_hash_workers` of the workers keep a core each.
        pub fn new(workers: u32, hashers: u32, own_hash_workers: u32) -> Self {
            let h = unsafe {
                avrf_init(0);
                avrf_pedersen_server_new(S::AVRF_SUITE, AVRF_FMT_MONTGOMERY, workers, hashers, own_hash_workers)
            };
            assert!(!h.is_null(), "avrf_pedersen_server_new failed (no CUDA device?)");
            static CHECKED: std::sync::Once = std::sync::Once::new();
            CHECKED.call_once(layout_self_check::<S>);
            Self { h, _s: PhantomData }
        }

        pub fn submit<'a>(&'a self, b: &'a Batch<S>) -> Ticket<'a, S> {
            let id = unsafe {
                avrf_pedersen_server_submit(
                    self.h, b.pk_com.len() as u64, b.ios.as_ptr() as *const u8, b.io_offsets.as_ptr(), b.ad.as_ptr(),
                    b.ad_offsets.as_ptr(), b.pk_com.as_ptr() as *const u8, b.r.as_ptr() as *const u8,
                    b.ok.as_ptr() as *const u8, b.s.as_ptr() as *const u8, b.sb.as_ptr() as *const u8,
                )
            };
            assert!(id >= 0, "libavrf_gpu system error {id}");
            Ticket { id, server: self, _batch: PhantomData }
        }

        /// A batch in wire format, the arrays of `BatchVerifier::push_compressed`.
        pub fn submit_compressed<'a>(
            &'a self, ios32: &'a [[u8; 64]], io_offsets: &'a [u32], ad_blob: &'a [u8], ad_offsets: &'a [u32],
            proofs: &'a [[u8; 160]],
        ) -> WireTicket<'a> {
            let n = proofs.len();
            assert!(io_offsets.len() == n + 1 && ad_offsets.len() == n + 1);
            let mut t = WireTicket::new(self.h, n);
            t.id = unsafe {
                avrf_pedersen_server_submit_compressed(
                    self.h, n as u64, ios32.as_ptr() as *const u8, io_offsets.as_ptr(), ad_blob.as_ptr(),
                    ad_offsets.as_ptr(), proofs.as_ptr() as *const u8, t.ok.as_mut_ptr(), &mut *t.n_bad,
                )
            };
            assert!(t.id >= 0, "libavrf_gpu system error {}", t.id);
            t
        }
    }

    impl<'a, S: GpuSuite + PedersenSuite> Ticket<'a, S> {
        /// Blocks for the verdict.
        pub fn wait(self) -> Result<(), Error> {
            let mut status = -1i32;
            let rc = unsafe { avrf_server_wait(self.server.h, self.id, &mut status) };
            status_to_result(rc, status)
        }
    }

    impl<S: GpuSuite + PedersenSuite> Drop for BatchServer<S> {
        fn drop(&mut self) {
            unsafe { avrf_server_free(self.h) } // finishes queued batches, joins the workers
        }
    }
    unsafe impl<S: GpuSuite + PedersenSuite> Send for BatchServer<S> {}
    unsafe impl<S: GpuSuite + PedersenSuite> Sync for BatchServer<S> {}
}
