// Per-proof transcript kernels of the batch verifiers: one thread per proof.
//   k_prepare      thin::BatchVerifier::prepare (reference src/thin.rs:209-226) + identity gate (thin.rs:266-271)
//   k_prepare_ped  pedersen::BatchItem::new (reference src/pedersen.rs:283-301)
//   k_tree_leaves  leaf digests of the opt-in tree seed (AVRF_WEIGHTS_TREE)
#pragma once
#include "msm.cuh"
#include "pedersen.cuh"

namespace avrf {
// A field element of the ABI must be < p in either format (arkworks' types cannot hold anything else); anything
// larger would be silently mis-reduced by the Montgomery arithmetic, so it is reported as an argument error.
template <int F>
__device__ __forceinline__ bool fe_in_range(const Fe& a) { return limbs_gt(AVRF_FC(F).p, a.v); }

template <int S>
__device__ __forceinline__ void load_affine_fmt(Affine& p, const Affine* src, int canonical, int* oob = nullptr) {
  load_fe(p.x, &src->x);
  load_fe(p.y, &src->y);
  if (oob) *oob |= !(fe_in_range<SuiteT<S>::FQ>(p.x) && fe_in_range<SuiteT<S>::FQ>(p.y));
  if (canonical) {
    to_mont<SuiteT<S>::FQ>(p.x, p.x);
    to_mont<SuiteT<S>::FQ>(p.y, p.y);
  }
}

template <int S>
__device__ __forceinline__ void store_affine_fmt(Affine* dst, const Affine& p, int canonical) {
  Affine q = p;
  if (canonical) {
    from_mont<SuiteT<S>::FQ>(q.x, q.x);
    from_mont<SuiteT<S>::FQ>(q.y, q.y);
  }
  store_fe(&dst->x, q.x);
  store_fe(&dst->y, q.y);
}

__device__ __forceinline__ void store_affinek(BaseRec* dst, const AffineK& k) {
  store_fe(&dst->x, k.x);
  store_fe(&dst->y, k.y);
  store_fe(&dst->k, k.k);
}

struct PrepArgs {
  const Affine* pk;
  const Affine* r;
  const Fe* s;
  const Affine* ios;        // I, O per pair
  const uint32_t* io_off;   // n+1
  const uint32_t* ad_off;   // n+1
  const uint8_t* ad;
  BaseRec* pts;             // MSM bases, order R, pk, (O_i, I_i)...  (thin.rs:291-312)
  uint32_t* cs;             // 16 words per proof
  uint32_t* z;              // 4 words per pair
  uint32_t* renc;           // 8 words per proof (tap)
  int* flags;               // [0] |= 1 when an identity pk / I / O is seen (thin.rs:266-271)
  uint32_t n;
  uint32_t first;           // this launch handles proofs first .. (chunked so the D2H + host hash can start early)
  int canonical;
};

// BatchVerifier::prepare for one proof per thread (thin.rs:209-226) fused with the base
// preparation (Montgomery image, k = d*x*y) and the identity gate (thin.rs:266-271).
template <int S>
__global__ void __launch_bounds__(128) k_prepare(PrepArgs a) {
  constexpr int FR = SuiteT<S>::FR;
  uint32_t j = a.first + blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.n) return;
  uint32_t io0 = a.io_off[j], io1 = a.io_off[j + 1], m = io1 - io0;
  size_t pbase = 2 * (size_t)j + 2 * (size_t)io0;
  bool bad = false;
  int oob = 0;                          // a coordinate or scalar >= its modulus: not a field element
  Sha512 t;
  uint32_t enc[8];
  Affine P;
  AffineK K;
  load_affine_fmt<S>(P, a.pk + j, a.canonical, &oob);
  bad |= affine_is_identity<S>(P);
  affine_compress<S>(enc, P);
  thin_transcript_begin<S>(t, m, enc);
  affine_to_k<S>(K, P);
  store_affinek(a.pts + pbase + 1, K);
  for (uint32_t i = 0; i < m; i++) {
    load_affine_fmt<S>(P, a.ios + 2 * (size_t)(io0 + i), a.canonical, &oob);       // input
    bad |= affine_is_identity<S>(P);
    affine_compress<S>(enc, P);
    sha512_put_words(t, enc);
    affine_to_k<S>(K, P);
    store_affinek(a.pts + pbase + 3 + 2 * i, K);
    load_affine_fmt<S>(P, a.ios + 2 * (size_t)(io0 + i) + 1, a.canonical, &oob);   // output
    bad |= affine_is_identity<S>(P);
    affine_compress<S>(enc, P);
    sha512_put_words(t, enc);
    affine_to_k<S>(K, P);
    store_affinek(a.pts + pbase + 2 + 2 * i, K);
  }
  uint32_t ad0 = a.ad_off[j], ad1 = a.ad_off[j + 1];
  thin_transcript_ad(t, a.ad + ad0, ad1 - ad0);
  uint32_t* zout = a.z + 4 * (size_t)io0;
  thin_delinearize(t, m, [&](uint32_t i, const uint32_t* z4) {
    zout[4 * i + 0] = z4[0]; zout[4 * i + 1] = z4[1]; zout[4 * i + 2] = z4[2]; zout[4 * i + 3] = z4[3];
  });
  load_affine_fmt<S>(P, a.r + j, a.canonical, &oob);
  affine_compress<S>(enc, P);
  affine_to_k<S>(K, P);
  store_affinek(a.pts + pbase, K);
  uint32_t c4[4];
  thin_challenge(t, enc, c4);
  Fe s;
  load_fe(s, a.s + j);
  oob |= !fe_in_range<FR>(s);
  if (!a.canonical) from_mont<FR>(s, s);
  uint4* cs = reinterpret_cast<uint4*>(a.cs + 16 * (size_t)j);
  cs[0] = make_uint4(c4[0], c4[1], c4[2], c4[3]);
  cs[1] = make_uint4(0, 0, 0, 0);
  cs[2] = make_uint4(s.v[0], s.v[1], s.v[2], s.v[3]);
  cs[3] = make_uint4(s.v[4], s.v[5], s.v[6], s.v[7]);
  uint4* re = reinterpret_cast<uint4*>(a.renc + 8 * (size_t)j);
  re[0] = make_uint4(enc[0], enc[1], enc[2], enc[3]);
  re[1] = make_uint4(enc[4], enc[5], enc[6], enc[7]);
  if (bad | (oob != 0)) atomicOr(a.flags, (bad ? 1 : 0) | (oob ? 2 : 0));
}

// AVRF_WEIGHTS_TREE: leaf digests of the (c,s) stream, one thread per TREE_LEAF proofs:
//   leaf_i = SHA512(0x00 || LE64(i) || stream[i*64*TREE_LEAF ...])   (i = global leaf index)
constexpr uint32_t TREE_LEAF = 32;
__global__ void __launch_bounds__(64) k_tree_leaves(const uint32_t* cs, uint32_t n, uint64_t first_leaf, uint64_t* out) {
  uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t nl = (n + TREE_LEAF - 1) / TREE_LEAF;
  if (l >= nl) return;
  Sha512 c;
  sha512_init(c);
  sha512_put_byte(c, 0);
  sha512_put_le64(c, first_leaf + l);
  uint32_t j0 = l * TREE_LEAF, j1 = min(n, j0 + TREE_LEAF);
  for (uint32_t j = j0; j < j1; j++) {
    const uint32_t* w = cs + 16 * (size_t)j;
    sha512_put_words(c, w);
    sha512_put_words(c, w + 8);
  }
  uint64_t d[8];
  sha512_final(c, d);
  for (int i = 0; i < 8; i++) out[8 * (size_t)l + i] = bswap64(d[i]);     // digest bytes in memory order
}

// pedersen::BatchItem::new for one proof per thread (reference src/pedersen.rs:283-301): the transcript and merged pair
// of pedersen.cuh (the merged pair normalised here), then || enc(Yb), c = challenge([R, Ok]).  Bases in the order of
// pedersen.rs:389-405.
struct PedPrepArgs {
  const Affine* pkcom;
  const Affine* r;
  const Affine* ok;
  const Fe* s;
  const Fe* sb;
  const Affine* ios;
  const uint32_t* io_off;
  const uint32_t* ad_off;
  const uint8_t* ad;
  BaseRec* pts;             // 5 per proof: O_m, Ok, I_m, Yb, R
  uint32_t* cs;             // 24 words per proof: c, 0, s, sb
  int* flags;
  uint32_t n;
  uint32_t first;
  int canonical;
};

template <int S>
__global__ void __launch_bounds__(128) k_prepare_ped(PedPrepArgs a) {
  constexpr int FQ = SuiteT<S>::FQ;
  constexpr int FR = SuiteT<S>::FR;
  uint32_t j = a.first + blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.n) return;
  uint32_t io0 = a.io_off[j], m = a.io_off[j + 1] - io0;
  bool bad = false;
  int oob = 0;                          // a coordinate or scalar >= its modulus: not a field element
  Sha512 t;
  uint32_t enc[8], enc2[8];
  Affine P, Im, Om;
  AffineK K;
  const Affine* base = a.ios + 2 * (size_t)io0;
  const int canonical = a.canonical;
  uint32_t ad0 = a.ad_off[j];
  ped_transcript<S>(t, m, [&](uint32_t k) {
    Affine Q;
    load_affine_fmt<S>(Q, base + k, canonical, &oob);
    bad |= affine_is_identity<S>(Q);
    return Q;
  }, a.ad + ad0, a.ad_off[j + 1] - ad0);
  auto get_io = [base, canonical](uint32_t k) {
    Affine Q;
    load_affine_fmt<S>(Q, base + k, canonical);
    return Q;
  };
  if (m == 0) {
    fe_zero(Im.x); fe_one<FQ>(Im.y);
    Om = Im;
  } else if (m == 1) {
    Im = get_io(0);
    Om = get_io(1);
  } else {
    Ext im, om;
    ped_merge<S, true>(im, om, t, m, get_io);
    Fe zz, inv, zi, zo;                                 // normalize_batch: one inversion for both
    mont_mul_c<FQ>(zz, im.z, om.z);
    fe_inv<FQ>(inv, zz);
    mont_mul_c<FQ>(zi, inv, om.z);
    mont_mul_c<FQ>(zo, inv, im.z);
    mont_mul_c<FQ>(Im.x, im.x, zi);
    mont_mul_c<FQ>(Im.y, im.y, zi);
    mont_mul_c<FQ>(Om.x, om.x, zo);
    mont_mul_c<FQ>(Om.y, om.y, zo);
  }
  BaseRec* out = a.pts + 5 * (size_t)j;
  affine_to_k<S>(K, Om);
  store_affinek(out + 0, K);
  affine_to_k<S>(K, Im);
  store_affinek(out + 2, K);
  load_affine_fmt<S>(P, a.pkcom + j, a.canonical, &oob);     // Yb
  bad |= affine_is_identity<S>(P);
  affine_compress<S>(enc, P);
  sha512_put_words(t, enc);
  affine_to_k<S>(K, P);
  store_affinek(out + 3, K);
  load_affine_fmt<S>(P, a.r + j, a.canonical, &oob);         // R
  affine_compress<S>(enc, P);
  affine_to_k<S>(K, P);
  store_affinek(out + 4, K);
  load_affine_fmt<S>(P, a.ok + j, a.canonical, &oob);        // Ok
  affine_compress<S>(enc2, P);
  affine_to_k<S>(K, P);
  store_affinek(out + 1, K);
  uint32_t c4[4];
  ped_challenge(t, enc, enc2, c4);
  Fe s, sb;
  load_fe(s, a.s + j);
  load_fe(sb, a.sb + j);
  oob |= !(fe_in_range<FR>(s) && fe_in_range<FR>(sb));
  if (!a.canonical) { from_mont<FR>(s, s); from_mont<FR>(sb, sb); }
  uint4* cs = reinterpret_cast<uint4*>(a.cs + 24 * (size_t)j);
  cs[0] = make_uint4(c4[0], c4[1], c4[2], c4[3]);
  cs[1] = make_uint4(0, 0, 0, 0);
  cs[2] = make_uint4(s.v[0], s.v[1], s.v[2], s.v[3]);
  cs[3] = make_uint4(s.v[4], s.v[5], s.v[6], s.v[7]);
  cs[4] = make_uint4(sb.v[0], sb.v[1], sb.v[2], sb.v[3]);
  cs[5] = make_uint4(sb.v[4], sb.v[5], sb.v[6], sb.v[7]);
  if (bad | (oob != 0)) atomicOr(a.flags, (bad ? 1 : 0) | (oob ? 2 : 0));
}

}  // namespace avrf
