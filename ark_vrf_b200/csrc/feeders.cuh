// Kernels either side of the batch-verification path (SURVEY.md 8a rows a10, a11, a15 and 8f):
// hash-to-curve, VRF outputs / public keys, bulk proving, point compression and output hashing,
// wire-format ingest, per-proof verdicts.  One thread per item.
#pragma once
#include "prepare.cuh"

namespace avrf {
__global__ void k_rebase(uint32_t* off, uint64_t count, uint32_t base) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) off[i] += base;
}

template <int S>
__global__ void __launch_bounds__(128) k_h2c(const uint8_t* msgs, const uint32_t* off, uint32_t n, Affine* out_aff,
                                             uint32_t* out_enc, uint8_t* ok, int canonical) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  Affine P;
  bool good = data_to_point<S>(P, msgs + off[j], off[j + 1] - off[j]);
  if (!good) {
    fe_zero(P.x);
    fe_one<SuiteT<S>::FQ>(P.y);
  }
  if (ok) ok[j] = good ? 1 : 0;
  if (out_enc) {
    uint32_t enc[8];
    affine_compress<S>(enc, P);
    for (int i = 0; i < 8; i++) out_enc[8 * (size_t)j + i] = enc[i];
  }
  if (out_aff) store_affine_fmt<S>(out_aff + j, P, canonical);
}

// device-internal Montgomery points -> the caller's format
template <int S>
__global__ void __launch_bounds__(128) k_refmt(const Affine* in, uint64_t n, Affine* out, int canonical) {
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  Affine P;
  load_fe(P.x, &in[j].x);
  load_fe(P.y, &in[j].y);
  store_affine_fmt<S>(out + j, P, canonical);
}

struct ProveArgs {
  const Fe* sk;
  const Affine* pk;
  const Affine* ios;
  const uint32_t* io_off;
  const uint32_t* ad_off;
  const uint8_t* ad;
  Affine* r;
  Fe* s;
  uint32_t n;
  int canonical;
};

template <int S>
__global__ void __launch_bounds__(128) k_prove(ProveArgs a) {
  constexpr int FR = SuiteT<S>::FR;
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.n) return;
  uint32_t io0 = a.io_off[j], m = a.io_off[j + 1] - io0;
  Affine pk, R;
  load_affine_fmt<S>(pk, a.pk + j, a.canonical);
  Fe sk, s;
  load_fe(sk, a.sk + j);
  if (!a.canonical) from_mont<FR>(sk, sk);
  uint32_t ad0 = a.ad_off[j];
  const Affine* base = a.ios + 2 * (size_t)io0;
  int canonical = a.canonical;
  // any number of I/O pairs: the points are read from device memory where they are needed (transcript, merge)
  thin_prove_one_g<S>(R, s, sk, pk, [base, canonical](uint32_t k) {
    Affine P;
    load_affine_fmt<S>(P, base + k, canonical);
    return P;
  }, m, a.ad + ad0, a.ad_off[j + 1] - ad0);
  store_affine_fmt<S>(a.r + j, R, a.canonical);
  if (!a.canonical) to_mont<FR>(s, s);
  store_fe(a.s + j, s);
}

// pedersen::Prover::prove (src/pedersen.rs:136-186), one proof per thread: ped_prove_one_g (pedersen.cuh).
struct PedProveArgs {
  const Fe* sk;
  const Affine* pk;
  const Affine* ios;
  const uint32_t* io_off;
  const uint32_t* ad_off;
  const uint8_t* ad;
  Affine* pkcom;
  Affine* r;
  Affine* ok;
  Fe* s;
  Fe* sb;
  Fe* blinding;             // may be null
  uint32_t n;
  int canonical;
};

template <int S>
__global__ void __launch_bounds__(128) k_prove_ped(PedProveArgs a) {
  constexpr int FR = SuiteT<S>::FR;
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.n) return;
  uint32_t io0 = a.io_off[j], m = a.io_off[j + 1] - io0;
  Affine pk, PKC, R, OK;
  load_affine_fmt<S>(pk, a.pk + j, a.canonical);
  Fe sk, s, sb, bl;
  load_fe(sk, a.sk + j);
  if (!a.canonical) from_mont<FR>(sk, sk);
  uint32_t ad0 = a.ad_off[j];
  const Affine* base = a.ios + 2 * (size_t)io0;
  int canonical = a.canonical;
  ped_prove_one_g<S>(PKC, R, OK, s, sb, bl, sk, pk, [base, canonical](uint32_t k) {
    Affine P;
    load_affine_fmt<S>(P, base + k, canonical);
    return P;
  }, m, a.ad + ad0, a.ad_off[j + 1] - ad0);
  store_affine_fmt<S>(a.pkcom + j, PKC, a.canonical);
  store_affine_fmt<S>(a.r + j, R, a.canonical);
  store_affine_fmt<S>(a.ok + j, OK, a.canonical);
  if (!a.canonical) { to_mont<FR>(s, s); to_mont<FR>(sb, sb); to_mont<FR>(bl, bl); }
  store_fe(a.s + j, s);
  store_fe(a.sb + j, sb);
  if (a.blinding) store_fe(a.blinding + j, bl);
}

template <int S>
__global__ void __launch_bounds__(128) k_compress(const Affine* in, uint64_t n, uint32_t* out, int canonical, int hash) {
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  Affine P;
  load_affine_fmt<S>(P, in + j, canonical);
  uint32_t enc[8], h[8];
  affine_compress<S>(enc, P);
  if (hash) {
    point_to_hash32<S>(h, enc);
    for (int i = 0; i < 8; i++) out[8 * j + i] = h[i];
  } else {
    for (int i = 0; i < 8; i++) out[8 * j + i] = enc[i];
  }
}

// ---------------------------------------------------------------------------------------
// Pipelined feeder kernels: no thread ever runs a field inversion of its own.
// A Fermat inversion is ~335 multiplications; hash-to-curve needs two per point (Elligator2 denominators,
// projective -> affine), a VRF output one, point decompression one.  The kernels below leave their
// denominators in an array, k_batch_inv inverts the whole array with Montgomery's trick (3 multiplications
// per element plus one inversion per 32 elements), and a finishing kernel multiplies through.
// ---------------------------------------------------------------------------------------

// In-place inversion of v[0..n): thread t owns v[t], v[t+T], ... (coalesced).  Zero stays zero.
template <int F>
__global__ void __launch_bounds__(128) k_batch_inv(Fe* v, Fe* scratch, uint64_t n) {
  const uint64_t T = (uint64_t)gridDim.x * blockDim.x, t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  Fe acc;
  fe_one<F>(acc);
  uint64_t last = t;
#pragma unroll 1
  for (uint64_t i = t; i < n; i += T) {
    Fe x;
    load_fe(x, v + i);
    store_fe(scratch + i, acc);                       // product of this thread's earlier non-zero elements
    if (!fe_is_zero(x)) acc = mont_mul_v<F>(acc, x);
    last = i;
  }
  fe_inv<F>(acc, acc);
#pragma unroll 1
  for (uint64_t i = last;; i -= T) {
    Fe x, pre;
    load_fe(x, v + i);
    if (!fe_is_zero(x)) {
      load_fe(pre, scratch + i);
      Fe inv = mont_mul_v<F>(acc, pre);
      acc = mont_mul_v<F>(acc, x);
      store_fe(v + i, inv);
    }
    if (i < T + t) break;
  }
}

// Elligator2 hash-to-curve, stage 1: message -> (u0, u1) and the product of the two map denominators.
template <int S>
__global__ void __launch_bounds__(128) k_h2f(const uint8_t* msgs, const uint32_t* off, uint32_t n, Fe* u01, Fe* den) {
  constexpr int FQ = SuiteT<S>::FQ;
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  Fe u0, u1, one, Z, d0, d1, t;
  ell2_hash_to_field<S>(u0, u1, msgs + off[j], off[j + 1] - off[j]);
  fe_one<FQ>(one);
  fe_set(Z, AVRF_CC(S).zz);
  mont_sqr_c<FQ>(t, u0);
  mont_mul_c<FQ>(t, t, Z);
  fe_add<FQ>(d0, one, t);                // 1 + Z u0^2
  mont_sqr_c<FQ>(t, u1);
  mont_mul_c<FQ>(t, t, Z);
  fe_add<FQ>(d1, one, t);
  if (fe_is_zero(d0)) d0 = one;          // upstream takes den = 1 there (SURVEY.md A.6)
  if (fe_is_zero(d1)) d1 = one;
  mont_mul_c<FQ>(t, d0, d1);
  store_fe(u01 + 2 * (size_t)j, u0);
  store_fe(u01 + 2 * (size_t)j + 1, u1);
  store_fe(den + j, t);
}

// Stage 2: both maps, their sum, cofactor clearing; leaves (X, Y) in xy and Z in zden (to be inverted).
template <int S>
__global__ void __launch_bounds__(128, 4) k_ell2_maps(const Fe* u01, Fe* zden, uint32_t n, Affine* xy) {
  constexpr int FQ = SuiteT<S>::FQ;
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  Fe u0, u1, inv, one, Z, d0, d1, t, i0, i1;
  load_fe(u0, u01 + 2 * (size_t)j);
  load_fe(u1, u01 + 2 * (size_t)j + 1);
  load_fe(inv, zden + j);                // 1 / (d0 d1)
  fe_one<FQ>(one);
  fe_set(Z, AVRF_CC(S).zz);
  mont_sqr_c<FQ>(t, u0);
  mont_mul_c<FQ>(t, t, Z);
  fe_add<FQ>(d0, one, t);
  mont_sqr_c<FQ>(t, u1);
  mont_mul_c<FQ>(t, t, Z);
  fe_add<FQ>(d1, one, t);
  bool z0 = fe_is_zero(d0), z1 = fe_is_zero(d1);
  if (z0) d0 = one;
  if (z1) d1 = one;
  mont_mul_c<FQ>(i0, inv, d1);
  mont_mul_c<FQ>(i1, inv, d0);
  Ext e0 = ell2_map_ext_v<S>(u0, i0, z0);
  Ext e1 = ell2_map_ext_v<S>(u1, i1, z1);
  ext_add_c<S>(e0, e0, e1);
  for (uint32_t i = 0; i < AVRF_CC(S).cof_log2; i++) ext_dbl_c<S>(e0, e0);
  store_fe(&xy[j].x, e0.x);
  store_fe(&xy[j].y, e0.y);
  store_fe(zden + j, e0.z);
}

// Last stage of every pipeline: (X, Y) * (1/Z) -> affine, optional compressed encoding / format conversion.
// zinv == 0 marks "no point" (ok = 0, identity written).
template <int S>
__global__ void __launch_bounds__(128) k_affine_finish(const Affine* xy, const Fe* zinv, uint64_t n, Affine* out_dev,
                                                       Affine* out_fmt, uint32_t* out_enc, uint8_t* ok, int canonical) {
  constexpr int FQ = SuiteT<S>::FQ;
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  Fe X, Y, zi;
  load_fe(X, &xy[j].x);
  load_fe(Y, &xy[j].y);
  load_fe(zi, zinv + j);
  Affine P;
  bool good = !fe_is_zero(zi);
  if (good) {
    mont_mul_c<FQ>(P.x, X, zi);
    mont_mul_c<FQ>(P.y, Y, zi);
  } else {
    fe_zero(P.x);
    fe_one<FQ>(P.y);
  }
  if (ok) ok[j] = good ? 1 : 0;
  if (out_dev) { store_fe(&out_dev[j].x, P.x); store_fe(&out_dev[j].y, P.y); }
  if (out_enc) {
    uint32_t enc[8];
    affine_compress<S>(enc, P);
    for (int i = 0; i < 8; i++) out_enc[8 * j + i] = enc[i];
  }
  if (out_fmt) store_affine_fmt<S>(out_fmt + j, P, canonical);
}

// out_j = sk_j * in_j, projective: (X, Y) to xy, Z to zden.  in == nullptr: the generator.  in_is_dev: the inputs are
// device-internal Montgomery points (the output of k_affine_finish), not caller data in `canonical` format.
// in_subgroup: the caller vouches that every input lies in the prime-order subgroup.
template <int S>
__global__ void __launch_bounds__(128, 4) k_scalar_mul_proj(const Fe* sk, uint32_t sk_stride_words, const Affine* in, uint32_t n,
                                                         Affine* xy, Fe* zden, int canonical, int in_is_dev, int in_subgroup) {
  constexpr int FR = SuiteT<S>::FR;
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  Fe k;
  load_fe(k, reinterpret_cast<const Fe*>(reinterpret_cast<const uint32_t*>(sk) + (size_t)j * sk_stride_words));
  if (!canonical) from_mont<FR>(k, k);
  Affine P;
  if (in) load_affine_fmt<S>(P, in + j, in_is_dev ? 0 : canonical);
  else { fe_set(P.x, AVRF_CC(S).gx); fe_set(P.y, AVRF_CC(S).gy); }
  Ext e, r;
  if (S == SUITE_BAND && in_subgroup) {
    // the point is known to lie in the prime-order subgroup (the library's own hash-to-curve output, or the
    // generator): GLV halves the doublings (curve.cuh)
    r = ext_scalar_mul_glv_v<S>(P, k);
  } else {
    affine_to_ext<S>(e, P);
    ext_scalar_mul<S>(r, e, k.v, 256);
  }
  store_fe(&xy[j].x, r.x);
  store_fe(&xy[j].y, r.y);
  store_fe(zden + j, r.z);
}

// The same for ONE secret shared by all inputs (the plan - GLV split, width-5 NAF - is computed once on the host):
// uniform sparse addition chain, Bandersnatch subgroup points only (curve.cuh, ext_scalar_mul_glv_plan_v).
template <int S>
__global__ void __launch_bounds__(128, 4) k_scalar_mul_plan(NafPlan pl, const Affine* in, uint32_t n, Affine* xy, Fe* zden,
                                                         int canonical, int in_is_dev) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  Affine P;
  if (in) load_affine_fmt<S>(P, in + j, in_is_dev ? 0 : canonical);
  else { fe_set(P.x, AVRF_CC(S).gx); fe_set(P.y, AVRF_CC(S).gy); }
  Ext r = ext_scalar_mul_glv_plan_v<S>(P, pl);
  store_fe(&xy[j].x, r.x);
  store_fe(&xy[j].y, r.y);
  store_fe(zden + j, r.z);
}

// CanonicalDeserialize with Validate::Yes of compressed points (ark-serialize 0.6; reference src/lib.rs:410-433 Public,
// :471-494 Input, :552-575 Output, src/thin.rs:42 Proof.r): y < p, x = sqrt((1-y^2)/(a-d y^2)) picked by the sign flag,
// prime-subgroup check, and for kind = 1 (Public / Input / Output) the identity is rejected as well.
// Stage 1: y -> numerator and denominator of x^2 = (1 - y^2) / (a - d y^2).
// flags[j]: bit 0 = sign flag of the encoding, bit 1 = y is canonical (< p) and the denominator is non-zero.
template <int S>
__global__ void __launch_bounds__(128) k_dec_prep(const uint32_t* in, uint64_t n, Fe* ynum, Fe* den, uint8_t* flags) {
  constexpr int FQ = SuiteT<S>::FQ;
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  Fe y, one, d, y2, num, dn, a1;
#pragma unroll
  for (int i = 0; i < 8; i++) y.v[i] = in[8 * j + i];
  uint8_t fl = (y.v[7] >> 31) & 1;
  y.v[7] &= 0x7fffffffu;
  bool good = limbs_gt(AVRF_FC(FQ).p, y.v);          // y < p
  fe_zero(dn);
  fe_zero(num);
  if (good) {
    to_mont<FQ>(y, y);
    fe_one<FQ>(one);
    fe_set(d, AVRF_CC(S).d);
    mont_sqr_c<FQ>(y2, y);
    fe_sub<FQ>(num, one, y2);              // 1 - y^2
    mont_mul_c<FQ>(dn, d, y2);
    a_times<S>(a1, one);
    fe_sub<FQ>(dn, a1, dn);                // a - d y^2
    good = !fe_is_zero(dn);
  } else {
    fe_zero(y);
  }
  store_fe(ynum + 2 * j, y);
  store_fe(ynum + 2 * j + 1, num);
  store_fe(den + j, dn);                   // zero when invalid: k_batch_inv leaves it alone
  flags[j] = fl | (good ? 2 : 0);
}

// Stage 2: x = sqrt(num / den) picked by the sign flag, identity rule, prime-subgroup check.
template <int S>
__global__ void __launch_bounds__(128) k_dec_finish(const Fe* ynum, const Fe* dinv, const uint8_t* flags, uint64_t n, int kind,
                                                    Affine* out, uint8_t* ok, int canonical) {
  constexpr int FQ = SuiteT<S>::FQ;
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  uint8_t fl = flags[j];
  Affine P;
  fe_zero(P.x);
  fe_one<FQ>(P.y);
  bool good = (fl & 2) != 0;
  if (good) {
    Fe y, num, inv, x2, x, xc;
    load_fe(y, ynum + 2 * j);
    load_fe(num, ynum + 2 * j + 1);
    load_fe(inv, dinv + j);
    mont_mul_c<FQ>(x2, num, inv);
    good = fe_sqrt<S>(x, x2);
    if (good) {
      from_mont<FQ>(xc, x);
      bool is_big = limbs_gt(xc.v, AVRF_FC(FQ).phalf);
      if (is_big != ((fl & 1) != 0)) fe_neg<FQ>(x, x);
      P.x = x;
      P.y = y;
    }
  }
  if (good && kind == 1 && affine_is_identity<S>(P)) good = false;
  if (good) good = in_prime_subgroup_v<S>(P);
  if (!good) { fe_zero(P.x); fe_one<FQ>(P.y); }
  ok[j] = good ? 1 : 0;
  store_affine_fmt<S>(out + j, P, canonical);
}

// Wire-format scalars (canonical little-endian, < r checked by the caller's verify) into the handle's format.
template <int S>
__global__ void __launch_bounds__(128) k_scalars_to_mont(Fe* s, uint64_t n) {
  constexpr int FR = SuiteT<S>::FR;
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  Fe x;
  load_fe(x, s + j);
  if (fe_in_range<FR>(x)) to_mont<FR>(x, x);       // out-of-range values stay as they are: k_prepare flags them
  store_fe(s + j, x);
}

// Per-proof decode verdict of a wire-format push: proof j is good when R_j, pk_j and all its I/O points decoded.
__global__ void __launch_bounds__(256) k_proof_ok(const uint8_t* ok_r, const uint8_t* ok_pk, const uint8_t* ok_ios,
                                                  const uint32_t* io_off, uint32_t io_base, uint64_t n, uint8_t* ok,
                                                  unsigned long long* n_bad) {
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  uint8_t g = ok_r[j] & ok_pk[j];
  for (uint32_t i = 2 * (io_off[j] - io_base); i < 2 * (io_off[j + 1] - io_base); i++) g &= ok_ios[i];
  ok[j] = g;
  if (!g) atomicAdd(n_bad, 1ull);
}

// Wire-format Pedersen proofs (pedersen::Proof::serialize_compressed, src/pedersen.rs:43-50): n records of 160 bytes,
// pk_com | r | ok | s | sb.  The three point encodings go to enc as pk_com (n) | R (n) | Ok (n), ahead of the I/O
// encodings the caller copies behind them, and the two scalars to sc as s (n) | sb (n).  One thread per 16-byte word:
// the loads are coalesced across the records.
__global__ void __launch_bounds__(256) k_ped_wire_unpack(const uint4* rec, uint64_t n, uint4* enc, uint4* sc) {
  uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= 10 * n) return;
  uint64_t j = t / 10;
  uint32_t w = (uint32_t)(t - 10 * j), field = w >> 1, half = w & 1;
  uint4 v = rec[t];
  if (field < 3) enc[2 * (field * n + j) + half] = v;
  else sc[2 * ((field - 3) * n + j) + half] = v;
}

// Per-proof decode verdict of a wire-format Pedersen push: proof j is good when pk_com, R and Ok decoded
// (ok_pts: pk_com (n) | R (n) | Ok (n)), every point of its I/O pairs decoded, and s, sb are canonical scalars (< r),
// which `Fr::deserialize_compressed` demands.
template <int S>
__global__ void __launch_bounds__(256) k_ped_proof_ok(const uint8_t* ok_pts, const uint8_t* ok_ios, const uint32_t* io_off,
                                                      uint32_t io_base, const Fe* sc, uint64_t n, uint8_t* ok,
                                                      unsigned long long* n_bad) {
  constexpr int FR = SuiteT<S>::FR;
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  uint8_t g = ok_pts[j] & ok_pts[n + j] & ok_pts[2 * n + j];
  for (uint32_t i = 2 * (io_off[j] - io_base); i < 2 * (io_off[j + 1] - io_base); i++) g &= ok_ios[i];
  Fe s, sb;
  load_fe(s, sc + j);
  load_fe(sb, sc + n + j);
  if (!(fe_in_range<FR>(s) && fe_in_range<FR>(sb))) g = 0;
  ok[j] = g;
  if (!g) atomicAdd(n_bad, 1ull);
}

// thin::Verifier::verify for every proof of a prepared batch (src/thin.rs:131-165), one thread per
// proof, reusing c_j and z_ij of k_prepare: status 0 Ok / 1 VerificationFailure / 2 InvalidData.
struct EachArgs {
  const Affine* pk;         // the pushed inputs (not the MSM bases, whose layout is suite specific)
  const Affine* r;
  const Affine* ios;
  int canonical;
  const uint32_t* cs;
  const uint32_t* z;
  const uint32_t* io_off;
  int32_t* status;
  uint32_t n;
};

template <int S>
__global__ void __launch_bounds__(128) k_verify_each(EachArgs a) {
  constexpr int FQ = SuiteT<S>::FQ;
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.n) return;
  uint32_t io0 = a.io_off[j], m = a.io_off[j + 1] - io0;
  Affine R, pk, t;
  load_affine_fmt<S>(R, a.r + j, a.canonical);
  load_affine_fmt<S>(pk, a.pk + j, a.canonical);
  bool bad = affine_is_identity<S>(pk);
  Ext im, om, e, q;
  {
    Affine g;
    fe_set(g.x, AVRF_CC(S).gx);
    fe_set(g.y, AVRF_CC(S).gy);
    affine_to_ext<S>(im, g);              // I_m = G + sum z_i I_i
  }
  affine_to_ext<S>(om, pk);               // O_m = pk + sum z_i O_i
  for (uint32_t i = 0; i < m; i++) {
    uint32_t z8[8] = {a.z[4 * (size_t)(io0 + i)], a.z[4 * (size_t)(io0 + i) + 1], a.z[4 * (size_t)(io0 + i) + 2],
                      a.z[4 * (size_t)(io0 + i) + 3], 0, 0, 0, 0};
    load_affine_fmt<S>(t, a.ios + 2 * (size_t)(io0 + i) + 1, a.canonical);   // O_i
    bad |= affine_is_identity<S>(t);
    affine_to_ext<S>(e, t);
    ext_scalar_mul<S>(q, e, z8, 128);
    ext_add_c<S>(om, om, q);
    load_affine_fmt<S>(t, a.ios + 2 * (size_t)(io0 + i), a.canonical);       // I_i
    bad |= affine_is_identity<S>(t);
    affine_to_ext<S>(e, t);
    ext_scalar_mul<S>(q, e, z8, 128);
    ext_add_c<S>(im, im, q);
  }
  const uint32_t* csj = a.cs + 16 * (size_t)j;
  uint32_t c8[8] = {csj[0], csj[1], csj[2], csj[3], 0, 0, 0, 0};
  uint32_t s8[8];
  for (int i = 0; i < 8; i++) s8[i] = csj[8 + i];
  ext_scalar_mul<S>(q, im, s8, 256);      // s * I_m
  ext_scalar_mul<S>(e, om, c8, 128);      // c * O_m
  ext_neg<S>(e, e);
  ext_add_c<S>(q, q, e);
  affine_to_ext<S>(e, R);
  ext_neg<S>(e, e);
  ext_add_c<S>(q, q, e);                  // s I_m - c O_m - R
  (void)FQ;
  a.status[j] = bad ? AVRF_INVALID_DATA : (ext_is_identity<S>(q) ? AVRF_OK : AVRF_VERIFICATION_FAILURE);
}

// pedersen::Verifier::verify for every proof of a prepared Pedersen batch (src/pedersen.rs:188-253), one thread per
// proof, reusing what k_prepare_ped left on the handle: c, s, sb (24 words per proof) and the bases O_m, Ok, I_m,
// pk_com, R (an identity accumulator plus one mixed addition turns a base record back into the point, whatever the
// suite's record layout).  The pushed pk_com and I/O points are read again only for the identity checks.
struct PedEachArgs {
  const Affine* pkcom;
  const Affine* ios;
  const uint32_t* io_off;
  int canonical;
  const BaseRec* pts;
  const uint32_t* cs;
  int32_t* status;
  uint32_t n;
};

template <int S>
__device__ __forceinline__ void base_to_ext(Ext& e, const BaseRec* b) {
  Fe x, y, k;
  load_fe(x, &b->x);
  load_fe(y, &b->y);
  load_fe(k, &b->k);
  ext_identity<S>(e);
  ext_madd<S>(e, x, y, k);
}

template <int S>
__global__ void __launch_bounds__(128) k_verify_each_ped(PedEachArgs a) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.n) return;
  uint32_t io0 = a.io_off[j], m = a.io_off[j + 1] - io0;
  Affine t;
  load_affine_fmt<S>(t, a.pkcom + j, a.canonical);
  bool bad = affine_is_identity<S>(t);
  for (uint32_t i = 0; i < 2 * m; i++) {
    load_affine_fmt<S>(t, a.ios + 2 * (size_t)io0 + i, a.canonical);
    bad |= affine_is_identity<S>(t);
  }
  if (bad) { a.status[j] = AVRF_INVALID_DATA; return; }
  const BaseRec* b = a.pts + 5 * (size_t)j;
  const uint32_t* csj = a.cs + 24 * (size_t)j;
  uint32_t c4[4] = {csj[0], csj[1], csj[2], csj[3]};
  Fe s, sb;
  for (int i = 0; i < 8; i++) { s.v[i] = csj[8 + i]; sb.v[i] = csj[16 + i]; }
  // base records in the order O_m, Ok, I_m, pk_com, R (k_prepare_ped)
  a.status[j] = ped_equations_hold<S>([b](int k) {
    Ext e;
    base_to_ext<S>(e, b + (k == PED_IM ? 2 : k == PED_OM ? 0 : k == PED_OK ? 1 : k));
    return e;
  }, c4, s, sb) ? AVRF_OK : AVRF_VERIFICATION_FAILURE;
}

}  // namespace avrf
