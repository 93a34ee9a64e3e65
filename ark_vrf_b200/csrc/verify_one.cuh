// thin::Verifier::verify for ONE proof (reference src/thin.rs:131-165 with merge_ios, src/utils/common.rs:389-419,
// and straus::short_msm, src/utils/straus.rs:89-100) as a single-warp kernel.
//
// The reference tests the exact group equation  s*I_m - c*O_m == R  with I_m = G + sum z_i I_i and
// O_m = pk + sum z_i O_i, all scalars taken as INTEGERS (s < r, c, z_i < 2^128).  No batch weight is involved,
// so a small-order component on R (or on any input) can never cancel.  Expanding the products,
//     s*G + sum_i (s z_i)*I_i - c*pk - sum_i (c z_i)*O_i - R == O,
// gives 2 + 2M independent scalar multiplications.  The integer s*z_i (381 bits) is reduced modulo h*r
// (h = cofactor): h*r is a multiple of the exponent of the whole curve group, so the product is unchanged on
// EVERY curve point, in the prime-order subgroup or not.  Each term runs on one quad of the warp (four lanes share
// the field multiplications of a point operation, msm.cuh), eight terms at a time; the accumulators of the
// quads are then folded by shuffles.  Latency: ~256 dependent doublings - a GPU is the wrong tool for ONE
// proof, this kernel exists so that the `Verifier` API is exact and needs no 2^19-bin MSM machinery.
#pragma once
#include "prepare.cuh"

namespace avrf {

struct OneArgs {
  const uint8_t* in;      // pk 64 | r 64 | s 32 | n_ios u32 | ad_len u32 | pad 8 | ios 128*M | ad
  uint32_t* z;            // scratch: 4 words per pair
  int32_t* status;        // [0] verdict, [1] flags (2: a value is not a field element)
  int canonical;
};

__device__ __forceinline__ void quad_bcast_ext(Ext& o, const Ext& p, int src_quad) {
  int src = src_quad * 4 + (threadIdx.x & 3);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    o.x.v[i] = __shfl_sync(0xffffffffu, p.x.v[i], src);
    o.y.v[i] = __shfl_sync(0xffffffffu, p.y.v[i], src);
    o.z.v[i] = __shfl_sync(0xffffffffu, p.z.v[i], src);
    o.t.v[i] = __shfl_sync(0xffffffffu, p.t.v[i], src);
  }
}

// acc += k * p for this lane's quad; k = 256-bit integer, fixed 4-bit windows over a 16-entry table kept in
// shared memory (every lane of the quad writes the same values).  Uniform control flow across the warp.
template <int S>
__device__ __forceinline__ void quad_scalar_mul_acc(Ext& acc, const Ext& p, const uint32_t* k, Ext* tbl) {
  Ext e;
  ext_identity<S>(e);
  tbl[0] = e;
  tbl[1] = p;
#pragma unroll 1
  for (int i = 2; i < 16; i++) {
    e = tbl[i - 1];
    quad_add<S>(e, p);
    tbl[i] = e;
  }
  e = tbl[(k[7] >> 28) & 15u];
#pragma unroll 1
  for (int w = 62; w >= 0; w--) {
    quad_dbl<S>(e);
    quad_dbl<S>(e);
    quad_dbl<S>(e);
    quad_dbl<S>(e);
    Ext q = tbl[(k[w >> 3] >> (4 * (w & 7))) & 15u];
    quad_add<S>(e, q);
  }
  quad_add<S>(acc, e);
}

// x = s * z as an integer, reduced modulo h*r (see the header comment).  s canonical < r, z < 2^128.
template <int S>
__device__ __forceinline__ void mul_mod_hr(Fe& out, const Fe& s, const Fe& z) {
  constexpr int FR = SuiteT<S>::FR;
  Fe zM, x;
  to_mont<FR>(zM, z);
  mont_mul_c<FR>(x, s, zM);                               // s*z mod r, canonical
  uint32_t h = 1u << AVRF_CC(S).cof_log2;
  uint32_t want = (s.v[0] * z.v[0]) & (h - 1);            // s*z mod h
#pragma unroll 1
  for (uint32_t i = 0; i < h && (x.v[0] & (h - 1)) != want; i++) {
    x.v[0] = add_cc(x.v[0], AVRF_FC(FR).p[0]);
#pragma unroll
    for (int l = 1; l < 7; l++) x.v[l] = addc_cc(x.v[l], AVRF_FC(FR).p[l]);
    x.v[7] = addc(x.v[7], AVRF_FC(FR).p[7]);              // < h*r < 2^256
  }
  out = x;
}

// c * z as a 256-bit integer (c, z < 2^128): schoolbook on the four low limbs.
__device__ __forceinline__ void mul128(Fe& out, const Fe& c, const Fe& z) {
  uint64_t acc[8];
#pragma unroll
  for (int i = 0; i < 8; i++) acc[i] = 0;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    uint64_t carry = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      uint64_t t = (uint64_t)c.v[i] * z.v[j] + (acc[i + j] & 0xffffffffu) + carry;
      acc[i + j] = t & 0xffffffffu;
      carry = t >> 32;
    }
    acc[i + 4] = carry;
  }
#pragma unroll
  for (int i = 0; i < 8; i++) out.v[i] = (uint32_t)acc[i];
}

template <int S>
__global__ void __launch_bounds__(32) k_verify_one(OneArgs a) {
  constexpr int FR = SuiteT<S>::FR;
  __shared__ Ext tbl[8][16];
  const int quad = threadIdx.x >> 2;
  const Affine* pkp = reinterpret_cast<const Affine*>(a.in);
  const Affine* rp = reinterpret_cast<const Affine*>(a.in + 64);
  const Fe* sp = reinterpret_cast<const Fe*>(a.in + 128);
  const uint32_t m = *reinterpret_cast<const uint32_t*>(a.in + 160);
  const uint32_t ad_len = *reinterpret_cast<const uint32_t*>(a.in + 164);
  const Affine* ios = reinterpret_cast<const Affine*>(a.in + 176);
  const uint8_t* ad = a.in + 176 + 128 * (size_t)m;
  // ---- transcript (every lane computes the same values: no divergence, no exchange) ----------------
  bool bad = false;
  int oob = 0;
  Sha512 t;
  uint32_t enc[8];
  Affine P;
  load_affine_fmt<S>(P, pkp, a.canonical, &oob);
  bad |= affine_is_identity<S>(P);
  affine_compress<S>(enc, P);
  thin_transcript_begin<S>(t, m, enc);
  for (uint32_t i = 0; i < 2 * m; i++) {
    load_affine_fmt<S>(P, ios + i, a.canonical, &oob);
    bad |= affine_is_identity<S>(P);
    affine_compress<S>(enc, P);
    sha512_put_words(t, enc);
  }
  thin_transcript_ad(t, ad, ad_len);
  uint32_t* zs = a.z;
  thin_delinearize(t, m, [&](uint32_t i, const uint32_t* z4) {
    zs[4 * i + 0] = z4[0]; zs[4 * i + 1] = z4[1]; zs[4 * i + 2] = z4[2]; zs[4 * i + 3] = z4[3];
  });
  Affine R;
  load_affine_fmt<S>(R, rp, a.canonical, &oob);
  affine_compress<S>(enc, R);
  uint32_t c4[4];
  thin_challenge(t, enc, c4);
  Fe s, c;
  load_fe(s, sp);
  oob |= !fe_in_range<FR>(s);
  if (!a.canonical) from_mont<FR>(s, s);
  fe_zero(c);
#pragma unroll
  for (int i = 0; i < 4; i++) c.v[i] = c4[i];
  __syncwarp();
  // ---- 2 + 2M terms, eight at a time, one per quad -------------------------------------------------
  // term 0: (s, G)   term 1: (c, -pk)   term 2+2i: (s z_i mod h r, I_i)   term 3+2i: (c z_i, -O_i)
  Ext acc;
  ext_identity<S>(acc);
  const uint32_t nterms = 2 + 2 * m;
  for (uint32_t base = 0; base < nterms; base += 8) {
    uint32_t tm = base + quad;
    Fe k;
    Ext p;
    fe_zero(k);
    ext_identity<S>(p);
    if (tm == 0) {
      Affine g;
      fe_set(g.x, AVRF_CC(S).gx);
      fe_set(g.y, AVRF_CC(S).gy);
      affine_to_ext<S>(p, g);
      k = s;
    } else if (tm == 1) {
      load_affine_fmt<S>(P, pkp, a.canonical);
      affine_to_ext<S>(p, P);
      ext_neg<S>(p, p);
      k = c;
    } else if (tm < nterms) {
      uint32_t i = (tm - 2) >> 1;
      Fe z;
      fe_zero(z);
#pragma unroll
      for (int q = 0; q < 4; q++) z.v[q] = zs[4 * i + q];
      if ((tm & 1) == 0) {
        load_affine_fmt<S>(P, ios + 2 * i, a.canonical);          // I_i
        affine_to_ext<S>(p, P);
        mul_mod_hr<S>(k, s, z);
      } else {
        load_affine_fmt<S>(P, ios + 2 * i + 1, a.canonical);      // O_i
        affine_to_ext<S>(p, P);
        ext_neg<S>(p, p);
        mul128(k, c, z);
      }
    }
    __syncwarp();
    quad_scalar_mul_acc<S>(acc, p, k.v, tbl[quad]);
  }
  // ---- fold the eight quads, subtract R, test ------------------------------------------------------
#pragma unroll 1
  for (int d = 4; d > 0; d >>= 1) {
    Ext o;
    quad_bcast_ext(o, acc, (quad + d) & 7);
    quad_add<S>(acc, o);
  }
  Ext rr;
  affine_to_ext<S>(rr, R);
  ext_neg<S>(rr, rr);
  quad_add<S>(acc, rr);
  if (threadIdx.x == 0) {
    a.status[0] = bad ? AVRF_INVALID_DATA : (ext_is_identity<S>(acc) ? AVRF_OK : AVRF_VERIFICATION_FAILURE);
    a.status[1] = oob ? 2 : 0;
  }
}

// pedersen::Verifier::verify (src/pedersen.rs:188-253) for ONE proof: ped_verify_one_g (pedersen.cuh) on one thread.
// Input: pk_com 64 | r 64 | ok 64 | s 32 | sb 32 | n_ios u32 | ad_len u32 | pad 8 | ios 128*M | ad.
struct PedOneArgs {
  const uint8_t* in;
  int32_t* status;          // [0] verdict, [1] flags (2: a value is not a field element)
  int canonical;
};

template <int S>
__global__ void __launch_bounds__(32) k_verify_one_ped(PedOneArgs a) {
  constexpr int FR = SuiteT<S>::FR;
  if (threadIdx.x != 0) return;
  const Affine* pts = reinterpret_cast<const Affine*>(a.in);
  const Fe* sp = reinterpret_cast<const Fe*>(a.in + 192);
  const uint32_t m = *reinterpret_cast<const uint32_t*>(a.in + 256);
  const uint32_t ad_len = *reinterpret_cast<const uint32_t*>(a.in + 260);
  const Affine* ios = reinterpret_cast<const Affine*>(a.in + 272);
  const uint8_t* ad = a.in + 272 + 128 * (size_t)m;
  const int canonical = a.canonical;
  int oob = 0;
  Affine PKC, R, OK;
  load_affine_fmt<S>(PKC, pts + 0, canonical, &oob);
  load_affine_fmt<S>(R, pts + 1, canonical, &oob);
  load_affine_fmt<S>(OK, pts + 2, canonical, &oob);
  for (uint32_t i = 0; i < 2 * m; i++) {
    Affine P;
    load_affine_fmt<S>(P, ios + i, canonical, &oob);
  }
  Fe s, sb;
  load_fe(s, sp);
  load_fe(sb, sp + 1);
  oob |= !(fe_in_range<FR>(s) && fe_in_range<FR>(sb));
  if (oob) {
    a.status[1] = 2;
    return;
  }
  if (!canonical) { from_mont<FR>(s, s); from_mont<FR>(sb, sb); }
  a.status[0] = ped_verify_one_g<S>([ios, canonical](uint32_t k) {
    Affine P;
    load_affine_fmt<S>(P, ios + k, canonical);
    return P;
  }, m, ad, ad_len, PKC, R, OK, s, sb);
  a.status[1] = 0;
}

}  // namespace avrf
