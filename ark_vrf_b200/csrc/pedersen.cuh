// Pedersen-VRF protocol pieces shared by the batch transcripts (k_prepare_ped), the prover (k_prove_ped) and the
// verifiers (k_verify_each_ped, k_verify_one_ped): one copy of the transcript, of the merge of the I/O pairs and of
// the two verification equations.  Host-compilable like thin.cuh (tests/hostemu/pedersen_emu.cpp).
//   transcript   utils::vrf_transcript without the Schnorr pair (reference src/utils/common.rs:159-225)
//   merge        common.rs:181-202,389-419
//   prove        pedersen::Prover::prove (src/pedersen.rs:136-186)
//   verify       pedersen::Verifier::verify (src/pedersen.rs:188-253)
#pragma once
#include "thin.cuh"

namespace avrf {

enum : uint32_t { DOM_PEDERSEN = 0x02, DOM_PEDERSEN_BLINDING = 0x12 };

// T = SUITE_ID || 0x02 || LE64(M) || enc(I_0) || enc(O_0) || ... || LE64(|ad|) || ad.  get_io(k) returns point k of
// the list I_0, O_0, I_1, O_1, ... as a Montgomery affine point.
template <int S, typename GetIo>
AVRF_HD void ped_transcript(Sha512& t, uint32_t m, GetIo get_io, const uint8_t* ad, uint32_t ad_len) {
  sha512_init(t);
  for (uint32_t i = 0; i < AVRF_CC(S).sid_len; i++) sha512_put_byte(t, AVRF_CC(S).suite_id[i]);
  sha512_put_byte(t, DOM_PEDERSEN);
  sha512_put_le64(t, m);
  uint32_t enc[8];
  for (uint32_t i = 0; i < 2 * m; i++) {
    Affine P = get_io(i);
    affine_compress<S>(enc, P);
    sha512_put_words(t, enc);
  }
  thin_transcript_ad(t, ad, ad_len);
}

// Merged pair in extended coordinates: the identity for M = 0, (I_0, O_0) for M = 1, sum z_i (I_i, O_i) with z_0 = 1
// and z_1 .. z_{M-1} from a fork of `t` otherwise.  OUT = false skips O_m (the prover needs I_m only).
template <int S, bool OUT, typename GetIo>
AVRF_HD void ped_merge(Ext& im, Ext& om, const Sha512& t, uint32_t m, GetIo get_io) {
  ext_identity<S>(im);
  ext_identity<S>(om);
  if (m == 0) return;
  affine_to_ext<S>(im, get_io(0));
  if (OUT) affine_to_ext<S>(om, get_io(1));
  thin_delinearize(t, m - 1, [&](uint32_t i, const uint32_t* z4) {
    uint32_t z8[8] = {z4[0], z4[1], z4[2], z4[3], 0, 0, 0, 0};
    Ext e, q;
    affine_to_ext<S>(e, get_io(2 * (i + 1)));
    ext_scalar_mul<S>(q, e, z8, 128);
    ext_add_c<S>(im, im, q);
    if (OUT) {
      affine_to_ext<S>(e, get_io(2 * (i + 1) + 1));
      ext_scalar_mul<S>(q, e, z8, 128);
      ext_add_c<S>(om, om, q);
    }
  });
}

// c = first 16 bytes of stream(T || enc(pk_com) || 0x40 || enc(R) || enc(Ok)); `t` must already hold enc(pk_com).
AVRF_HD void ped_challenge(Sha512& t, const uint32_t* r_enc, const uint32_t* ok_enc, uint32_t* c4) {
  sha512_put_byte(t, DOM_CHALLENGE);
  sha512_put_words(t, r_enc);
  sha512_put_words(t, ok_enc);
  uint64_t seed[8], blk[8];
  sha512_final(t, seed);
  sha512_xof_block(blk, seed, 0);
  digest_le128(c4, blk, 0);
}

template <int S>
AVRF_HD void blinding_base_ext(Ext& b) {
  Affine B;
  fe_set(B.x, AVRF_CC(S).bx);
  fe_set(B.y, AVRF_CC(S).by);
  affine_to_ext<S>(b, B);
}

// The two equations of pedersen.rs:233-250, each tested on its own with INTEGER scalars (s, sb < r; c < 2^128) and no
// weight, so the verdict is exact on every curve point, in the prime-order subgroup or not:
//     s*I_m - c*O_m == Ok      and      s*G + sb*B - c*pk_com == R
// pt(k) returns point k (PED_IM .. PED_R) in extended coordinates when it is needed, so that no more than two
// points are live at a time.
enum : int { PED_IM, PED_OM, PED_OK, PED_PKCOM, PED_R };
template <int S, typename GetPt>
AVRF_HD bool ped_equations_hold(GetPt pt, const uint32_t* c4, const Fe& s, const Fe& sb) {
  uint32_t c8[8] = {c4[0], c4[1], c4[2], c4[3], 0, 0, 0, 0};
  Ext q, e;
  ext_scalar_mul<S>(q, pt(PED_IM), s.v, 256);
  ext_scalar_mul<S>(e, pt(PED_OM), c8, 128);
  ext_neg<S>(e, e);
  ext_add_c<S>(q, q, e);
  ext_neg<S>(e, pt(PED_OK));
  ext_add_c<S>(q, q, e);
  const bool first = ext_is_identity<S>(q);
  Affine g;
  fe_set(g.x, AVRF_CC(S).gx);
  fe_set(g.y, AVRF_CC(S).gy);
  affine_to_ext<S>(e, g);
  ext_scalar_mul<S>(q, e, s.v, 256);
  blinding_base_ext<S>(e);
  ext_scalar_mul<S>(e, e, sb.v, 256);
  ext_add_c<S>(q, q, e);
  ext_scalar_mul<S>(e, pt(PED_PKCOM), c8, 128);
  ext_neg<S>(e, e);
  ext_add_c<S>(q, q, e);
  ext_neg<S>(e, pt(PED_R));
  ext_add_c<S>(q, q, e);
  return first && ext_is_identity<S>(q);
}

// pedersen::Prover::prove for one proof.  sk canonical; pk = sk*G, Montgomery affine.  Outputs pk_com, R, Ok
// (Montgomery affine) and s, sb, blinding (canonical).  Four full-width scalar multiplications; R and Ok share one
// inversion (pk_com is normalised on its own: its encoding enters the transcript that derives k and kb).
template <int S, typename GetIo>
AVRF_HD void ped_prove_one_g(Affine& PKC, Affine& R, Affine& OK, Fe& s_out, Fe& sb_out, Fe& bl, const Fe& sk,
                             const Affine& pk, GetIo get_io, uint32_t m, const uint8_t* ad, uint32_t ad_len) {
  constexpr int FQ = SuiteT<S>::FQ;
  constexpr int FR = SuiteT<S>::FR;
  Sha512 t;
  ped_transcript<S>(t, m, get_io, ad, ad_len);
  Ext im, om;
  ped_merge<S, false>(im, om, t, m, get_io);
  {
    Sha512 tb = t;
    sha512_put_byte(tb, DOM_PEDERSEN_BLINDING);              // PedersenSuite::blinding (pedersen.rs:28-31)
    thin_nonce<S>(bl, tb, sk);
  }
  Ext q, e;
  blinding_base_ext<S>(e);
  ext_scalar_mul<S>(q, e, bl.v, 256);
  affine_to_ext<S>(e, pk);
  ext_add_c<S>(q, q, e);
  ext_to_affine<S>(PKC, q);                                  // pk_com = pk + blinding*B
  uint32_t enc[8], enc2[8];
  affine_compress<S>(enc, PKC);
  sha512_put_words(t, enc);
  Fe k, kb;
  thin_nonce<S>(k, t, sk);
  thin_nonce<S>(kb, t, bl);
  Ext rr, oo;
  ext_scalar_mul<S>(oo, im, k.v, 256);                       // Ok = k*I_m
  {
    Affine g;
    fe_set(g.x, AVRF_CC(S).gx);
    fe_set(g.y, AVRF_CC(S).gy);
    affine_to_ext<S>(e, g);
  }
  ext_scalar_mul<S>(rr, e, k.v, 256);
  blinding_base_ext<S>(e);
  ext_scalar_mul<S>(q, e, kb.v, 256);
  ext_add_c<S>(rr, rr, q);                                   // R = k*G + kb*B
  Fe zz, inv, zi;                                            // one inversion for both
  mont_mul_c<FQ>(zz, rr.z, oo.z);
  fe_inv<FQ>(inv, zz);
  mont_mul_c<FQ>(zi, inv, oo.z);
  mont_mul_c<FQ>(R.x, rr.x, zi);
  mont_mul_c<FQ>(R.y, rr.y, zi);
  mont_mul_c<FQ>(zi, inv, rr.z);
  mont_mul_c<FQ>(OK.x, oo.x, zi);
  mont_mul_c<FQ>(OK.y, oo.y, zi);
  affine_compress<S>(enc, R);
  affine_compress<S>(enc2, OK);
  uint32_t c4[4];
  ped_challenge(t, enc, enc2, c4);
  // s = k + c*sk, sb = kb + c*blinding (mod r)
  Fe c8, xm, cx;
  fe_zero(c8);
  for (int i = 0; i < 4; i++) c8.v[i] = c4[i];
  to_mont<FR>(xm, sk);
  mont_mul_c<FR>(cx, c8, xm);
  fe_add<FR>(s_out, k, cx);
  to_mont<FR>(xm, bl);
  mont_mul_c<FR>(cx, c8, xm);
  fe_add<FR>(sb_out, kb, cx);
}

// pedersen::Verifier::verify for one proof: status 0 Ok / 1 VerificationFailure / 2 InvalidData (an identity pk_com or
// I/O point; it takes precedence over the equations).  Points Montgomery affine, s and sb canonical.
template <int S, typename GetIo>
AVRF_HD int ped_verify_one_g(GetIo get_io, uint32_t m, const uint8_t* ad, uint32_t ad_len, const Affine& pkcom,
                             const Affine& R, const Affine& OK, const Fe& s, const Fe& sb) {
  bool bad = affine_is_identity<S>(pkcom);
  for (uint32_t i = 0; i < 2 * m; i++) bad |= affine_is_identity<S>(get_io(i));
  if (bad) return 2;                                         // AVRF_INVALID_DATA
  Sha512 t;
  ped_transcript<S>(t, m, get_io, ad, ad_len);
  Ext im, om;
  ped_merge<S, true>(im, om, t, m, get_io);
  uint32_t enc[8], enc2[8];
  affine_compress<S>(enc, pkcom);
  sha512_put_words(t, enc);
  affine_compress<S>(enc, R);
  affine_compress<S>(enc2, OK);
  uint32_t c4[4];
  ped_challenge(t, enc, enc2, c4);
  return ped_equations_hold<S>([&](int k) {
    Ext e = k == PED_IM ? im : om;
    if (k >= PED_OK) affine_to_ext<S>(e, k == PED_OK ? OK : k == PED_PKCOM ? pkcom : R);
    return e;
  }, c4, s, sb) ? 0 : 1;
}

}  // namespace avrf
