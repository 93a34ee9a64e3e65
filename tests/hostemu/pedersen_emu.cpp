// Test-only host build of the Pedersen-VRF device functions (ark_vrf_b200/csrc/pedersen.cuh: transcript, merge, prover,
// single verifier, the two equations) with the PTX carry flag emulated in C, as hostemu.cpp does for the arithmetic.
// NOT part of the product: libavrf_gpu.so never links it.
#include "../../ark_vrf_b200/csrc/pedersen.cuh"
#include <string.h>
using namespace avrf;

// points: Montgomery affine (16 words), I/O pairs 32 words each; scalars canonical (8 words)
template <int S> static void prove_t(const uint32_t* sk8, const uint32_t* pk16, const uint32_t* ios, uint32_t m,
                                     const uint8_t* ad, uint32_t ad_len, uint32_t* pkc16, uint32_t* r16, uint32_t* ok16,
                                     uint32_t* s8, uint32_t* sb8, uint32_t* bl8) {
  Fe sk, s, sb, bl;
  memcpy(sk.v, sk8, 32);
  Affine pk, PKC, R, OK;
  memcpy(&pk, pk16, 64);
  const Affine* io = reinterpret_cast<const Affine*>(ios);
  ped_prove_one_g<S>(PKC, R, OK, s, sb, bl, sk, pk, [io](uint32_t k) { return io[k]; }, m, ad, ad_len);
  memcpy(pkc16, &PKC, 64); memcpy(r16, &R, 64); memcpy(ok16, &OK, 64);
  memcpy(s8, s.v, 32); memcpy(sb8, sb.v, 32); memcpy(bl8, bl.v, 32);
}

template <int S> static int verify_t(const uint32_t* ios, uint32_t m, const uint8_t* ad, uint32_t ad_len,
                                     const uint32_t* pkc16, const uint32_t* r16, const uint32_t* ok16, const uint32_t* s8,
                                     const uint32_t* sb8) {
  Affine PKC, R, OK;
  memcpy(&PKC, pkc16, 64); memcpy(&R, r16, 64); memcpy(&OK, ok16, 64);
  Fe s, sb;
  memcpy(s.v, s8, 32); memcpy(sb.v, sb8, 32);
  const Affine* io = reinterpret_cast<const Affine*>(ios);
  return ped_verify_one_g<S>([io](uint32_t k) { return io[k]; }, m, ad, ad_len, PKC, R, OK, s, sb);
}

extern "C" {
void emu_ped_prove(int suite, const uint32_t* sk8, const uint32_t* pk16, const uint32_t* ios, uint32_t m, const uint8_t* ad,
                   uint32_t ad_len, uint32_t* pkc16, uint32_t* r16, uint32_t* ok16, uint32_t* s8, uint32_t* sb8, uint32_t* bl8) {
  if (suite == 0) prove_t<0>(sk8, pk16, ios, m, ad, ad_len, pkc16, r16, ok16, s8, sb8, bl8);
  else if (suite == 1) prove_t<1>(sk8, pk16, ios, m, ad, ad_len, pkc16, r16, ok16, s8, sb8, bl8);
  else prove_t<2>(sk8, pk16, ios, m, ad, ad_len, pkc16, r16, ok16, s8, sb8, bl8);
}
int emu_ped_verify(int suite, const uint32_t* ios, uint32_t m, const uint8_t* ad, uint32_t ad_len, const uint32_t* pkc16,
                   const uint32_t* r16, const uint32_t* ok16, const uint32_t* s8, const uint32_t* sb8) {
  if (suite == 0) return verify_t<0>(ios, m, ad, ad_len, pkc16, r16, ok16, s8, sb8);
  if (suite == 1) return verify_t<1>(ios, m, ad, ad_len, pkc16, r16, ok16, s8, sb8);
  return verify_t<2>(ios, m, ad, ad_len, pkc16, r16, ok16, s8, sb8);
}
}
