/* avrf_oracle.c - CPU restatement (plain C) of ark-vrf's Thin-VRF hot path.
 *
 * TEST INFRASTRUCTURE ONLY: the checker for tests/, __graft_entry__.smoke() and the
 * `cpu_baseline` / `--impl reference` legs of bench.py.  Nothing in ark_vrf_b200/ links or
 * calls it.  Parity status: PINNED - tests/test_oracle_c.py replays the reference's golden
 * vectors (tests/golden/ *_thin.json) through this file and cross-checks it against the
 * independent Python restatement (oracle/pyref.py).
 *
 * The reference (Rust, arkworks 0.6 crates not vendored, no Rust toolchain in this image)
 * cannot be compiled here, so this is a restatement; each function cites the reference
 * file:line it follows (paths relative to /root/reference/).  Third-party behaviour restated
 * from the published algorithms: ark-ff 0.6 Montgomery fields (4x64-bit limbs, R = 2^256),
 * ark-ec 0.6 twisted-Edwards group law / VariableBaseMSM (signed-digit Pippenger, window
 * c = ln(n)+2, one worker per window under `parallel`) / Elligator2Map, ark-serialize 0.6
 * compressed encodings, sha2 0.10 SHA-512.
 */
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <math.h>

typedef uint64_t u64;
typedef unsigned __int128 u128;

typedef struct {
  const char* suite_id; int sid_len;
  u64 p[4], r[4]; int a; u64 d[4], gx[4], gy[4], mont_j[4], mont_k[4], ell2_z[4];
  int cof_log2, has_ell2;
} orc_suite_params;
#include "oracle_constants.h"

/* ------------------------------------------------------------------------------------ */
/* SHA-512 (sha2 0.10)                                                                  */
/* ------------------------------------------------------------------------------------ */
/* OpenSSL's SHA-512 block function (assembly: AVX2 / BMI2 on x86-64), the counterpart of the `asm` feature of the sha2 crate
 * that the reference's published numbers were taken with (Cargo.toml:103-108, benches/SUMMARY.md:3-15).  The low-level
 * context is a plain struct, so a transcript fork (transcript.rs:118-130) is a struct copy. */
#define OPENSSL_SUPPRESS_DEPRECATED 1
#include <openssl/sha.h>
typedef SHA512_CTX sha512_t;
static void sha_init(sha512_t* s) { SHA512_Init(s); }
static void sha_update(sha512_t* s, const void* data, size_t n) { SHA512_Update(s, data, n); }
static void sha_final(sha512_t* s, uint8_t out[64]) { SHA512_Final(out, s); }

/* Transcript (src/utils/transcript.rs:176-274): absorb = SHA-512 update; squeeze = counter mode */
typedef struct { sha512_t h; int squeezing; uint8_t seed[64]; u64 pos; uint8_t block[64]; u64 block_idx; } tr_t;
static void tr_new(tr_t* t, const void* label, size_t n) { sha_init(&t->h); t->squeezing = 0; t->pos = 0; t->block_idx = ~(u64)0; sha_update(&t->h, label, n); }
static void tr_absorb(tr_t* t, const void* d, size_t n) { sha_update(&t->h, d, n); }
static void tr_absorb_u8(tr_t* t, uint8_t b) { sha_update(&t->h, &b, 1); }
static void tr_absorb_le64(tr_t* t, u64 v) { uint8_t b[8]; for (int i = 0; i < 8; i++) b[i] = (uint8_t)(v >> (8 * i)); sha_update(&t->h, b, 8); }
static void tr_squeeze(tr_t* t, uint8_t* out, size_t n) {             /* transcript.rs:191-194,230-273 */
  if (!t->squeezing) { sha_final(&t->h, t->seed); t->squeezing = 1; t->pos = 0; }
  while (n) {
    u64 blk = t->pos / 64, off = t->pos % 64;
    if (blk != t->block_idx) {                                          /* DigestXofReader buffer, transcript.rs:258-265 */
      sha512_t c; uint8_t ctr[8];
      for (int i = 0; i < 8; i++) ctr[i] = (uint8_t)(blk >> (8 * i));
      sha_init(&c); sha_update(&c, t->seed, 64); sha_update(&c, ctr, 8); sha_final(&c, t->block); t->block_idx = blk;
    }
    size_t take = 64 - off; if (take > n) take = n;
    memcpy(out, t->block + off, take); out += take; n -= take; t->pos += take;
  }
}

/* ------------------------------------------------------------------------------------ */
/* Prime fields, 4x64 Montgomery (ark-ff 0.6 MontBackend)                               */
/* ------------------------------------------------------------------------------------ */
typedef struct { u64 v[4]; } fe;
typedef struct { u64 p[4], one[4], r2[4], n0, pm2[4], phalf[4]; int bits; } fctx;

static int ge4(const u64* a, const u64* b) { for (int i = 3; i >= 0; i--) { if (a[i] != b[i]) return a[i] > b[i]; } return 1; }
static u64 add4(u64* r, const u64* a, const u64* b) { u128 c = 0; for (int i = 0; i < 4; i++) { c += (u128)a[i] + b[i]; r[i] = (u64)c; c >>= 64; } return (u64)c; }
static u64 sub4(u64* r, const u64* a, const u64* b) { u128 br = 0; for (int i = 0; i < 4; i++) { u128 t = (u128)a[i] - b[i] - br; r[i] = (u64)t; br = (t >> 64) & 1; } return (u64)br; }

static inline void f_add(const fctx* F, fe* r, const fe* a, const fe* b) { u64 t[4]; add4(t, a->v, b->v); if (ge4(t, F->p)) sub4(t, t, F->p); memcpy(r->v, t, 32); }
static inline void f_sub(const fctx* F, fe* r, const fe* a, const fe* b) { u64 t[4]; if (sub4(t, a->v, b->v)) add4(t, t, F->p); memcpy(r->v, t, 32); }
static inline int f_is_zero(const fe* a) { return (a->v[0] | a->v[1] | a->v[2] | a->v[3]) == 0; }
static inline int f_eq(const fe* a, const fe* b) { return memcmp(a->v, b->v, 32) == 0; }
static inline void f_neg(const fctx* F, fe* r, const fe* a) { if (f_is_zero(a)) { *r = *a; return; } u64 t[4]; sub4(t, F->p, a->v); memcpy(r->v, t, 32); }

/* Montgomery multiplication, 4 x 64-bit limbs, CIOS with the "no-carry" shortcut that ark-ff 0.6 (and gnark) use for
 * moduli whose top bit is clear - every modulus in scope is < 2^255.  Written in unsigned __int128: with -mbmi2 gcc
 * emits one mulx per product and add/adc chains.  (A hand-scheduled _mulx_u64 / _addcarryx_u64 variant, the shape of
 * ark-ff's `asm` feature, reference Cargo.toml:103-108, was tried and measured slower under gcc 13, which does not
 * keep the two carry chains in adcx / adox; the anchor for this port is the published 14.3 ms at N = 256.) */
static inline void f_mul(const fctx* F, fe* r, const fe* a, const fe* b) {
  u64 t[4] = {0, 0, 0, 0};
  for (int i = 0; i < 4; i++) {
    u128 A = (u128)a->v[0] * b->v[i] + t[0];
    u64 m = (u64)A * F->n0;
    u128 C = (u128)m * F->p[0] + (u64)A;
    for (int j = 1; j < 4; j++) {
      A = (u128)a->v[j] * b->v[i] + t[j] + (u64)(A >> 64);
      C = (u128)m * F->p[j] + (u64)A + (u64)(C >> 64);
      t[j - 1] = (u64)C;
    }
    t[3] = (u64)(A >> 64) + (u64)(C >> 64);
  }
  if (ge4(t, F->p)) sub4(t, t, F->p);
  memcpy(r->v, t, 32);
}
static inline void f_sqr(const fctx* F, fe* r, const fe* a) { f_mul(F, r, a, a); }
static void f_to_mont(const fctx* F, fe* r, const fe* a) { fe r2; memcpy(r2.v, F->r2, 32); f_mul(F, r, a, &r2); }
static void f_from_mont(const fctx* F, fe* r, const fe* a) { fe one = {{1, 0, 0, 0}}; f_mul(F, r, a, &one); }
static void f_one(const fctx* F, fe* r) { memcpy(r->v, F->one, 32); }
static void f_pow(const fctx* F, fe* r, const fe* a, const u64* e) {
  fe acc; f_one(F, &acc);
  for (int i = 255; i >= 0; i--) { f_sqr(F, &acc, &acc); if ((e[i >> 6] >> (i & 63)) & 1) f_mul(F, &acc, &acc, a); }
  *r = acc;
}
static void f_inv(const fctx* F, fe* r, const fe* a) { f_pow(F, r, a, F->pm2); }
static void f_reduce(const fctx* F, u64* a) { while (ge4(a, F->p)) sub4(a, a, F->p); }

static void fctx_init(fctx* F, const u64* p) {
  memcpy(F->p, p, 32);
  u64 inv = 1; for (int i = 0; i < 6; i++) inv *= 2 - p[0] * inv;      /* p^-1 mod 2^64 */
  F->n0 = (u64)0 - inv;
  u64 x[4] = {1, 0, 0, 0};
  for (int i = 0; i < 512; i++) {                                      /* x = 2^i mod p */
    if (i == 256) memcpy(F->one, x, 32);
    u64 c = add4(x, x, x); if (c || ge4(x, p)) sub4(x, x, p);
  }
  memcpy(F->r2, x, 32);
  u64 two[4] = {2, 0, 0, 0}, one[4] = {1, 0, 0, 0};
  sub4(F->pm2, p, two);
  sub4(F->phalf, p, one);
  for (int i = 0; i < 4; i++) F->phalf[i] = (F->phalf[i] >> 1) | (i < 3 ? F->phalf[i + 1] << 63 : 0);
  F->bits = 256; while (!((p[(F->bits - 1) >> 6] >> ((F->bits - 1) & 63)) & 1)) F->bits--;
}

/* ------------------------------------------------------------------------------------ */
/* Suite context                                                                         */
/* ------------------------------------------------------------------------------------ */
typedef struct { fe x, y; } aff;              /* Montgomery coordinates */
typedef struct { fe x, y, z, t; } ext;

typedef struct {
  const orc_suite_params* P; fctx Fq, Fr; fe d, jk, k2inv, kk, zz, ts_root; u64 ts_exp[4]; int ts_s; aff G; int init;
} sctx;
static sctx SC[3];
static pthread_once_t sc_once = PTHREAD_ONCE_INIT;

static void fq_set(const sctx* S, fe* r, const u64* canon) { fe t; memcpy(t.v, canon, 32); f_to_mont(&S->Fq, r, &t); }

static void sc_init_all(void) {
  for (int s = 0; s < 3; s++) {
    sctx* S = &SC[s]; S->P = &ORC_PARAMS[s];
    fctx_init(&S->Fq, S->P->p); fctx_init(&S->Fr, S->P->r);
    fq_set(S, &S->d, S->P->d); fq_set(S, &S->G.x, S->P->gx); fq_set(S, &S->G.y, S->P->gy);
    if (S->P->has_ell2) {
      fe J, K, ki; fq_set(S, &J, S->P->mont_j); fq_set(S, &K, S->P->mont_k); fq_set(S, &S->zz, S->P->ell2_z);
      f_inv(&S->Fq, &ki, &K); f_mul(&S->Fq, &S->jk, &J, &ki); f_sqr(&S->Fq, &S->k2inv, &ki); S->kk = K;
    }
    /* Tonelli-Shanks parameters: p - 1 = 2^s q */
    u64 q[4], one[4] = {1, 0, 0, 0}; sub4(q, S->P->p, one); S->ts_s = 0;
    while (!(q[0] & 1)) { for (int i = 0; i < 4; i++) q[i] = (q[i] >> 1) | (i < 3 ? q[i + 1] << 63 : 0); S->ts_s++; }
    u64 qm1[4]; sub4(qm1, q, one);
    for (int i = 0; i < 4; i++) S->ts_exp[i] = (qm1[i] >> 1) | (i < 3 ? qm1[i + 1] << 63 : 0);
    for (u64 z = 2;; z++) {
      fe zc = {{z, 0, 0, 0}}, zm, l, mone, o; f_to_mont(&S->Fq, &zm, &zc); f_pow(&S->Fq, &l, &zm, S->Fq.phalf);
      f_one(&S->Fq, &o); f_neg(&S->Fq, &mone, &o);
      if (f_eq(&l, &mone)) { f_pow(&S->Fq, &S->ts_root, &zm, q); break; }
    }
    S->init = 1;
  }
}
static const sctx* suite(int s) { pthread_once(&sc_once, sc_init_all); return (s >= 0 && s < 3) ? &SC[s] : NULL; }

/* ------------------------------------------------------------------------------------ */
/* Twisted Edwards group law (ark-ec 0.6 twisted_edwards, extended coordinates)          */
/* ------------------------------------------------------------------------------------ */
static void mul_a(const sctx* S, fe* r, const fe* x) {                 /* r = a * x */
  const fctx* F = &S->Fq;
  if (S->P->a == 1) { *r = *x; return; }
  if (S->P->a == -1) { f_neg(F, r, x); return; }
  fe t; f_add(F, &t, x, x); f_add(F, &t, &t, &t); f_add(F, &t, &t, x); f_neg(F, r, &t);   /* -5 */
}
static void ext_id(const sctx* S, ext* p) { memset(p, 0, sizeof *p); f_one(&S->Fq, &p->y); f_one(&S->Fq, &p->z); }
static int ext_is_id(const ext* p) { return f_is_zero(&p->x) && f_eq(&p->y, &p->z); }
static void ext_from_aff(const sctx* S, ext* r, const aff* a) { r->x = a->x; r->y = a->y; f_one(&S->Fq, &r->z); f_mul(&S->Fq, &r->t, &a->x, &a->y); }
static void ext_add(const sctx* S, ext* r, const ext* p, const ext* q) {   /* add-2008-hwcd */
  const fctx* F = &S->Fq; fe A, B, C, D, E, Ff, G, H, t0, t1;
  f_mul(F, &A, &p->x, &q->x); f_mul(F, &B, &p->y, &q->y); f_mul(F, &C, &p->t, &q->t); f_mul(F, &C, &C, &S->d);
  f_mul(F, &D, &p->z, &q->z); f_add(F, &t0, &p->x, &p->y); f_add(F, &t1, &q->x, &q->y); f_mul(F, &E, &t0, &t1);
  f_sub(F, &E, &E, &A); f_sub(F, &E, &E, &B); f_sub(F, &Ff, &D, &C); f_add(F, &G, &D, &C);
  mul_a(S, &t0, &A); f_sub(F, &H, &B, &t0);
  f_mul(F, &r->x, &E, &Ff); f_mul(F, &r->y, &G, &H); f_mul(F, &r->t, &E, &H); f_mul(F, &r->z, &Ff, &G);
}
static void ext_madd(const sctx* S, ext* r, const ext* p, const aff* q, int neg) {   /* mixed, Z2 = 1 */
  const fctx* F = &S->Fq; fe A, B, C, E, Ff, G, H, t0, t1, qx = q->x;
  if (neg) f_neg(F, &qx, &qx);
  f_mul(F, &A, &p->x, &qx); f_mul(F, &B, &p->y, &q->y); f_mul(F, &t0, &qx, &q->y); f_mul(F, &C, &p->t, &t0); f_mul(F, &C, &C, &S->d);
  f_add(F, &t0, &p->x, &p->y); f_add(F, &t1, &qx, &q->y); f_mul(F, &E, &t0, &t1);
  f_sub(F, &E, &E, &A); f_sub(F, &E, &E, &B); f_sub(F, &Ff, &p->z, &C); f_add(F, &G, &p->z, &C);
  mul_a(S, &t0, &A); f_sub(F, &H, &B, &t0);
  f_mul(F, &r->x, &E, &Ff); f_mul(F, &r->y, &G, &H); f_mul(F, &r->t, &E, &H); f_mul(F, &r->z, &Ff, &G);
}
static void ext_dbl(const sctx* S, ext* r, const ext* p) {             /* dbl-2008-hwcd */
  const fctx* F = &S->Fq; fe A, B, C, D, E, Ff, G, H, t0;
  f_sqr(F, &A, &p->x); f_sqr(F, &B, &p->y); f_sqr(F, &C, &p->z); f_add(F, &C, &C, &C); mul_a(S, &D, &A);
  f_add(F, &t0, &p->x, &p->y); f_sqr(F, &E, &t0); f_sub(F, &E, &E, &A); f_sub(F, &E, &E, &B);
  f_add(F, &G, &D, &B); f_sub(F, &Ff, &G, &C); f_sub(F, &H, &D, &B);
  f_mul(F, &r->x, &E, &Ff); f_mul(F, &r->y, &G, &H); f_mul(F, &r->t, &E, &H); f_mul(F, &r->z, &Ff, &G);
}
static void ext_neg(const sctx* S, ext* r, const ext* p) { *r = *p; f_neg(&S->Fq, &r->x, &p->x); f_neg(&S->Fq, &r->t, &p->t); }
static void ext_to_aff(const sctx* S, aff* r, const ext* p) { fe zi; f_inv(&S->Fq, &zi, &p->z); f_mul(&S->Fq, &r->x, &p->x, &zi); f_mul(&S->Fq, &r->y, &p->y, &zi); }
static void ext_mul(const sctx* S, ext* r, const ext* p, const u64* k) {   /* double-and-add, MSB first */
  ext acc; ext_id(S, &acc);
  for (int i = 255; i >= 0; i--) { ext_dbl(S, &acc, &acc); if ((k[i >> 6] >> (i & 63)) & 1) ext_add(S, &acc, &acc, p); }
  *r = acc;
}
static int aff_is_id(const sctx* S, const aff* a) { fe o; f_one(&S->Fq, &o); return f_is_zero(&a->x) && f_eq(&a->y, &o); }

/* encodings (ark-serialize 0.6 compressed; SURVEY.md A.2) */
static void aff_load(const sctx* S, aff* r, const uint8_t* b64) { fe t; memcpy(t.v, b64, 32); f_to_mont(&S->Fq, &r->x, &t); memcpy(t.v, b64 + 32, 32); f_to_mont(&S->Fq, &r->y, &t); }
static void aff_store(const sctx* S, uint8_t* b64, const aff* a) { fe t; f_from_mont(&S->Fq, &t, &a->x); memcpy(b64, t.v, 32); f_from_mont(&S->Fq, &t, &a->y); memcpy(b64 + 32, t.v, 32); }
static void aff_enc(const sctx* S, uint8_t out[32], const aff* a) {
  fe x, y; f_from_mont(&S->Fq, &x, &a->x); f_from_mont(&S->Fq, &y, &a->y);
  memcpy(out, y.v, 32);
  if (!ge4(S->Fq.phalf, x.v)) out[31] |= 0x80;                         /* x > (p-1)/2  <=>  x > p - x */
}

/* Tonelli-Shanks; returns 0 for non-residues */
static int f_sqrt(const sctx* S, fe* r, const fe* a) {
  const fctx* F = &S->Fq; fe one, w, x, b, z; f_one(F, &one);
  if (f_is_zero(a)) { *r = *a; return 1; }
  f_pow(F, &w, a, S->ts_exp); f_mul(F, &x, a, &w); f_mul(F, &b, &x, &w); z = S->ts_root; int v = S->ts_s;
  while (!f_eq(&b, &one)) {
    int k = 0; fe t = b;
    while (!f_eq(&t, &one)) { f_sqr(F, &t, &t); k++; if (k == v) return 0; }
    fe g = z; for (int i = 0; i + k + 1 < v; i++) f_sqr(F, &g, &g);
    f_sqr(F, &z, &g); f_mul(F, &b, &b, &z); f_mul(F, &x, &x, &g); v = k;
  }
  *r = x; return 1;
}

/* ark-ec Affine::get_point_from_y_unchecked */
static int point_from_y(const sctx* S, aff* out, const fe* y, int greatest) {
  const fctx* F = &S->Fq; fe one, y2, num, den, a1, inv, x2, x, xc;
  f_one(F, &one); f_sqr(F, &y2, y); f_sub(F, &num, &one, &y2); f_mul(F, &den, &S->d, &y2); mul_a(S, &a1, &one); f_sub(F, &den, &a1, &den);
  if (f_is_zero(&den)) return 0;
  f_inv(F, &inv, &den); f_mul(F, &x2, &num, &inv);
  if (!f_sqrt(S, &x, &x2)) return 0;
  f_from_mont(F, &xc, &x);
  int big = !ge4(F->phalf, xc.v);
  if (big != greatest) f_neg(F, &x, &x);
  out->x = x; out->y = *y; return 1;
}

/* ------------------------------------------------------------------------------------ */
/* Hash-to-curve (src/utils/hash_to_curve.rs)                                            */
/* ------------------------------------------------------------------------------------ */
static void fe_from_be48(const fctx* F, fe* r_mont, const uint8_t* b) {   /* from_be_bytes_mod_order, 48 B */
  fe lo, hi, t; memset(&hi, 0, sizeof hi);
  for (int i = 0; i < 4; i++) { u64 v = 0; for (int k = 0; k < 8; k++) v = (v << 8) | b[16 + 8 * (3 - i) + k]; lo.v[i] = v; }
  for (int i = 0; i < 2; i++) { u64 v = 0; for (int k = 0; k < 8; k++) v = (v << 8) | b[8 * (1 - i) + k]; hi.v[i] = v; }
  f_reduce(F, lo.v); f_to_mont(F, &lo, &lo); f_to_mont(F, &t, &hi); f_to_mont(F, &t, &t); f_add(F, r_mont, &lo, &t);
}
static void ell2_map(const sctx* S, aff* out, const fe* u) {              /* SURVEY.md A.6 */
  const fctx* F = &S->Fq; fe one, t, den, inv, x1, gx, y, x, yc, s, tt, tv1, tv2; int sgn;
  f_one(F, &one); f_sqr(F, &t, u); f_mul(F, &t, &t, &S->zz); f_add(F, &den, &one, &t);
  if (f_is_zero(&den)) den = one;
  f_inv(F, &inv, &den); f_mul(F, &x1, &S->jk, &inv); f_neg(F, &x1, &x1);
#define GX(r, xx) do { fe a_; f_add(F, &a_, (xx), &S->jk); f_mul(F, &a_, &a_, (xx)); f_add(F, &a_, &a_, &S->k2inv); f_mul(F, (r), &a_, (xx)); } while (0)
  GX(&gx, &x1);
  if (!f_is_zero(&gx) && f_sqrt(S, &y, &gx)) { x = x1; sgn = 1; }
  else { f_add(F, &x, &x1, &S->jk); f_neg(F, &x, &x); GX(&gx, &x); f_sqrt(S, &y, &gx); sgn = 0; }
  f_from_mont(F, &yc, &y);
  if ((int)(yc.v[0] & 1) != sgn) f_neg(F, &y, &y);
  f_mul(F, &s, &x, &S->kk); f_mul(F, &tt, &y, &S->kk); f_add(F, &tv1, &s, &one); f_mul(F, &tv2, &tv1, &tt);
  if (f_is_zero(&tv2)) { memset(&out->x, 0, sizeof(fe)); out->y = one; return; }
  f_inv(F, &inv, &tv2); f_mul(F, &t, &tv1, &s); f_mul(F, &out->x, &t, &inv);
  f_sub(F, &t, &s, &one); f_mul(F, &t, &t, &tt); f_mul(F, &out->y, &t, &inv);
}
static void h2c_ell2(const sctx* S, aff* out, const uint8_t* msg, size_t len) {   /* hash_to_curve.rs:66-100 */
  uint8_t dstp[40], b0[64], b1[64], b2[64], zpad[48] = {0}, hdr[3] = {0, 96, 0}, x[64], u[96], one = 1, two = 2;
  int dl = S->P->sid_len + 1;
  memcpy(dstp, S->P->suite_id, S->P->sid_len); dstp[dl - 1] = 0x60; dstp[dl] = (uint8_t)dl;
  sha512_t h;
  sha_init(&h); sha_update(&h, zpad, 48); sha_update(&h, msg, len); sha_update(&h, hdr, 3); sha_update(&h, dstp, dl + 1); sha_final(&h, b0);
  sha_init(&h); sha_update(&h, b0, 64); sha_update(&h, &one, 1); sha_update(&h, dstp, dl + 1); sha_final(&h, b1);
  for (int i = 0; i < 64; i++) x[i] = b0[i] ^ b1[i];
  sha_init(&h); sha_update(&h, x, 64); sha_update(&h, &two, 1); sha_update(&h, dstp, dl + 1); sha_final(&h, b2);
  memcpy(u, b1, 64); memcpy(u + 64, b2, 32);
  fe u0, u1; fe_from_be48(&S->Fq, &u0, u); fe_from_be48(&S->Fq, &u1, u + 48);
  aff q0, q1; ell2_map(S, &q0, &u0); ell2_map(S, &q1, &u1);
  ext e0, e1; ext_from_aff(S, &e0, &q0); ext_from_aff(S, &e1, &q1); ext_add(S, &e0, &e0, &e1);
  for (int i = 0; i < S->P->cof_log2; i++) ext_dbl(S, &e0, &e0);
  ext_to_aff(S, out, &e0);
}
static int h2c_tai(const sctx* S, aff* out, const uint8_t* msg, size_t len) {     /* hash_to_curve.rs:34-57 */
  tr_t prefix; tr_new(&prefix, S->P->suite_id, S->P->sid_len); tr_absorb_u8(&prefix, 0x60); tr_absorb_le64(&prefix, len); tr_absorb(&prefix, msg, len);
  for (int ctr = 0; ctr < 256; ctr++) {
    tr_t t = prefix; tr_absorb_u8(&t, (uint8_t)ctr);
    uint8_t hb[32]; tr_squeeze(&t, hb, 32);
    int flag = hb[31] >> 7; hb[31] &= (uint8_t)(0xFF >> (256 - S->Fq.bits));
    fe y; memcpy(y.v, hb, 32);
    if (ge4(y.v, S->Fq.p)) continue;
    f_to_mont(&S->Fq, &y, &y);
    aff P; if (!point_from_y(S, &P, &y, flag)) continue;
    ext e; ext_from_aff(S, &e, &P);
    for (int i = 0; i < S->P->cof_log2; i++) ext_dbl(S, &e, &e);
    if (ext_is_id(&e)) continue;
    ext_to_aff(S, out, &e); return 1;
  }
  return 0;
}
static int data_to_point(const sctx* S, aff* out, const uint8_t* msg, size_t len) { if (S->P->has_ell2) { h2c_ell2(S, out, msg, len); return 1; } return h2c_tai(S, out, msg, len); }

/* ------------------------------------------------------------------------------------ */
/* Protocol hashing (src/utils/common.rs)                                                */
/* ------------------------------------------------------------------------------------ */
static void fr_from_le(const fctx* F, fe* r_canon, const uint8_t* b, int n) {     /* from_le_bytes_mod_order, n <= 48 */
  uint8_t buf[48] = {0}; memcpy(buf, b, n);
  fe lo, hi, t; memcpy(lo.v, buf, 32); memset(&hi, 0, sizeof hi); memcpy(hi.v, buf + 32, 16);
  f_reduce(F, lo.v); f_to_mont(F, &t, &hi); f_add(F, r_canon, &lo, &t);
}
static void challenge_scalar(const sctx* S, tr_t* t, fe* r_canon) { uint8_t b[16]; tr_squeeze(t, b, 16); fr_from_le(&S->Fr, r_canon, b, 16); }   /* common.rs:72-76 */
static void nonce(const sctx* S, fe* k_canon, const fe* sk_canon, const tr_t* t0) {        /* common.rs:313-328 */
  tr_t te = *t0, tn = *t0; uint8_t skh[64], out[48];
  tr_absorb_u8(&te, 0x10); tr_absorb(&te, sk_canon->v, 32); tr_squeeze(&te, skh, 64);
  tr_absorb_u8(&tn, 0x11); tr_absorb(&tn, skh, 64);
  int n = (S->Fr.bits + 128 + 7) / 8; tr_squeeze(&tn, out, n); fr_from_le(&S->Fr, k_canon, out, n);
}
/* vrf_transcript_base + chain_ios (common.rs:159-173,231-240): T and zs[1..m] (canonical) */
static void thin_transcript(const sctx* S, tr_t* t, fe* zs, const aff* pk, const aff* ios, int m, const uint8_t* ad, size_t ad_len) {
  uint8_t e[32];
  tr_new(t, S->P->suite_id, S->P->sid_len); tr_absorb_u8(t, 0x01); tr_absorb_le64(t, (u64)m + 1);
  aff_enc(S, e, &S->G); tr_absorb(t, e, 32); aff_enc(S, e, pk); tr_absorb(t, e, 32);
  for (int i = 0; i < 2 * m; i++) { aff_enc(S, e, &ios[i]); tr_absorb(t, e, 32); }
  tr_absorb_le64(t, ad_len); tr_absorb(t, ad, ad_len);
  if (m) { tr_t tz = *t; tr_absorb_u8(&tz, 0x30); for (int i = 0; i < m; i++) challenge_scalar(S, &tz, &zs[i]); }
}
static void challenge(const sctx* S, tr_t* t, const aff* R, fe* c_canon) { uint8_t e[32]; tr_absorb_u8(t, 0x40); aff_enc(S, e, R); tr_absorb(t, e, 32); challenge_scalar(S, t, c_canon); }

/* ------------------------------------------------------------------------------------ */
/* C ABI (canonical little-endian bytes everywhere)                                      */
/* ------------------------------------------------------------------------------------ */
enum { ORC_OK = 0, ORC_VERIFICATION_FAILURE = 1, ORC_INVALID_DATA = 2 };

int orc_hash_to_curve(int s, const uint8_t* msg, size_t len, uint8_t out64[64]) {
  const sctx* S = suite(s); aff P; if (!S || !data_to_point(S, &P, msg, len)) return 0; aff_store(S, out64, &P); return 1;
}
void orc_point_compress(int s, const uint8_t in64[64], uint8_t out32[32]) { const sctx* S = suite(s); aff P; aff_load(S, &P, in64); aff_enc(S, out32, &P); }
void orc_scalar_mul(int s, const uint8_t k32[32], const uint8_t* in64, uint8_t out64[64]) {   /* in64 NULL: generator */
  const sctx* S = suite(s); aff P; if (in64) aff_load(S, &P, in64); else P = S->G;
  ext e; ext_from_aff(S, &e, &P); u64 k[4]; memcpy(k, k32, 32); ext_mul(S, &e, &e, k); ext_to_aff(S, &P, &e); aff_store(S, out64, &P);
}
void orc_secret_from_seed(int s, const uint8_t seed[32], uint8_t sk32[32]) {                   /* lib.rs:346-369 */
  const sctx* S = suite(s); fe sk0, k; fr_from_le(&S->Fr, &sk0, seed, 32);
  for (int cnt = 0;; cnt++) {
    tr_t t; tr_new(&t, S->P->suite_id, S->P->sid_len); tr_absorb(&t, seed, 32); if (cnt) tr_absorb_u8(&t, (uint8_t)cnt);
    nonce(S, &k, &sk0, &t); if (!f_is_zero(&k)) break;
  }
  memcpy(sk32, k.v, 32);
}
void orc_point_to_hash(int s, const uint8_t in64[64], uint8_t out32[32]) {                      /* common.rs:290-305 */
  const sctx* S = suite(s); aff P; uint8_t e[32]; aff_load(S, &P, in64); aff_enc(S, e, &P);
  tr_t t; tr_new(&t, S->P->suite_id, S->P->sid_len); tr_absorb_u8(&t, 0x20); tr_absorb(&t, e, 32); tr_squeeze(&t, out32, 32);
}

#define MAX_IOS 64
static void merged_input(const sctx* S, ext* im, const aff* ios, const fe* zs, int m) {   /* I_m = G + sum z_i I_i */
  ext_from_aff(S, im, &S->G);
  for (int i = 0; i < m; i++) { ext e; ext_from_aff(S, &e, &ios[2 * i]); ext_mul(S, &e, &e, zs[i].v); ext_add(S, im, im, &e); }
}

/* thin::Prover::prove (src/thin.rs:111-129) */
int orc_thin_prove(int s, const uint8_t sk32[32], const uint8_t* ios128, int m, const uint8_t* ad, size_t ad_len, uint8_t r64[64], uint8_t s32[32]) {
  const sctx* S = suite(s); if (!S || m > MAX_IOS) return -1;
  fe sk, zs[MAX_IOS], k, c, skm, cs; memcpy(sk.v, sk32, 32);
  aff pk, ios[2 * MAX_IOS], R; ext e;
  memset(ios, 0, sizeof ios);
  ext_from_aff(S, &e, &S->G); ext_mul(S, &e, &e, sk.v); ext_to_aff(S, &pk, &e);
  for (int i = 0; i < 2 * m; i++) aff_load(S, &ios[i], ios128 + 64 * i);
  tr_t t; thin_transcript(S, &t, zs, &pk, ios, m, ad, ad_len);
  ext im; merged_input(S, &im, ios, zs, m);
  nonce(S, &k, &sk, &t);
  ext_mul(S, &e, &im, k.v); ext_to_aff(S, &R, &e);
  challenge(S, &t, &R, &c);
  f_to_mont(&S->Fr, &skm, &sk); f_mul(&S->Fr, &cs, &c, &skm); f_add(&S->Fr, &cs, &cs, &k);
  aff_store(S, r64, &R); memcpy(s32, cs.v, 32); return 0;
}

/* thin::Verifier::verify (src/thin.rs:131-165) */
int orc_thin_verify(int s, const uint8_t pk64[64], const uint8_t* ios128, int m, const uint8_t* ad, size_t ad_len, const uint8_t r64[64], const uint8_t s32[32]) {
  const sctx* S = suite(s); if (!S || m > MAX_IOS) return -1;
  aff pk, ios[2 * MAX_IOS], R; fe zs[MAX_IOS], c, sv; memcpy(sv.v, s32, 32);
  memset(ios, 0, sizeof ios);
  aff_load(S, &pk, pk64); aff_load(S, &R, r64);
  if (aff_is_id(S, &pk)) return ORC_INVALID_DATA;
  for (int i = 0; i < 2 * m; i++) { aff_load(S, &ios[i], ios128 + 64 * i); if (aff_is_id(S, &ios[i])) return ORC_INVALID_DATA; }
  tr_t t; thin_transcript(S, &t, zs, &pk, ios, m, ad, ad_len);
  ext im, om, e; merged_input(S, &im, ios, zs, m);
  ext_from_aff(S, &om, &pk);
  for (int i = 0; i < m; i++) { ext_from_aff(S, &e, &ios[2 * i + 1]); ext_mul(S, &e, &e, zs[i].v); ext_add(S, &om, &om, &e); }
  challenge(S, &t, &R, &c);
  ext lhs, rhs; ext_mul(S, &lhs, &im, sv.v); ext_mul(S, &rhs, &om, c.v); ext_neg(S, &rhs, &rhs); ext_add(S, &lhs, &lhs, &rhs);
  ext_from_aff(S, &e, &R); ext_neg(S, &e, &e); ext_add(S, &lhs, &lhs, &e);
  return ext_is_id(&lhs) ? ORC_OK : ORC_VERIFICATION_FAILURE;
}

/* ---- batch verification (src/thin.rs:209-325) ---------------------------------------- */
typedef struct {
  const sctx* S; size_t n; const uint8_t *pk, *ios, *ad, *r, *s; const uint32_t *io_off, *ad_off;
  aff* bases; fe* scalars;            /* MSM terms, order of thin.rs:291-312, then G */
  fe* c; fe* z;                       /* per proof c; per pair z */
  int invalid; size_t lo, hi;
} prep_job;

static void* prepare_worker(void* arg) {                                 /* BatchVerifier::prepare, thin.rs:209-226 */
  prep_job* j = (prep_job*)arg; const sctx* S = j->S;
  for (size_t i = j->lo; i < j->hi; i++) {
    uint32_t io0 = j->io_off[i], m = j->io_off[i + 1] - io0; size_t pb = 2 * i + 2 * (size_t)io0;
    aff pk, R, ios[2 * MAX_IOS]; fe zs[MAX_IOS];
    aff_load(S, &pk, j->pk + 64 * i); aff_load(S, &R, j->r + 64 * i);
    if (aff_is_id(S, &pk)) j->invalid = 1;
    for (uint32_t q = 0; q < 2 * m; q++) { aff_load(S, &ios[q], j->ios + 128 * (size_t)io0 + 64 * q); if (aff_is_id(S, &ios[q])) j->invalid = 1; }
    tr_t t; thin_transcript(S, &t, zs, &pk, ios, (int)m, j->ad + j->ad_off[i], j->ad_off[i + 1] - j->ad_off[i]);
    challenge(S, &t, &R, &j->c[i]);
    j->bases[pb] = R; j->bases[pb + 1] = pk;
    for (uint32_t q = 0; q < m; q++) { j->bases[pb + 2 + 2 * q] = ios[2 * q + 1]; j->bases[pb + 3 + 2 * q] = ios[2 * q]; j->z[io0 + q] = zs[q]; }
  }
  return NULL;
}

/* ark-ec 0.6 VariableBaseMSM::msm_bigint_wnaf restated: signed digits of width c, one job per window */
typedef struct { const sctx* S; const aff* bases; const int32_t* digits; size_t n; int nwin, c, w0, w1; ext* wsum; } win_job;
static void* window_worker(void* arg) {
  win_job* j = (win_job*)arg; const sctx* S = j->S; size_t nb = (size_t)1 << (j->c - 1);
  ext* buckets = (ext*)malloc(nb * sizeof(ext));
  for (int w = j->w0; w < j->w1; w++) {
    for (size_t b = 0; b < nb; b++) ext_id(S, &buckets[b]);
    for (size_t i = 0; i < j->n; i++) {
      int32_t d = j->digits[i * j->nwin + w];
      if (d > 0) ext_madd(S, &buckets[d - 1], &buckets[d - 1], &j->bases[i], 0);
      else if (d < 0) ext_madd(S, &buckets[-d - 1], &buckets[-d - 1], &j->bases[i], 1);
    }
    ext run, acc; ext_id(S, &run); ext_id(S, &acc);
    for (size_t b = nb; b-- > 0;) { ext_add(S, &run, &run, &buckets[b]); ext_add(S, &acc, &acc, &run); }
    j->wsum[w] = acc;
  }
  free(buckets); return NULL;
}
/* `bits`: scalar width the windows must cover (ark-ec: the scalar field's MODULUS_BIT_SIZE); the last window's
 * signed digit absorbs the final carry as long as every scalar is below 2^bits. */
static void msm(const sctx* S, ext* out, const aff* bases, const fe* scalars, size_t n, int bits, int nthreads) {
  int c = n < 32 ? 3 : (int)(log((double)n)) + 2;                         /* ark-ec ln_without_floats(n) + 2 */
  int nwin = (bits + c - 1) / c + 1;
  int32_t* digits = (int32_t*)malloc(n * (size_t)nwin * sizeof(int32_t));
  for (size_t i = 0; i < n; i++) {                                        /* make_digits: signed radix 2^c */
    u64 carry = 0; const u64* k = scalars[i].v;
    for (int w = 0; w < nwin; w++) {
      int bit = w * c; u64 v = 0;
      if (bit < 256) { v = k[bit >> 6] >> (bit & 63); if ((bit & 63) + c > 64 && (bit >> 6) < 3) v |= k[(bit >> 6) + 1] << (64 - (bit & 63)); v &= ((u64)1 << c) - 1; }
      v += carry; carry = (v + ((u64)1 << (c - 1))) >> c;
      digits[i * nwin + w] = (int32_t)((int64_t)v - (int64_t)(carry << c));
    }
  }
  ext* wsum = (ext*)malloc(nwin * sizeof(ext));
  if (nthreads > nwin) nthreads = nwin; if (nthreads < 1) nthreads = 1;
  pthread_t th[256]; win_job jobs[256]; if (nthreads > 256) nthreads = 256;
  for (int t = 0; t < nthreads; t++) {
    jobs[t] = (win_job){S, bases, digits, n, nwin, c, (int)((long)nwin * t / nthreads), (int)((long)nwin * (t + 1) / nthreads), wsum};
    pthread_create(&th[t], NULL, window_worker, &jobs[t]);
  }
  for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
  ext acc = wsum[nwin - 1];
  for (int w = nwin - 2; w >= 0; w--) { for (int i = 0; i < c; i++) ext_dbl(S, &acc, &acc); ext_add(S, &acc, &acc, &wsum[w]); }
  *out = acc; free(wsum); free(digits);
}

static double now_s(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + 1e-9 * ts.tv_nsec; }

/* BatchVerifier::push x n then verify.  taps (each may be NULL): c16 (16 B/proof), z16 (16 B/pair), seed64, w16
 * (16 B/proof), scalars32 (32 B/term).  times[0] = prepare seconds, times[1] = verify seconds. */
int orc_thin_batch_verify(int s, size_t n, const uint8_t* pk, const uint8_t* ios, const uint32_t* io_off, const uint8_t* ad,
                          const uint32_t* ad_off, const uint8_t* r, const uint8_t* sv, int nthreads, double* times,
                          uint8_t* c16, uint8_t* z16, uint8_t* seed64, uint8_t* w16, uint8_t* scalars32) {
  const sctx* S = suite(s); if (!S) return -1;
  if (n == 0) return ORC_OK;                                              /* thin.rs:262-264 */
  if (nthreads < 1) nthreads = 1; if (nthreads > 256) nthreads = 256;
  size_t nio = io_off[n], np = 2 * n + 2 * nio + 1;
  aff* bases = (aff*)malloc(np * sizeof(aff)); fe* scalars = (fe*)malloc(np * sizeof(fe));
  fe* c = (fe*)malloc(n * sizeof(fe)); fe* z = (fe*)malloc((nio + 1) * sizeof(fe));
  double t0 = now_s();
  pthread_t th[256]; prep_job jobs[256];
  for (int t = 0; t < nthreads; t++) {
    jobs[t] = (prep_job){S, n, pk, ios, ad, r, sv, io_off, ad_off, bases, scalars, c, z, 0, n * t / nthreads, n * (t + 1) / nthreads};
    pthread_create(&th[t], NULL, prepare_worker, &jobs[t]);
  }
  int invalid = 0;
  for (int t = 0; t < nthreads; t++) { pthread_join(th[t], NULL); invalid |= jobs[t].invalid; }
  double t1 = now_s();
  int status;
  if (c16) for (size_t i = 0; i < n; i++) memcpy(c16 + 16 * i, c[i].v, 16);
  if (z16) for (size_t i = 0; i < nio; i++) memcpy(z16 + 16 * i, z[i].v, 16);
  if (invalid) { status = ORC_INVALID_DATA; goto done; }                  /* thin.rs:266-271 */
  {
    tr_t t; tr_new(&t, S->P->suite_id, S->P->sid_len); tr_absorb_u8(&t, 0x50);                 /* thin.rs:274-279 */
    for (size_t i = 0; i < n; i++) { tr_absorb(&t, c[i].v, 32); tr_absorb(&t, sv + 32 * i, 32); }
    const fctx* F = &S->Fr; fe g; memset(&g, 0, sizeof g);
    for (size_t i = 0; i < n; i++) {                                                           /* thin.rs:287-313 */
      fe w, wm, wc, ws, sc; challenge_scalar(S, &t, &w);
      if (i == 0 && seed64) memcpy(seed64, t.seed, 64);
      if (w16) memcpy(w16 + 16 * i, w.v, 16);
      memcpy(sc.v, sv + 32 * i, 32);
      f_to_mont(F, &wm, &w); f_mul(F, &wc, &wm, &c[i]); f_mul(F, &ws, &wm, &sc);
      uint32_t io0 = io_off[i], m = io_off[i + 1] - io0; size_t pb = 2 * i + 2 * (size_t)io0;
      scalars[pb] = w; scalars[pb + 1] = wc; f_sub(F, &g, &g, &ws);
      for (uint32_t q = 0; q < m; q++) {
        fe zm, a; f_to_mont(F, &zm, &z[io0 + q]);
        f_mul(F, &scalars[pb + 2 + 2 * q], &wc, &zm); f_mul(F, &a, &ws, &zm); f_neg(F, &scalars[pb + 3 + 2 * q], &a);
      }
    }
    bases[np - 1] = S->G; scalars[np - 1] = g;                                                 /* thin.rs:315-317 */
    if (scalars32) memcpy(scalars32, scalars, 32 * np);
    ext res; msm(S, &res, bases, scalars, np, S->Fr.bits, nthreads);                           /* thin.rs:319 */
    status = ext_is_id(&res) ? ORC_OK : ORC_VERIFICATION_FAILURE;                              /* thin.rs:320-324 */
  }
done:
  if (times) { times[0] = t1 - t0; times[1] = now_s() - t1; }
  free(bases); free(scalars); free(c); free(z);
  return status;
}

/* sum_i k_i * P_i by the same msm() the batch verifier runs, for checking another MSM against it.  bases64: n canonical
 * affine points (any curve point: nothing is reduced into the subgroup); scalars32: n canonical little-endian integers,
 * any value below 2^256, used as they are (not reduced mod r, so a small-order component of a base keeps the exact
 * residue of its scalar).  out64: the canonical affine sum.  Returns 1 if the sum is the identity, 0 if not, -1 on a
 * bad suite. */
int orc_msm(int s, size_t n, const uint8_t* bases64, const uint8_t* scalars32, int nthreads, uint8_t out64[64]) {
  const sctx* S = suite(s); if (!S) return -1;
  ext res; ext_id(S, &res);
  if (n) {
    aff* bases = (aff*)malloc(n * sizeof(aff)); fe* scalars = (fe*)malloc(n * sizeof(fe));
    for (size_t i = 0; i < n; i++) { aff_load(S, &bases[i], bases64 + 64 * i); memcpy(scalars[i].v, scalars32 + 32 * i, 32); }
    msm(S, &res, bases, scalars, n, 256, nthreads < 1 ? 1 : nthreads);
    free(bases); free(scalars);
  }
  aff P; ext_to_aff(S, &P, &res); aff_store(S, out64, &P);
  return ext_is_id(&res);
}

/* ---- synthetic workload of SURVEY.md section 8(d), generated with the restated prover ----
 * signer k: sk = Secret::from_seed(LE64(k) || 0^24); proof j signed by k = j mod K;
 * I_{j,i} = data_to_point(LE64(j) || LE32(i)); O = sk * I; ad_j = "ad-<j>"; deterministic prove. */
typedef struct { int s; size_t first, lo, hi; int m, K; const uint8_t* sks; const uint8_t* pks; uint8_t *pk, *ios, *r, *sv; } synth_job;
static void* synth_worker(void* arg) {
  synth_job* j = (synth_job*)arg; const sctx* S = suite(j->s);
  for (size_t q = j->lo; q < j->hi; q++) {
    size_t idx = j->first + q; int k = (int)(idx % (size_t)j->K);
    memcpy(j->pk + 64 * q, j->pks + 64 * k, 64);
    for (int i = 0; i < j->m; i++) {
      uint8_t msg[12]; for (int b = 0; b < 8; b++) msg[b] = (uint8_t)((u64)idx >> (8 * b)); for (int b = 0; b < 4; b++) msg[8 + b] = (uint8_t)((uint32_t)i >> (8 * b));
      aff P; data_to_point(S, &P, msg, 12);
      uint8_t* io = j->ios + 128 * (q * j->m + i);
      aff_store(S, io, &P); orc_scalar_mul(j->s, j->sks + 32 * k, io, io + 64);
    }
    char ad[32]; int al = 0; { char tmp[24]; size_t v = idx; int n = 0; do { tmp[n++] = (char)('0' + v % 10); v /= 10; } while (v); ad[0] = 'a'; ad[1] = 'd'; ad[2] = '-'; al = 3; while (n) ad[al++] = tmp[--n]; }
    orc_thin_prove(j->s, j->sks + 32 * k, j->ios + 128 * q * j->m, j->m, (const uint8_t*)ad, (size_t)al, j->r + 64 * q, j->sv + 32 * q);
  }
  return NULL;
}
/* Outputs: pk (64n), ios (128 n m), r (64n), s (32n), all canonical.  ad_j is "ad-<first+j>" (caller rebuilds offsets). */
int orc_synth_batch(int s, size_t first, size_t n, int m, int signers, int nthreads, uint8_t* pk, uint8_t* ios, uint8_t* r, uint8_t* sv) {
  if (!suite(s) || m > MAX_IOS) return -1;
  int K = signers < 1 ? 1 : signers;
  uint8_t* sks = (uint8_t*)malloc(32 * (size_t)K); uint8_t* pks = (uint8_t*)malloc(64 * (size_t)K);
  for (int k = 0; k < K; k++) { uint8_t seed[32] = {0}; for (int b = 0; b < 8; b++) seed[b] = (uint8_t)((u64)k >> (8 * b)); orc_secret_from_seed(s, seed, sks + 32 * k); orc_scalar_mul(s, sks + 32 * k, NULL, pks + 64 * k); }
  if (nthreads < 1) nthreads = 1; if (nthreads > 256) nthreads = 256;
  pthread_t th[256]; synth_job jobs[256];
  for (int t = 0; t < nthreads; t++) { jobs[t] = (synth_job){s, first, n * t / nthreads, n * (t + 1) / nthreads, m, K, sks, pks, pk, ios, r, sv}; pthread_create(&th[t], NULL, synth_worker, &jobs[t]); }
  for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
  free(sks); free(pks); return 0;
}
