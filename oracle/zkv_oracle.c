/* ORACLE -- TEST INFRASTRUCTURE ONLY (checker + CPU baseline; never shipped, never on the product path).
 *
 * CPU restatement of the reference verification path, one function per reference item:
 *   zkvo_ec_add / zkvo_ec_mul / zkvo_ec_pairing   EVM precompiles 0x06/0x07/0x08 as the reference
 *        calls them (contracts/src/common/groth16.rs:60-73, 109-128); EIP-196/197 byte semantics.
 *   groth16_verify            contracts/src/common/groth16.rs:23-49 (+ compute_vk_x :51-58,
 *                             negate_g1 :75-84, verify_pairing :86-107)
 *   zkvo_risc0_*              contracts/src/risc0/verifier.rs:58-76,78-104,128-197;
 *                             risc0/types.rs:44-95; risc0/crypto.rs:95-195
 *   zkvo_sp1_*                contracts/src/sp1/verifier.rs:58-111; sp1/types.rs:21-38
 * The reference's Rust cannot be built here (no cargo/rustc; BN254 lives in node-side precompiles),
 * so this file is a "port" baseline.  Pinned by: the two fixtures in examples/.../interact.rs
 * (tests/golden/reference_constants.json), the SURVEY section 4 known answers, and the independent
 * Python referee oracle/pyref/bn254_py.py.
 */
#include <stdio.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif
#include "bn254.h"

/* ------------------------------------------------------------------ SHA-256 (FIPS 180-4) */
static const uint32_t SHA_K[64] = {
    0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01, 0x243185be,
    0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa,
    0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967, 0x27b70a85,
    0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85, 0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3,
    0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f,
    0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};
#define ROR(x, n) (((x) >> (n)) | ((x) << (32 - (n))))
static void sha_block(uint32_t h[8], const uint8_t *blk) {
    uint32_t w[64];
    for (int i = 0; i < 16; i++) w[i] = (uint32_t)blk[4 * i] << 24 | (uint32_t)blk[4 * i + 1] << 16 | (uint32_t)blk[4 * i + 2] << 8 | blk[4 * i + 3];
    for (int i = 16; i < 64; i++) {
        uint32_t s0 = ROR(w[i - 15], 7) ^ ROR(w[i - 15], 18) ^ (w[i - 15] >> 3), s1 = ROR(w[i - 2], 17) ^ ROR(w[i - 2], 19) ^ (w[i - 2] >> 10);
        w[i] = w[i - 16] + s0 + w[i - 7] + s1;
    }
    uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
    for (int i = 0; i < 64; i++) {
        uint32_t t1 = hh + (ROR(e, 6) ^ ROR(e, 11) ^ ROR(e, 25)) + ((e & f) ^ (~e & g)) + SHA_K[i] + w[i];
        uint32_t t2 = (ROR(a, 2) ^ ROR(a, 13) ^ ROR(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
        hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
    }
    h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
}
static void sha256(uint8_t out[32], const uint8_t *msg, size_t len) {
    uint32_t h[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    size_t i = 0;
    for (; i + 64 <= len; i += 64) sha_block(h, msg + i);
    uint8_t tail[128]; size_t rem = len - i; memset(tail, 0, sizeof tail); memcpy(tail, msg + i, rem);
    tail[rem] = 0x80; size_t tl = (rem + 9 <= 64) ? 64 : 128; uint64_t bits = (uint64_t)len * 8;
    for (int k = 0; k < 8; k++) tail[tl - 1 - k] = (uint8_t)(bits >> (8 * k));
    sha_block(h, tail); if (tl == 128) sha_block(h, tail + 64);
    for (int k = 0; k < 8; k++) { out[4 * k] = h[k] >> 24; out[4 * k + 1] = h[k] >> 16; out[4 * k + 2] = h[k] >> 8; out[4 * k + 3] = h[k]; }
}

/* ------------------------------------------------------------------ EIP-196/197 decoding */
static int dec_g1(g1a *p, const uint8_t *b) {
    uint64_t x[4], y[4]; be32_to_limbs(x, b); be32_to_limbs(y, b + 32);
    if (limbs_geq(x, FP_P) || limbs_geq(y, FP_P)) return -1;
    if (!(x[0] | x[1] | x[2] | x[3] | y[0] | y[1] | y[2] | y[3])) { p->inf = 1; p->x = FP_ZERO; p->y = FP_ZERO; return 0; }
    fp_from_limbs(&p->x, x); fp_from_limbs(&p->y, y); p->inf = 0;
    return g1_on_curve(&p->x, &p->y) ? 0 : -1;
}
static void enc_g1(uint8_t *b, const g1a *p) {
    if (p->inf) { memset(b, 0, 64); return; }
    fp_to_be32(b, &p->x); fp_to_be32(b + 32, &p->y);
}
/* G2 wire order: x_im, x_re, y_im, y_re (SURVEY section 4; groth16.rs:115-118 emits x[0],x[1],y[0],y[1]) */
static int dec_g2(g2a *q, const uint8_t *b) {
    uint64_t v[4][4]; uint64_t any = 0;
    for (int i = 0; i < 4; i++) { be32_to_limbs(v[i], b + 32 * i); if (limbs_geq(v[i], FP_P)) return -1; any |= v[i][0] | v[i][1] | v[i][2] | v[i][3]; }
    if (!any) { q->inf = 1; q->x = F2_ZERO; q->y = F2_ZERO; return 0; }
    fp_from_limbs(&q->x.c1, v[0]); fp_from_limbs(&q->x.c0, v[1]); fp_from_limbs(&q->y.c1, v[2]); fp_from_limbs(&q->y.c0, v[3]); q->inf = 0;
    if (!g2_on_curve(&q->x, &q->y)) return -1;
    return g2_in_subgroup(q) ? 0 : -1;
}
static void enc_g2(uint8_t *b, const g2a *q) {
    if (q->inf) { memset(b, 0, 128); return; }
    fp_to_be32(b, &q->x.c1); fp_to_be32(b + 32, &q->x.c0); fp_to_be32(b + 64, &q->y.c1); fp_to_be32(b + 96, &q->y.c0);
}

/* precompile 0x06: 0 = ok, -1 = call reverted */
int zkvo_ec_add(const uint8_t *in, size_t len, uint8_t out[64]) {
    bn254_init();
    uint8_t buf[128]; memset(buf, 0, 128); memcpy(buf, in, len < 128 ? len : 128);
    g1a a, b; if (dec_g1(&a, buf) || dec_g1(&b, buf + 64)) return -1;
    g1j ja, jb, jr; g1_from_affine(&ja, &a); g1_from_affine(&jb, &b); g1_add(&jr, &ja, &jb);
    g1a r; g1_to_affine(&r, &jr); enc_g1(out, &r); return 0;
}
/* precompile 0x07 */
int zkvo_ec_mul(const uint8_t *in, size_t len, uint8_t out[64]) {
    bn254_init();
    uint8_t buf[96]; memset(buf, 0, 96); memcpy(buf, in, len < 96 ? len : 96);
    g1a a; if (dec_g1(&a, buf)) return -1;
    uint64_t k[4]; be32_to_limbs(k, buf + 64);
    g1j ja, jr; g1_from_affine(&ja, &a); g1_mul(&jr, &ja, k);
    g1a r; g1_to_affine(&r, &jr); enc_g1(out, &r); return 0;
}
/* precompile 0x08; optionally exports the Miller value and GT (384 B each) for parity tests */
static int ec_pairing_ex(const uint8_t *in, size_t len, uint8_t out[32], uint8_t *miller_out, uint8_t *gt_out) {
    bn254_init();
    if (len % 192) return -1;
    int n = (int)(len / 192); if (n > ORACLE_MAX_PAIRS) return -2;
    pair_t pr[ORACLE_MAX_PAIRS];
    for (int i = 0; i < n; i++) if (dec_g1(&pr[i].p, in + 192 * i) || dec_g2(&pr[i].q, in + 192 * i + 64)) return -1;
    fp12 m, gt; miller_multi(&m, pr, n); final_exp(&gt, &m);
    memset(out, 0, 32); out[31] = f12_eq(&gt, &F12_ONE) ? 1 : 0;
    if (miller_out) f12_to_bytes(miller_out, &m);
    if (gt_out) f12_to_bytes(gt_out, &gt);
    return 0;
}
int zkvo_ec_pairing(const uint8_t *in, size_t len, uint8_t out[32]) { return ec_pairing_ex(in, len, out, NULL, NULL); }
int zkvo_ec_pairing_debug(const uint8_t *in, size_t len, uint8_t out[32], uint8_t *miller_out, uint8_t *gt_out) { return ec_pairing_ex(in, len, out, miller_out, gt_out); }
int zkvo_final_exp(const uint8_t in[384], uint8_t out[384]) {
    bn254_init(); fp12 m, gt; if (f12_from_bytes(&m, in)) return -1; final_exp(&gt, &m); f12_to_bytes(out, &gt); return 0;
}
/* Fp12 helpers for the test-suite (values are 12 x BE-32 in tower order) */
int zkvo_fp12_mul(const uint8_t a[384], const uint8_t b[384], uint8_t out[384]) {
    bn254_init(); fp12 x, y, z; if (f12_from_bytes(&x, a) || f12_from_bytes(&y, b)) return -1; f12_mul(&z, &x, &y); f12_to_bytes(out, &z); return 0;
}
int zkvo_fp12_cyc_sqr(const uint8_t a[384], uint8_t out[384]) {
    bn254_init(); fp12 x, z; if (f12_from_bytes(&x, a)) return -1; f12_cyc_sqr(&z, &x); f12_to_bytes(out, &z); return 0;
}
int zkvo_fp_mul(const uint8_t a[32], const uint8_t b[32], uint8_t out[32]) {   /* plain (non-Montgomery) a*b mod p */
    bn254_init(); uint64_t x[4], y[4]; be32_to_limbs(x, a); be32_to_limbs(y, b); fp fx, fy, fz; fp_from_limbs(&fx, x); fp_from_limbs(&fy, y); fp_mul(&fz, &fx, &fy); fp_to_be32(out, &fz); return 0;
}
int zkvo_ate_naf(int8_t *out, int cap) { bn254_init(); if (cap < ATE_NAF_LEN) return -1; memcpy(out, ATE_NAF, ATE_NAF_LEN); return ATE_NAF_LEN; }

/* test-data helpers (synthetic proof generation): unchecked scalar multiples */
int zkvo_g1_mul(const uint8_t pt[64], const uint8_t k[32], uint8_t out[64]) {
    uint8_t buf[96]; memcpy(buf, pt, 64); memcpy(buf + 64, k, 32); return zkvo_ec_mul(buf, 96, out);
}
int zkvo_g2_mul(const uint8_t pt[128], const uint8_t k[32], uint8_t out[128]) {  /* on-twist check only: also used to build wrong-subgroup points */
    bn254_init();
    uint64_t v[4][4]; for (int i = 0; i < 4; i++) { be32_to_limbs(v[i], pt + 32 * i); if (limbs_geq(v[i], FP_P)) return -1; }
    g2a q; fp_from_limbs(&q.x.c1, v[0]); fp_from_limbs(&q.x.c0, v[1]); fp_from_limbs(&q.y.c1, v[2]); fp_from_limbs(&q.y.c0, v[3]); q.inf = 0;
    if (!g2_on_curve(&q.x, &q.y)) return -1;
    uint64_t s[4]; be32_to_limbs(s, k);
    g2j j, r; j.x = q.x; j.y = q.y; j.z = F2_ONE; g2_mul(&r, &j, s);
    g2a a; g2_to_affine(&a, &r); enc_g2(out, &a); return 0;
}
int zkvo_g2_add(const uint8_t a[128], const uint8_t b[128], uint8_t out[128]) {  /* no subgroup check */
    bn254_init(); g2j ja, jb, jr; g2a q;
    const uint8_t *src[2] = {a, b}; g2j *dst[2] = {&ja, &jb};
    for (int s = 0; s < 2; s++) {
        uint64_t v[4][4]; uint64_t any = 0; for (int i = 0; i < 4; i++) { be32_to_limbs(v[i], src[s] + 32 * i); any |= v[i][0] | v[i][1] | v[i][2] | v[i][3]; }
        if (!any) { dst[s]->x = F2_ONE; dst[s]->y = F2_ONE; dst[s]->z = F2_ZERO; continue; }
        fp_from_limbs(&dst[s]->x.c1, v[0]); fp_from_limbs(&dst[s]->x.c0, v[1]); fp_from_limbs(&dst[s]->y.c1, v[2]); fp_from_limbs(&dst[s]->y.c0, v[3]); dst[s]->z = F2_ONE;
    }
    g2_add(&jr, &ja, &jb); g2_to_affine(&q, &jr); enc_g2(out, &q); return 0;
}
/* y = sqrt(x^3 + b') on the twist for building arbitrary (mostly wrong-subgroup) twist points; returns -1 if no root */
int zkvo_g2_from_x(const uint8_t x_im_re[64], uint8_t out[128]) {
    bn254_init();
    uint64_t v0[4], v1[4]; be32_to_limbs(v0, x_im_re); be32_to_limbs(v1, x_im_re + 32);
    if (limbs_geq(v0, FP_P) || limbs_geq(v1, FP_P)) return -1;
    fp2 x, rhs, y; fp_from_limbs(&x.c1, v0); fp_from_limbs(&x.c0, v1);
    f2_sqr(&rhs, &x); f2_mul(&rhs, &rhs, &x); f2_add(&rhs, &rhs, &TWIST_B);
    /* sqrt in Fp2, p = 3 mod 4 (Adj-Rodriguez-Henriquez alg. 9) */
    uint64_t e1[4], e2[4];  /* (p-3)/4, (p-1)/2 */
    { uint64_t t[4]; memcpy(t, FP_P, 32); t[0] -= 3; for (int i = 0; i < 4; i++) e1[i] = (t[i] >> 2) | (i < 3 ? t[i + 1] << 62 : 0);
      memcpy(t, FP_P, 32); t[0] -= 1; for (int i = 0; i < 4; i++) e2[i] = (t[i] >> 1) | (i < 3 ? t[i + 1] << 63 : 0); }
    fp2 a1, alpha, a0, x0, t;
    f2_pow(&a1, &rhs, e1, 4); f2_sqr(&alpha, &a1); f2_mul(&alpha, &alpha, &rhs);
    f2_conj(&t, &alpha); f2_mul(&a0, &t, &alpha);
    fp2 m1; fp_neg(&m1.c0, &FP_ONE); m1.c1 = FP_ZERO;
    if (f2_eq(&a0, &m1)) return -1;
    f2_mul(&x0, &a1, &rhs);
    if (f2_eq(&alpha, &m1)) { fp2 i_; i_.c0 = FP_ZERO; i_.c1 = FP_ONE; f2_mul(&y, &i_, &x0); }
    else { fp2 b; f2_add(&b, &F2_ONE, &alpha); f2_pow(&b, &b, e2, 4); f2_mul(&y, &b, &x0); }
    f2_sqr(&t, &y); if (!f2_eq(&t, &rhs)) return -1;
    g2a q; q.x = x; q.y = y; q.inf = 0; enc_g2(out, &q); return 0;
}

/* ------------------------------------------------------------------ Groth16 driver (groth16.rs:23-49) */
typedef struct {
    int vm;                 /* 0 = Risc0, 1 = Sp1   (common/types.rs:25-26) */
    int n_ic;
    uint8_t alpha[64], beta[128], gamma[128], delta[128];
    uint8_t ic[16 * 64];
} vk_t;

static int u256_geq_r(const uint8_t *be) { uint64_t v[4]; be32_to_limbs(v, be); return limbs_geq(v, FR_R); }

/* proof = 8 x BE-32 (a0,a1,b00,b01,b10,b11,c0,c1); signals = k x BE-32.  Returns 1 = true, 0 = false. */
static int groth16_verify(const vk_t *vk, const uint8_t *proof, const uint8_t *signals, int k, uint8_t *miller_out, uint8_t *gt_out) {
    if (k + 1 != vk->n_ic) return 0;                                   /* groth16.rs:32 */
    for (int i = 0; i < k; i++) if (u256_geq_r(signals + 32 * i)) return 0;
    uint8_t vkx[64], mul_in[96], add_in[128], mul_out[64];             /* compute_vk_x, groth16.rs:51-58 */
    memcpy(vkx, vk->ic, 64);
    for (int i = 0; i < k; i++) {
        memcpy(mul_in, vk->ic + 64 * (i + 1), 64); memcpy(mul_in + 64, signals + 32 * i, 32);
        if (zkvo_ec_mul(mul_in, 96, mul_out)) return 0;
        memcpy(add_in, vkx, 64); memcpy(add_in + 64, mul_out, 64);
        if (zkvo_ec_add(add_in, 128, vkx)) return 0;
    }
    uint8_t a[64]; memcpy(a, proof, 64);
    if (vk->vm == 0) {                                                 /* negate_g1, groth16.rs:75-84: Q.wrapping_sub(y) mod 2^256 */
        int zero = 1; for (int i = 0; i < 64; i++) if (a[i]) zero = 0;
        if (!zero) { uint64_t y[4], r[4]; be32_to_limbs(y, a + 32); limbs_sub(r, FP_P, y); limbs_to_be32(a + 32, r); }
    }
    uint8_t cd[768];                                                   /* pairing_check calldata, groth16.rs:110-119 */
    memcpy(cd, a, 64);              memcpy(cd + 64, proof + 64, 128);
    memcpy(cd + 192, vk->alpha, 64); memcpy(cd + 256, vk->beta, 128);
    memcpy(cd + 384, vkx, 64);      memcpy(cd + 448, vk->gamma, 128);
    memcpy(cd + 576, proof + 192, 64); memcpy(cd + 640, vk->delta, 128);
    uint8_t ret[32];
    if (ec_pairing_ex(cd, 768, ret, miller_out, gt_out)) return 0;     /* unwrap_or(false), groth16.rs:106 */
    for (int i = 0; i < 32; i++) if (ret[i]) return 1;
    return 0;
}

/* status vocabulary shared with include/zkv.h (SURVEY section 8b) */
enum { ST_OK = 0, ST_INVALID_INITIALIZATION = 1, ST_INVALID_PROOF_DATA = 2, ST_SELECTOR_MISMATCH = 3, ST_VERIFICATION_FAILED = 4 };

void zkvo_vk_pack(vk_t *vk, int vm, const uint8_t *alpha, const uint8_t *beta, const uint8_t *gamma, const uint8_t *delta, const uint8_t *ic, int n_ic) {
    vk->vm = vm; vk->n_ic = n_ic; memcpy(vk->alpha, alpha, 64); memcpy(vk->beta, beta, 128); memcpy(vk->gamma, gamma, 128); memcpy(vk->delta, delta, 128);
    memcpy(vk->ic, ic, 64 * (size_t)n_ic);
}
size_t zkvo_vk_sizeof(void) { return sizeof(vk_t); }

int zkvo_groth16_verify(const vk_t *vk, const uint8_t *proof, const uint8_t *signals, int k) {
    bn254_init(); return groth16_verify(vk, proof, signals, k, NULL, NULL) ? ST_OK : ST_VERIFICATION_FAILED;
}
int zkvo_groth16_verify_debug(const vk_t *vk, const uint8_t *proof, const uint8_t *signals, int k, uint8_t *miller_out, uint8_t *gt_out) {
    bn254_init(); return groth16_verify(vk, proof, signals, k, miller_out, gt_out) ? ST_OK : ST_VERIFICATION_FAILED;
}
void zkvo_groth16_verify_batch(const vk_t *vk, const uint8_t *proofs, const uint8_t *signals, int k, long n, uint8_t *status) {
    bn254_init();
#pragma omp parallel for schedule(dynamic, 4)
    for (long i = 0; i < n; i++) status[i] = groth16_verify(vk, proofs + 256 * i, signals + 32 * (size_t)k * i, k, NULL, NULL) ? ST_OK : ST_VERIFICATION_FAILED;
}

/* ------------------------------------------------------------------ RISC Zero front-end */
static const uint8_t SYS0[32] = {0xa3, 0xac, 0xc2, 0x71, 0x17, 0x41, 0x89, 0x96, 0x34, 0x0b, 0x84, 0xe5, 0xa9, 0x0f, 0x3e, 0xf4,
                                 0xc4, 0x9d, 0x22, 0xc7, 0x9e, 0x44, 0xaa, 0xd8, 0x22, 0xec, 0x9c, 0x31, 0x3e, 0x1e, 0xb8, 0xe2};   /* risc0/config.rs:5-9 */
typedef struct {
    int initialized;
    uint8_t control_root_0[16], control_root_1[16], bn254_control_id[32], selector[4];  /* risc0/verifier.rs:44-52 */
    vk_t vk;
} risc0_t;

static void sha_str(uint8_t out[32], const char *s) { sha256(out, (const uint8_t *)s, strlen(s)); }
static void reverse32(uint8_t out[32], const uint8_t in[32]) { for (int i = 0; i < 32; i++) out[i] = in[31 - i]; }
static void split_digest(uint8_t lo[16], uint8_t hi[16], const uint8_t d[32]) {   /* risc0/crypto.rs:103-110 */
    uint8_t rev[32]; reverse32(rev, d); memcpy(lo, rev + 16, 16); memcpy(hi, rev, 16);
}
/* risc0/crypto.rs:136-195 (generalised to the instance's vk so that synthetic vks get a consistent selector) */
static void vk_digest(uint8_t out[32], const vk_t *vk) {
    uint8_t ic_tag[32], vk_tag[32], cur[32], buf[32 * 7 + 2];
    sha_str(ic_tag, "risc0_groth16.VerifyingKey.IC"); sha_str(vk_tag, "risc0_groth16.VerifyingKey");
    memset(cur, 0, 32);
    for (int i = vk->n_ic - 1; i >= 0; i--) {      /* tagged_list / tagged_list_cons :124-134 */
        memcpy(buf, ic_tag, 32); sha256(buf + 32, vk->ic + 64 * i, 64); memcpy(buf + 64, cur, 32); buf[96] = 0x02; buf[97] = 0x00;
        sha256(cur, buf, 98);
    }
    memcpy(buf, vk_tag, 32); sha256(buf + 32, vk->alpha, 64); sha256(buf + 64, vk->beta, 128); sha256(buf + 96, vk->gamma, 128); sha256(buf + 128, vk->delta, 128);
    memcpy(buf + 160, cur, 32); buf[192] = 0x05; buf[193] = 0x00;
    sha256(out, buf, 194);
}
static void claim_digest(uint8_t out[32], const uint8_t image_id[32], const uint8_t journal[32]) {   /* risc0/types.rs:44-95 */
    uint8_t buf[170], od[32];
    sha_str(buf, "risc0.Output"); memcpy(buf + 32, journal, 32); memset(buf + 64, 0, 32); buf[96] = 0x02; buf[97] = 0x00;
    sha256(od, buf, 98);
    sha_str(buf, "risc0.ReceiptClaim"); memset(buf + 32, 0, 32); memcpy(buf + 64, image_id, 32); memcpy(buf + 96, SYS0, 32); memcpy(buf + 128, od, 32);
    memset(buf + 160, 0, 8); buf[168] = 0x04; buf[169] = 0x00;
    sha256(out, buf, 170);
}
size_t zkvo_risc0_sizeof(void) { return sizeof(risc0_t); }
void zkvo_risc0_new(risc0_t *h, const vk_t *vk) { memset(h, 0, sizeof *h); h->vk = *vk; h->vk.vm = 0; }
/* initialize, risc0/verifier.rs:58-76 ; returns 0 or -1 = AlreadyInitialized */
int zkvo_risc0_initialize(risc0_t *h, const uint8_t control_root[32], const uint8_t bn254_control_id[32]) {
    if (h->initialized) return -1;
    split_digest(h->control_root_0, h->control_root_1, control_root);
    memcpy(h->bn254_control_id, bn254_control_id, 32);
    uint8_t buf[32 * 4 + 2], d[32];                                   /* calculate_selector :128-144 */
    sha_str(buf, "risc0.Groth16ReceiptVerifierParameters"); memcpy(buf + 32, control_root, 32); reverse32(buf + 64, bn254_control_id);
    vk_digest(buf + 96, &h->vk); buf[128] = 0x03; buf[129] = 0x00;
    sha256(d, buf, 130); memcpy(h->selector, d, 4);
    h->initialized = 1; return 0;
}
void zkvo_risc0_get_selector(const risc0_t *h, uint8_t out[4]) { memcpy(out, h->selector, 4); }
void zkvo_risc0_get_vk_digest(const risc0_t *h, uint8_t out[32]) { vk_digest(out, &h->vk); }
void zkvo_risc0_claim_digest(const uint8_t image_id[32], const uint8_t journal[32], uint8_t out[32]) { claim_digest(out, image_id, journal); }
void zkvo_risc0_signals(const risc0_t *h, const uint8_t claim[32], uint8_t out[160]) {               /* verifier.rs:172-179 */
    uint8_t lo[16], hi[16]; split_digest(lo, hi, claim); memset(out, 0, 160);
    memcpy(out + 16, h->control_root_0, 16); memcpy(out + 48, h->control_root_1, 16); memcpy(out + 80, lo, 16); memcpy(out + 112, hi, 16);
    memcpy(out + 128, h->bn254_control_id, 32);
}
/* verify_integrity_internal, risc0/verifier.rs:146-197 */
int zkvo_risc0_verify_integrity(const risc0_t *h, const uint8_t *seal, size_t seal_len, const uint8_t claim[32]) {
    bn254_init();
    if (!h->initialized) return ST_INVALID_INITIALIZATION;             /* :84-86 / :99-101 */
    if (seal_len < 4) return ST_INVALID_PROOF_DATA;
    if (memcmp(seal, h->selector, 4)) return ST_SELECTOR_MISMATCH;
    if (seal_len - 4 != 256) return ST_INVALID_PROOF_DATA;            /* strict abi_decode of 8 x uint256 (SURVEY 8a R4) */
    uint8_t sig[160]; zkvo_risc0_signals(h, claim, sig);
    return groth16_verify(&h->vk, seal + 4, sig, 5, NULL, NULL) ? ST_OK : ST_VERIFICATION_FAILED;
}
int zkvo_risc0_verify(const risc0_t *h, const uint8_t *seal, size_t seal_len, const uint8_t image_id[32], const uint8_t journal[32]) {   /* :78-92 */
    if (!h->initialized) return ST_INVALID_INITIALIZATION;
    uint8_t cd[32]; claim_digest(cd, image_id, journal);
    return zkvo_risc0_verify_integrity(h, seal, seal_len, cd);
}
void zkvo_risc0_verify_batch(const risc0_t *h, const uint8_t *seals, const uint64_t *seal_off, const uint8_t *image_ids, const uint8_t *journals, long n, uint8_t *status) {
    bn254_init();
#pragma omp parallel for schedule(dynamic, 4)
    for (long i = 0; i < n; i++) status[i] = (uint8_t)zkvo_risc0_verify(h, seals + seal_off[i], seal_off[i + 1] - seal_off[i], image_ids + 32 * i, journals + 32 * i);
}
void zkvo_risc0_verify_integrity_batch(const risc0_t *h, const uint8_t *seals, const uint64_t *seal_off, const uint8_t *claims, long n, uint8_t *status) {
    bn254_init();
#pragma omp parallel for schedule(dynamic, 4)
    for (long i = 0; i < n; i++) status[i] = (uint8_t)zkvo_risc0_verify_integrity(h, seals + seal_off[i], seal_off[i + 1] - seal_off[i], claims + 32 * i);
}

/* ------------------------------------------------------------------ SP1 front-end (sp1/verifier.rs:58-111) */
void zkvo_sp1_hash_public_values(const uint8_t *pv, size_t len, uint8_t out[32]) {   /* sp1/types.rs:34-38; (h & (2^253-1)) % R is the identity since 2^253 < R */
    sha256(out, pv, len); out[0] &= 0x1f;
}
int zkvo_sp1_verify(const vk_t *vk, const uint8_t selector[4], const uint8_t vkey[32], const uint8_t *pv, size_t pv_len, const uint8_t *proof, size_t proof_len) {
    bn254_init();
    if (proof_len < 4) return ST_INVALID_PROOF_DATA;
    if (memcmp(proof, selector, 4)) return ST_SELECTOR_MISMATCH;
    if (proof_len - 4 != 256) return ST_INVALID_PROOF_DATA;
    uint8_t sig[64]; memcpy(sig, vkey, 32); zkvo_sp1_hash_public_values(pv, pv_len, sig + 32);
    return groth16_verify(vk, proof + 4, sig, 2, NULL, NULL) ? ST_OK : ST_VERIFICATION_FAILED;
}
void zkvo_sp1_verify_batch(const vk_t *vk, const uint8_t selector[4], const uint8_t *vkeys, const uint8_t *pv, const uint64_t *pv_off, const uint8_t *proofs, const uint64_t *proof_off, long n, uint8_t *status) {
    bn254_init();
#pragma omp parallel for schedule(dynamic, 4)
    for (long i = 0; i < n; i++) status[i] = (uint8_t)zkvo_sp1_verify(vk, selector, vkeys + 32 * i, pv + pv_off[i], pv_off[i + 1] - pv_off[i], proofs + proof_off[i], proof_off[i + 1] - proof_off[i]);
}
/* config 5: n instances of a 4-pair check, 768 B each -> bit + optional 384-B GT */
void zkvo_pairing4_batch(const uint8_t *in, long n, uint8_t *ok, uint8_t *gt_out, uint8_t *miller_out) {
    bn254_init();
#pragma omp parallel for schedule(dynamic, 4)
    for (long i = 0; i < n; i++) {
        uint8_t ret[32];
        int rc = ec_pairing_ex(in + 768 * i, 768, ret, miller_out ? miller_out + 384 * i : NULL, gt_out ? gt_out + 384 * i : NULL);
        ok[i] = (rc == 0) ? ret[31] : 2;   /* 2 = call reverted */
    }
}
int zkvo_max_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
void zkvo_sha256(const uint8_t *msg, size_t len, uint8_t out[32]) { sha256(out, msg, len); }
