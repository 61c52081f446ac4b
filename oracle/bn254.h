/* ORACLE -- TEST INFRASTRUCTURE ONLY.  CPU restatement of the BN254 arithmetic the reference
 * delegates to the EVM precompiles 0x06/0x07/0x08
 * (/root/reference/contracts/src/common/groth16.rs:12-14,54-55,121-125).  The precompile
 * backend is NOT part of the reference tree and is not version-pinned by it (no Cargo.lock);
 * semantics follow EIP-196/197 (SURVEY.md section 8a row P0).
 *
 * PARITY STATUS: accept/reject pinned by the reference's two embedded fixtures
 * (examples/.../interact.rs) and by the independent Python referee oracle/pyref/bn254_py.py;
 * Fp12 Miller / final-exponentiation VALUES are a convention defined HERE ("parity unpinned"
 * at the Fp12 level: the reference holds no Fp12 vectors).  See DESIGN.md section 3.
 *
 * Nothing on the product path may include, link or call this file.
 *
 * Representation: Fp = 4x64-bit Montgomery (R = 2^256); Fp2 = Fp[u]/(u^2+1);
 * Fp6 = Fp2[v]/(v^3 - (9+u)); Fp12 = Fp6[w]/(w^2 - v); D-type twist y^2 = x^3 + 3/(9+u).
 */
#ifndef ZKV_ORACLE_BN254_H
#define ZKV_ORACLE_BN254_H
#include <stdint.h>
#include <string.h>

typedef unsigned __int128 u128;
typedef struct { uint64_t l[4]; } fp;
typedef struct { fp c0, c1; } fp2;
typedef struct { fp2 c0, c1, c2; } fp6;
typedef struct { fp6 c0, c1; } fp12;

/* p = Q of groth16.rs:10 ; r = R of groth16.rs:9 (little-endian 64-bit limbs) */
static const uint64_t FP_P[4] = {0x3C208C16D87CFD47ull, 0x97816A916871CA8Dull, 0xB85045B68181585Dull, 0x30644E72E131A029ull};
static const uint64_t FR_R[4] = {0x43E1F593F0000001ull, 0x2833E84879B97091ull, 0xB85045B68181585Dull, 0x30644E72E131A029ull};
#define BN_U 4965661367192848881ull

static uint64_t FP_INV64;     /* -p^-1 mod 2^64 */
static fp FP_ONE, FP_R2, FP_ZERO;
static fp2 F2_ZERO, F2_ONE, TWIST_B, XI;
static fp2 FROB_G[3][6];      /* FROB_G[k-1][i] = xi^(i*(p^k-1)/6) */
static int8_t ATE_NAF[72]; static int ATE_NAF_LEN;

/* ------------------------------------------------------------------ Fp */
static inline int fp_is_zero(const fp *a) { return (a->l[0] | a->l[1] | a->l[2] | a->l[3]) == 0; }
static inline int fp_eq(const fp *a, const fp *b) { return memcmp(a, b, sizeof(fp)) == 0; }
static inline int limbs_geq(const uint64_t a[4], const uint64_t b[4]) {
    for (int i = 3; i >= 0; i--) { if (a[i] > b[i]) return 1; if (a[i] < b[i]) return 0; }
    return 1;
}
static inline uint64_t limbs_sub(uint64_t r[4], const uint64_t a[4], const uint64_t b[4]) {
    u128 br = 0;
    for (int i = 0; i < 4; i++) { u128 t = (u128)a[i] - b[i] - (uint64_t)br; r[i] = (uint64_t)t; br = (t >> 64) & 1; }
    return (uint64_t)br;
}
static inline uint64_t limbs_add(uint64_t r[4], const uint64_t a[4], const uint64_t b[4]) {
    u128 c = 0;
    for (int i = 0; i < 4; i++) { c += (u128)a[i] + b[i]; r[i] = (uint64_t)c; c >>= 64; }
    return (uint64_t)c;
}
static inline void fp_add(fp *r, const fp *a, const fp *b) {
    limbs_add(r->l, a->l, b->l);               /* p < 2^254: no carry out */
    if (limbs_geq(r->l, FP_P)) limbs_sub(r->l, r->l, FP_P);
}
static inline void fp_sub(fp *r, const fp *a, const fp *b) {
    if (limbs_sub(r->l, a->l, b->l)) limbs_add(r->l, r->l, FP_P);
}
static inline void fp_neg(fp *r, const fp *a) {
    if (fp_is_zero(a)) *r = *a; else limbs_sub(r->l, FP_P, a->l);
}
static inline void fp_dbl(fp *r, const fp *a) { fp_add(r, a, a); }
static inline void fp_half(fp *r, const fp *a) {
    uint64_t t[4]; uint64_t c = 0;
    if (a->l[0] & 1) c = limbs_add(t, a->l, FP_P); else memcpy(t, a->l, 32);
    for (int i = 0; i < 3; i++) r->l[i] = (t[i] >> 1) | (t[i + 1] << 63);
    r->l[3] = (t[3] >> 1) | (c << 63);
}
/* CIOS Montgomery multiplication */
static inline void fp_mul(fp *r, const fp *a, const fp *b) {
    uint64_t t[6] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < 4; i++) {
        u128 c = 0;
        for (int j = 0; j < 4; j++) { c += (u128)a->l[j] * b->l[i] + t[j]; t[j] = (uint64_t)c; c >>= 64; }
        c += t[4]; t[4] = (uint64_t)c; t[5] = (uint64_t)(c >> 64);
        uint64_t m = t[0] * FP_INV64;
        c = (u128)m * FP_P[0] + t[0]; c >>= 64;
        for (int j = 1; j < 4; j++) { c += (u128)m * FP_P[j] + t[j]; t[j - 1] = (uint64_t)c; c >>= 64; }
        c += t[4]; t[3] = (uint64_t)c; t[4] = t[5] + (uint64_t)(c >> 64);
    }
    if (t[4] || limbs_geq(t, FP_P)) limbs_sub(r->l, t, FP_P); else memcpy(r->l, t, 32);
}
static inline void fp_sqr(fp *r, const fp *a) { fp_mul(r, a, a); }
static void fp_pow(fp *r, const fp *a, const uint64_t e[4]) {
    fp acc = FP_ONE;
    for (int i = 255; i >= 0; i--) {
        fp_sqr(&acc, &acc);
        if ((e[i >> 6] >> (i & 63)) & 1) fp_mul(&acc, &acc, a);
    }
    *r = acc;
}
static void fp_inv(fp *r, const fp *a) {   /* a^(p-2); inv(0) = 0 */
    uint64_t e[4] = {FP_P[0] - 2, FP_P[1], FP_P[2], FP_P[3]};
    fp_pow(r, a, e);
}
static void fp_from_limbs(fp *r, const uint64_t v[4]) { fp t; memcpy(t.l, v, 32); fp_mul(r, &t, &FP_R2); }
static void fp_to_limbs(uint64_t v[4], const fp *a) { fp one = {{1, 0, 0, 0}}, t; fp_mul(&t, a, &one); memcpy(v, t.l, 32); }
static void fp_from_u64(fp *r, uint64_t x) { uint64_t v[4] = {x, 0, 0, 0}; fp_from_limbs(r, v); }
/* 32-byte big-endian <-> limbs */
static void be32_to_limbs(uint64_t v[4], const uint8_t *b) {
    for (int i = 0; i < 4; i++) { uint64_t x = 0; for (int j = 0; j < 8; j++) x = (x << 8) | b[(3 - i) * 8 + j]; v[i] = x; }
}
static void limbs_to_be32(uint8_t *b, const uint64_t v[4]) {
    for (int i = 0; i < 4; i++) for (int j = 0; j < 8; j++) b[(3 - i) * 8 + j] = (uint8_t)(v[i] >> (56 - 8 * j));
}
static void fp_to_be32(uint8_t *b, const fp *a) { uint64_t v[4]; fp_to_limbs(v, a); limbs_to_be32(b, v); }

/* ------------------------------------------------------------------ Fp2 */
static inline int f2_is_zero(const fp2 *a) { return fp_is_zero(&a->c0) && fp_is_zero(&a->c1); }
static inline int f2_eq(const fp2 *a, const fp2 *b) { return fp_eq(&a->c0, &b->c0) && fp_eq(&a->c1, &b->c1); }
static inline void f2_add(fp2 *r, const fp2 *a, const fp2 *b) { fp_add(&r->c0, &a->c0, &b->c0); fp_add(&r->c1, &a->c1, &b->c1); }
static inline void f2_sub(fp2 *r, const fp2 *a, const fp2 *b) { fp_sub(&r->c0, &a->c0, &b->c0); fp_sub(&r->c1, &a->c1, &b->c1); }
static inline void f2_neg(fp2 *r, const fp2 *a) { fp_neg(&r->c0, &a->c0); fp_neg(&r->c1, &a->c1); }
static inline void f2_dbl(fp2 *r, const fp2 *a) { f2_add(r, a, a); }
static inline void f2_half(fp2 *r, const fp2 *a) { fp_half(&r->c0, &a->c0); fp_half(&r->c1, &a->c1); }
static inline void f2_conj(fp2 *r, const fp2 *a) { r->c0 = a->c0; fp_neg(&r->c1, &a->c1); }
static inline void f2_mul(fp2 *r, const fp2 *a, const fp2 *b) {
    fp t0, t1, s0, s1, t2;
    fp_mul(&t0, &a->c0, &b->c0); fp_mul(&t1, &a->c1, &b->c1);
    fp_add(&s0, &a->c0, &a->c1); fp_add(&s1, &b->c0, &b->c1);
    fp_mul(&t2, &s0, &s1);
    fp_sub(&r->c0, &t0, &t1);
    fp_sub(&t2, &t2, &t0); fp_sub(&r->c1, &t2, &t1);
}
static inline void f2_sqr(fp2 *r, const fp2 *a) {
    fp s, d, m;
    fp_add(&s, &a->c0, &a->c1); fp_sub(&d, &a->c0, &a->c1); fp_mul(&m, &a->c0, &a->c1);
    fp_mul(&r->c0, &s, &d); fp_dbl(&r->c1, &m);
}
static inline void f2_mul_fp(fp2 *r, const fp2 *a, const fp *k) { fp_mul(&r->c0, &a->c0, k); fp_mul(&r->c1, &a->c1, k); }
static inline void f2_mul_xi(fp2 *r, const fp2 *a) {   /* (9+u)(a0+a1 u) = (9a0-a1) + (9a1+a0)u */
    fp t0, t1, n0, n1;
    fp_dbl(&t0, &a->c0); fp_dbl(&t0, &t0); fp_dbl(&t0, &t0); fp_add(&t0, &t0, &a->c0);
    fp_dbl(&t1, &a->c1); fp_dbl(&t1, &t1); fp_dbl(&t1, &t1); fp_add(&t1, &t1, &a->c1);
    fp_sub(&n0, &t0, &a->c1); fp_add(&n1, &t1, &a->c0);
    r->c0 = n0; r->c1 = n1;
}
static void f2_inv(fp2 *r, const fp2 *a) {
    fp n, t;
    fp_sqr(&n, &a->c0); fp_sqr(&t, &a->c1); fp_add(&n, &n, &t); fp_inv(&n, &n);
    fp_mul(&r->c0, &a->c0, &n); fp_mul(&t, &a->c1, &n); fp_neg(&r->c1, &t);
}
static void f2_pow(fp2 *r, const fp2 *a, const uint64_t *e, int nlimbs) {
    fp2 acc = F2_ONE;
    for (int i = nlimbs * 64 - 1; i >= 0; i--) {
        f2_sqr(&acc, &acc);
        if ((e[i >> 6] >> (i & 63)) & 1) f2_mul(&acc, &acc, a);
    }
    *r = acc;
}

/* ------------------------------------------------------------------ Fp6 */
static inline void f6_add(fp6 *r, const fp6 *a, const fp6 *b) { f2_add(&r->c0, &a->c0, &b->c0); f2_add(&r->c1, &a->c1, &b->c1); f2_add(&r->c2, &a->c2, &b->c2); }
static inline void f6_sub(fp6 *r, const fp6 *a, const fp6 *b) { f2_sub(&r->c0, &a->c0, &b->c0); f2_sub(&r->c1, &a->c1, &b->c1); f2_sub(&r->c2, &a->c2, &b->c2); }
static inline void f6_neg(fp6 *r, const fp6 *a) { f2_neg(&r->c0, &a->c0); f2_neg(&r->c1, &a->c1); f2_neg(&r->c2, &a->c2); }
static inline void f6_mul_v(fp6 *r, const fp6 *a) { fp2 t; f2_mul_xi(&t, &a->c2); r->c2 = a->c1; r->c1 = a->c0; r->c0 = t; }
static void f6_mul(fp6 *r, const fp6 *a, const fp6 *b) {
    fp2 v0, v1, v2, t0, t1, t2, x0, x1, x2;
    f2_mul(&v0, &a->c0, &b->c0); f2_mul(&v1, &a->c1, &b->c1); f2_mul(&v2, &a->c2, &b->c2);
    /* c0 = v0 + xi((a1+a2)(b1+b2) - v1 - v2) */
    f2_add(&t0, &a->c1, &a->c2); f2_add(&t1, &b->c1, &b->c2); f2_mul(&t2, &t0, &t1);
    f2_sub(&t2, &t2, &v1); f2_sub(&t2, &t2, &v2); f2_mul_xi(&t2, &t2); f2_add(&x0, &t2, &v0);
    /* c1 = (a0+a1)(b0+b1) - v0 - v1 + xi v2 */
    f2_add(&t0, &a->c0, &a->c1); f2_add(&t1, &b->c0, &b->c1); f2_mul(&t2, &t0, &t1);
    f2_sub(&t2, &t2, &v0); f2_sub(&t2, &t2, &v1); f2_mul_xi(&t0, &v2); f2_add(&x1, &t2, &t0);
    /* c2 = (a0+a2)(b0+b2) - v0 - v2 + v1 */
    f2_add(&t0, &a->c0, &a->c2); f2_add(&t1, &b->c0, &b->c2); f2_mul(&t2, &t0, &t1);
    f2_sub(&t2, &t2, &v0); f2_sub(&t2, &t2, &v2); f2_add(&x2, &t2, &v1);
    r->c0 = x0; r->c1 = x1; r->c2 = x2;
}
static void f6_inv(fp6 *r, const fp6 *a) {
    fp2 A, B, C, t, F;
    f2_sqr(&A, &a->c0); f2_mul(&t, &a->c1, &a->c2); f2_mul_xi(&t, &t); f2_sub(&A, &A, &t);          /* a0^2 - xi a1 a2 */
    f2_sqr(&B, &a->c2); f2_mul_xi(&B, &B); f2_mul(&t, &a->c0, &a->c1); f2_sub(&B, &B, &t);          /* xi a2^2 - a0 a1 */
    f2_sqr(&C, &a->c1); f2_mul(&t, &a->c0, &a->c2); f2_sub(&C, &C, &t);                             /* a1^2 - a0 a2 */
    f2_mul(&F, &a->c0, &A);
    f2_mul(&t, &a->c2, &B); f2_mul_xi(&t, &t); f2_add(&F, &F, &t);
    f2_mul(&t, &a->c1, &C); f2_mul_xi(&t, &t); f2_add(&F, &F, &t);
    f2_inv(&F, &F);
    f2_mul(&r->c0, &A, &F); f2_mul(&r->c1, &B, &F); f2_mul(&r->c2, &C, &F);
}

/* ------------------------------------------------------------------ Fp12 */
static fp12 F12_ONE;
static inline int f12_eq(const fp12 *a, const fp12 *b) { return memcmp(a, b, sizeof(fp12)) == 0; }
static void f12_mul(fp12 *r, const fp12 *a, const fp12 *b) {
    fp6 t0, t1, s0, s1, m;
    f6_mul(&t0, &a->c0, &b->c0); f6_mul(&t1, &a->c1, &b->c1);
    f6_add(&s0, &a->c0, &a->c1); f6_add(&s1, &b->c0, &b->c1); f6_mul(&m, &s0, &s1);
    f6_sub(&m, &m, &t0); f6_sub(&r->c1, &m, &t1);
    f6_mul_v(&t1, &t1); f6_add(&r->c0, &t0, &t1);
}
static void f12_sqr(fp12 *r, const fp12 *a) { f12_mul(r, a, a); }
static inline void f12_conj(fp12 *r, const fp12 *a) { r->c0 = a->c0; f6_neg(&r->c1, &a->c1); }
static void f12_inv(fp12 *r, const fp12 *a) {
    fp6 t0, t1;
    f6_mul(&t0, &a->c0, &a->c0); f6_mul(&t1, &a->c1, &a->c1); f6_mul_v(&t1, &t1); f6_sub(&t0, &t0, &t1);
    f6_inv(&t0, &t0);
    f6_mul(&r->c0, &a->c0, &t0); f6_mul(&t1, &a->c1, &t0); f6_neg(&r->c1, &t1);
}
/* f * (l0 + (l3 + l4 v) w)  -- the sparse line product ("034") */
static void f12_mul_line(fp12 *r, const fp12 *f, const fp2 *l0, const fp2 *l3, const fp2 *l4) {
    fp12 l; memset(&l, 0, sizeof l);
    l.c0.c0 = *l0; l.c1.c0 = *l3; l.c1.c1 = *l4;
    /* (a0 + a1 w)(b0 + b1 w), b0 = (l0,0,0), b1 = (l3,l4,0) */
    fp6 t0, t1, s0, s1, m;
    const fp6 *a0 = &f->c0, *a1 = &f->c1;
    f2_mul(&t0.c0, &a0->c0, l0); f2_mul(&t0.c1, &a0->c1, l0); f2_mul(&t0.c2, &a0->c2, l0);
    f6_mul(&t1, a1, &l.c1);
    f6_add(&s0, a0, a1); s1 = l.c1; f2_add(&s1.c0, &s1.c0, l0); f6_mul(&m, &s0, &s1);
    f6_sub(&m, &m, &t0); f6_sub(&r->c1, &m, &t1);
    f6_mul_v(&t1, &t1); f6_add(&r->c0, &t0, &t1);
}
/* Frobenius f^(p^k), k = 1..3 */
static void f12_frob(fp12 *r, const fp12 *a, int k) {
    const fp2 *g = FROB_G[k - 1];
    fp2 c[6] = {a->c0.c0, a->c1.c0, a->c0.c1, a->c1.c1, a->c0.c2, a->c1.c2};  /* coefficient of w^i */
    for (int i = 0; i < 6; i++) { if (k & 1) f2_conj(&c[i], &c[i]); if (i) f2_mul(&c[i], &c[i], &g[i]); }
    r->c0.c0 = c[0]; r->c1.c0 = c[1]; r->c0.c1 = c[2]; r->c1.c1 = c[3]; r->c0.c2 = c[4]; r->c1.c2 = c[5];
}
/* Granger-Scott squaring, valid in the cyclotomic subgroup */
static void f12_cyc_sqr(fp12 *r, const fp12 *a) {
    const fp2 *z0 = &a->c0.c0, *z4 = &a->c0.c1, *z3 = &a->c0.c2, *z2 = &a->c1.c0, *z1 = &a->c1.c1, *z5 = &a->c1.c2;
    fp2 t0, t1, t2, t3, tmp, s;
    /* (z0 + z1 s)^2 over Fp4 etc. */
    f2_mul(&tmp, z0, z1); f2_add(&t0, z0, z1); f2_mul_xi(&s, z1); f2_add(&s, &s, z0); f2_mul(&t0, &t0, &s);
    f2_sub(&t0, &t0, &tmp); f2_mul_xi(&s, &tmp); f2_sub(&t0, &t0, &s); f2_dbl(&t1, &tmp);
    fp2 t0b, t1b, t0c, t1c;
    f2_mul(&tmp, z2, z3); f2_add(&t0b, z2, z3); f2_mul_xi(&s, z3); f2_add(&s, &s, z2); f2_mul(&t0b, &t0b, &s);
    f2_sub(&t0b, &t0b, &tmp); f2_mul_xi(&s, &tmp); f2_sub(&t0b, &t0b, &s); f2_dbl(&t1b, &tmp);
    f2_mul(&tmp, z4, z5); f2_add(&t0c, z4, z5); f2_mul_xi(&s, z5); f2_add(&s, &s, z4); f2_mul(&t0c, &t0c, &s);
    f2_sub(&t0c, &t0c, &tmp); f2_mul_xi(&s, &tmp); f2_sub(&t0c, &t0c, &s); f2_dbl(&t1c, &tmp);
    fp2 o0, o1, o2, o3, o4, o5;
    /* z0' = 3 t0 - 2 z0 ; z1' = 3 t1 + 2 z1 */
    f2_sub(&o0, &t0, z0); f2_dbl(&o0, &o0); f2_add(&o0, &o0, &t0);
    f2_add(&o1, &t1, z1); f2_dbl(&o1, &o1); f2_add(&o1, &o1, &t1);
    /* z2' = 3 xi t1c + 2 z2 ; z3' = 3 t0c - 2 z3 */
    f2_mul_xi(&t2, &t1c);
    f2_add(&o2, &t2, z2); f2_dbl(&o2, &o2); f2_add(&o2, &o2, &t2);
    f2_sub(&o3, &t0c, z3); f2_dbl(&o3, &o3); f2_add(&o3, &o3, &t0c);
    /* z4' = 3 t0b - 2 z4 ; z5' = 3 t1b + 2 z5 */
    f2_sub(&o4, &t0b, z4); f2_dbl(&o4, &o4); f2_add(&o4, &o4, &t0b);
    f2_add(&o5, &t1b, z5); f2_dbl(&o5, &o5); f2_add(&o5, &o5, &t1b);
    (void)t3;
    r->c0.c0 = o0; r->c0.c1 = o4; r->c0.c2 = o3; r->c1.c0 = o2; r->c1.c1 = o1; r->c1.c2 = o5;
}
static void f12_to_bytes(uint8_t *out, const fp12 *a) {  /* 12 x BE-32, tower order c0.c0.c0, c0.c0.c1, c0.c1.c0 ... */
    const fp *w = (const fp *)a;
    for (int i = 0; i < 12; i++) fp_to_be32(out + 32 * i, &w[i]);
}
static int f12_from_bytes(fp12 *a, const uint8_t *in) {
    fp *w = (fp *)a;
    for (int i = 0; i < 12; i++) { uint64_t v[4]; be32_to_limbs(v, in + 32 * i); if (limbs_geq(v, FP_P)) return -1; fp_from_limbs(&w[i], v); }
    return 0;
}

/* ------------------------------------------------------------------ G1 (Jacobian, z=0 is infinity) */
typedef struct { fp x, y, z; } g1j;
typedef struct { fp x, y; int inf; } g1a;
static void g1_dbl(g1j *r, const g1j *p) {
    if (fp_is_zero(&p->z)) { *r = *p; return; }
    fp A, B, C, D, E, F, t, x3, y3, z3;
    fp_sqr(&A, &p->x); fp_sqr(&B, &p->y); fp_sqr(&C, &B);
    fp_add(&t, &p->x, &B); fp_sqr(&t, &t); fp_sub(&t, &t, &A); fp_sub(&t, &t, &C); fp_dbl(&D, &t);
    fp_dbl(&E, &A); fp_add(&E, &E, &A); fp_sqr(&F, &E);
    fp_dbl(&t, &D); fp_sub(&x3, &F, &t);
    fp_sub(&t, &D, &x3); fp_mul(&y3, &E, &t); fp_dbl(&t, &C); fp_dbl(&t, &t); fp_dbl(&t, &t); fp_sub(&y3, &y3, &t);
    fp_mul(&z3, &p->y, &p->z); fp_dbl(&z3, &z3);
    r->x = x3; r->y = y3; r->z = z3;
}
static void g1_add(g1j *r, const g1j *p, const g1j *q) {
    if (fp_is_zero(&p->z)) { *r = *q; return; }
    if (fp_is_zero(&q->z)) { *r = *p; return; }
    fp z1z1, z2z2, u1, u2, s1, s2, h, rr, t, hh, hhh, v, x3, y3, z3;
    fp_sqr(&z1z1, &p->z); fp_sqr(&z2z2, &q->z);
    fp_mul(&u1, &p->x, &z2z2); fp_mul(&u2, &q->x, &z1z1);
    fp_mul(&s1, &p->y, &q->z); fp_mul(&s1, &s1, &z2z2);
    fp_mul(&s2, &q->y, &p->z); fp_mul(&s2, &s2, &z1z1);
    fp_sub(&h, &u2, &u1); fp_sub(&rr, &s2, &s1);
    if (fp_is_zero(&h)) {
        if (fp_is_zero(&rr)) { g1_dbl(r, p); return; }
        r->x = FP_ONE; r->y = FP_ONE; r->z = FP_ZERO; return;
    }
    fp_sqr(&hh, &h); fp_mul(&hhh, &hh, &h); fp_mul(&v, &u1, &hh);
    fp_sqr(&x3, &rr); fp_sub(&x3, &x3, &hhh); fp_dbl(&t, &v); fp_sub(&x3, &x3, &t);
    fp_sub(&t, &v, &x3); fp_mul(&y3, &rr, &t); fp_mul(&t, &s1, &hhh); fp_sub(&y3, &y3, &t);
    fp_mul(&z3, &p->z, &q->z); fp_mul(&z3, &z3, &h);
    r->x = x3; r->y = y3; r->z = z3;
}
static void g1_mul(g1j *r, const g1j *p, const uint64_t k[4]) {
    g1j acc; acc.x = FP_ONE; acc.y = FP_ONE; acc.z = FP_ZERO;
    for (int i = 255; i >= 0; i--) {
        g1_dbl(&acc, &acc);
        if ((k[i >> 6] >> (i & 63)) & 1) g1_add(&acc, &acc, p);
    }
    *r = acc;
}
static void g1_to_affine(g1a *r, const g1j *p) {
    if (fp_is_zero(&p->z)) { r->inf = 1; r->x = FP_ZERO; r->y = FP_ZERO; return; }
    fp zi, zi2; fp_inv(&zi, &p->z); fp_sqr(&zi2, &zi);
    fp_mul(&r->x, &p->x, &zi2); fp_mul(&zi2, &zi2, &zi); fp_mul(&r->y, &p->y, &zi2); r->inf = 0;
}
static void g1_from_affine(g1j *r, const g1a *p) {
    if (p->inf) { r->x = FP_ONE; r->y = FP_ONE; r->z = FP_ZERO; } else { r->x = p->x; r->y = p->y; r->z = FP_ONE; }
}
static int g1_on_curve(const fp *x, const fp *y) {
    fp l, rr, three; fp_sqr(&l, y); fp_sqr(&rr, x); fp_mul(&rr, &rr, x); fp_from_u64(&three, 3); fp_add(&rr, &rr, &three);
    return fp_eq(&l, &rr);
}

/* ------------------------------------------------------------------ G2 on the twist (Jacobian over Fp2) */
typedef struct { fp2 x, y, z; } g2j;
typedef struct { fp2 x, y; int inf; } g2a;
static void g2_dbl(g2j *r, const g2j *p) {
    if (f2_is_zero(&p->z)) { *r = *p; return; }
    fp2 A, B, C, D, E, F, t, x3, y3, z3;
    f2_sqr(&A, &p->x); f2_sqr(&B, &p->y); f2_sqr(&C, &B);
    f2_add(&t, &p->x, &B); f2_sqr(&t, &t); f2_sub(&t, &t, &A); f2_sub(&t, &t, &C); f2_dbl(&D, &t);
    f2_dbl(&E, &A); f2_add(&E, &E, &A); f2_sqr(&F, &E);
    f2_dbl(&t, &D); f2_sub(&x3, &F, &t);
    f2_sub(&t, &D, &x3); f2_mul(&y3, &E, &t); f2_dbl(&t, &C); f2_dbl(&t, &t); f2_dbl(&t, &t); f2_sub(&y3, &y3, &t);
    f2_mul(&z3, &p->y, &p->z); f2_dbl(&z3, &z3);
    r->x = x3; r->y = y3; r->z = z3;
}
static void g2_add(g2j *r, const g2j *p, const g2j *q) {
    if (f2_is_zero(&p->z)) { *r = *q; return; }
    if (f2_is_zero(&q->z)) { *r = *p; return; }
    fp2 z1z1, z2z2, u1, u2, s1, s2, h, rr, t, hh, hhh, v, x3, y3, z3;
    f2_sqr(&z1z1, &p->z); f2_sqr(&z2z2, &q->z);
    f2_mul(&u1, &p->x, &z2z2); f2_mul(&u2, &q->x, &z1z1);
    f2_mul(&s1, &p->y, &q->z); f2_mul(&s1, &s1, &z2z2);
    f2_mul(&s2, &q->y, &p->z); f2_mul(&s2, &s2, &z1z1);
    f2_sub(&h, &u2, &u1); f2_sub(&rr, &s2, &s1);
    if (f2_is_zero(&h)) {
        if (f2_is_zero(&rr)) { g2_dbl(r, p); return; }
        r->x = F2_ONE; r->y = F2_ONE; r->z = F2_ZERO; return;
    }
    f2_sqr(&hh, &h); f2_mul(&hhh, &hh, &h); f2_mul(&v, &u1, &hh);
    f2_sqr(&x3, &rr); f2_sub(&x3, &x3, &hhh); f2_dbl(&t, &v); f2_sub(&x3, &x3, &t);
    f2_sub(&t, &v, &x3); f2_mul(&y3, &rr, &t); f2_mul(&t, &s1, &hhh); f2_sub(&y3, &y3, &t);
    f2_mul(&z3, &p->z, &q->z); f2_mul(&z3, &z3, &h);
    r->x = x3; r->y = y3; r->z = z3;
}
static void g2_mul(g2j *r, const g2j *p, const uint64_t k[4]) {
    g2j acc; acc.x = F2_ONE; acc.y = F2_ONE; acc.z = F2_ZERO;
    for (int i = 255; i >= 0; i--) {
        g2_dbl(&acc, &acc);
        if ((k[i >> 6] >> (i & 63)) & 1) g2_add(&acc, &acc, p);
    }
    *r = acc;
}
static void g2_to_affine(g2a *r, const g2j *p) {
    if (f2_is_zero(&p->z)) { r->inf = 1; r->x = F2_ZERO; r->y = F2_ZERO; return; }
    fp2 zi, zi2; f2_inv(&zi, &p->z); f2_sqr(&zi2, &zi);
    f2_mul(&r->x, &p->x, &zi2); f2_mul(&zi2, &zi2, &zi); f2_mul(&r->y, &p->y, &zi2); r->inf = 0;
}
static int g2_on_curve(const fp2 *x, const fp2 *y) {
    fp2 l, rr; f2_sqr(&l, y); f2_sqr(&rr, x); f2_mul(&rr, &rr, x); f2_add(&rr, &rr, &TWIST_B);
    return f2_eq(&l, &rr);
}
/* substrate-bn style membership test: [r]Q == infinity */
static int g2_in_subgroup(const g2a *q) {
    g2j p, t; p.x = q->x; p.y = q->y; p.z = F2_ONE;
    g2_mul(&t, &p, FR_R);
    return f2_is_zero(&t.z);
}

/* ------------------------------------------------------------------ Miller loop (convention of DESIGN.md section 3)
 * R kept in homogeneous projective coordinates (X,Y,Z), x = X/Z, y = Y/Z.  Lines are the
 * triples (l0,l3,l4) meaning l0*yP + l3*xP*w + l4*v*w.                                          */
static void line_dbl(g2j *R, fp2 *l0, fp2 *l3, fp2 *l4) {
    fp2 A, B, C, E, F, G, H, I, J, E2, t;
    f2_mul(&A, &R->x, &R->y); f2_half(&A, &A);
    f2_sqr(&B, &R->y); f2_sqr(&C, &R->z);
    f2_dbl(&t, &C); f2_add(&t, &t, &C); f2_mul(&E, &TWIST_B, &t);
    f2_dbl(&F, &E); f2_add(&F, &F, &E);
    f2_add(&G, &B, &F); f2_half(&G, &G);
    f2_add(&H, &R->y, &R->z); f2_sqr(&H, &H); f2_add(&t, &B, &C); f2_sub(&H, &H, &t);
    f2_sub(&I, &E, &B);
    f2_sqr(&J, &R->x);
    f2_sqr(&E2, &E);
    f2_sub(&t, &B, &F); f2_mul(&R->x, &A, &t);
    f2_sqr(&G, &G); f2_dbl(&t, &E2); f2_add(&t, &t, &E2); f2_sub(&R->y, &G, &t);
    f2_mul(&R->z, &B, &H);
    f2_neg(l0, &H); f2_dbl(l3, &J); f2_add(l3, l3, &J); *l4 = I;
}
static void line_add(g2j *R, const fp2 *qx, const fp2 *qy, fp2 *l0, fp2 *l3, fp2 *l4) {
    fp2 th, la, C, D, E, F, G, H, t, t2;
    f2_mul(&t, qy, &R->z); f2_sub(&th, &R->y, &t);
    f2_mul(&t, qx, &R->z); f2_sub(&la, &R->x, &t);
    f2_sqr(&C, &th); f2_sqr(&D, &la); f2_mul(&E, &la, &D); f2_mul(&F, &R->z, &C); f2_mul(&G, &R->x, &D);
    f2_add(&H, &E, &F); f2_dbl(&t, &G); f2_sub(&H, &H, &t);
    f2_mul(&t, &th, qx); f2_mul(&t2, &la, qy); f2_sub(l4, &t, &t2);
    *l0 = la; f2_neg(l3, &th);
    f2_sub(&t, &G, &H); f2_mul(&t, &th, &t); f2_mul(&t2, &E, &R->y); f2_sub(&R->y, &t, &t2);
    f2_mul(&R->x, &la, &H);
    f2_mul(&R->z, &R->z, &E);
}
static void g2_frob_affine(fp2 *x, fp2 *y, int k) {  /* pi^k on the twist, k=1,2 */
    if (k & 1) { f2_conj(x, x); f2_conj(y, y); }
    f2_mul(x, x, &FROB_G[k - 1][2]); f2_mul(y, y, &FROB_G[k - 1][3]);
}
typedef struct { g1a p; g2a q; } pair_t;
/* multi-Miller: prod over pairs; pairs with an infinity member are skipped */
#define ORACLE_MAX_PAIRS 64     /* the library's ecPairing limit (include/zkv.h); the precompile itself has none */
static void miller_multi(fp12 *out, const pair_t *pairs, int n) {
    fp12 f = F12_ONE;
    g2j R[ORACLE_MAX_PAIRS]; int act[ORACLE_MAX_PAIRS]; int na = 0;
    for (int i = 0; i < n; i++) { act[i] = !(pairs[i].p.inf || pairs[i].q.inf); if (act[i]) { R[i].x = pairs[i].q.x; R[i].y = pairs[i].q.y; R[i].z = F2_ONE; na++; } }
    if (!na) { *out = f; return; }
    fp2 l0, l3, l4, a, b;
    for (int d = ATE_NAF_LEN - 2; d >= 0; d--) {
        f12_sqr(&f, &f);
        for (int i = 0; i < n; i++) if (act[i]) {
            line_dbl(&R[i], &l0, &l3, &l4);
            f2_mul_fp(&a, &l0, &pairs[i].p.y); f2_mul_fp(&b, &l3, &pairs[i].p.x);
            f12_mul_line(&f, &f, &a, &b, &l4);
        }
        if (ATE_NAF[d]) for (int i = 0; i < n; i++) if (act[i]) {
            fp2 qy = pairs[i].q.y; if (ATE_NAF[d] < 0) f2_neg(&qy, &qy);
            line_add(&R[i], &pairs[i].q.x, &qy, &l0, &l3, &l4);
            f2_mul_fp(&a, &l0, &pairs[i].p.y); f2_mul_fp(&b, &l3, &pairs[i].p.x);
            f12_mul_line(&f, &f, &a, &b, &l4);
        }
    }
    for (int i = 0; i < n; i++) if (act[i]) {
        fp2 x1 = pairs[i].q.x, y1 = pairs[i].q.y; g2_frob_affine(&x1, &y1, 1);
        fp2 x2 = pairs[i].q.x, y2 = pairs[i].q.y; g2_frob_affine(&x2, &y2, 2); f2_neg(&y2, &y2);
        line_add(&R[i], &x1, &y1, &l0, &l3, &l4);
        f2_mul_fp(&a, &l0, &pairs[i].p.y); f2_mul_fp(&b, &l3, &pairs[i].p.x); f12_mul_line(&f, &f, &a, &b, &l4);
        line_add(&R[i], &x2, &y2, &l0, &l3, &l4);
        f2_mul_fp(&a, &l0, &pairs[i].p.y); f2_mul_fp(&b, &l3, &pairs[i].p.x); f12_mul_line(&f, &f, &a, &b, &l4);
    }
    *out = f;
}
static void f12_pow_u(fp12 *r, const fp12 *a) {     /* a^u, a in the cyclotomic subgroup */
    fp12 acc = *a;
    for (int i = 61; i >= 0; i--) { f12_cyc_sqr(&acc, &acc); if ((BN_U >> i) & 1) f12_mul(&acc, &acc, a); }
    *r = acc;
}
/* GT = m^((p^6-1)(p^2+1)(L0 + L1 p + L2 p^2 + L3 p^3)); the Li are in DESIGN.md / bn254_py.py */
static void final_exp(fp12 *out, const fp12 *m) {
    fp12 f, t, fi;
    f12_conj(&t, m); f12_inv(&fi, m); f12_mul(&f, &t, &fi);          /* m^(p^6-1) */
    f12_frob(&t, &f, 2); f12_mul(&f, &t, &f);                        /* ^(p^2+1) */
    fp12 fu, f2u, f4u, f6u, f6u2, f12u2, f12u3, a, b, t0, t1;
    f12_pow_u(&fu, &f);
    f12_cyc_sqr(&f2u, &fu); f12_cyc_sqr(&f4u, &f2u); f12_mul(&f6u, &f4u, &f2u);
    f12_pow_u(&f6u2, &f6u); f12_cyc_sqr(&f12u2, &f6u2); f12_pow_u(&f12u3, &f12u2);
    f12_mul(&a, &f12u3, &f6u2); f12_mul(&a, &a, &f6u);               /* a = f^(12u^3+6u^2+6u) = f^L2 */
    f12_conj(&t, &f2u); f12_mul(&b, &a, &t);                         /* b = f^L1 */
    f12_mul(&t0, &a, &f6u2); f12_mul(&t0, &t0, &f);                  /* f^L0 */
    f12_frob(&t1, &b, 1); f12_mul(&t0, &t0, &t1);
    f12_frob(&t1, &a, 2); f12_mul(&t0, &t0, &t1);
    f12_conj(&t, &f); f12_mul(&t1, &b, &t); f12_frob(&t1, &t1, 3);  /* (b/f)^(p^3) = f^(L3 p^3) */
    f12_mul(out, &t0, &t1);
}

/* ------------------------------------------------------------------ one-time constant setup */
static void bn254_init(void) {
    static int done = 0; if (done) return;
    uint64_t inv = 1; for (int i = 0; i < 6; i++) inv *= 2 - FP_P[0] * inv; FP_INV64 = (uint64_t)(0 - inv);
    /* R mod p and R^2 mod p by repeated doubling of 1 */
    uint64_t v[4] = {1, 0, 0, 0};
    for (int i = 0; i < 512; i++) {
        uint64_t c = limbs_add(v, v, v);
        if (c || limbs_geq(v, FP_P)) limbs_sub(v, v, FP_P);
        if (i == 255) memcpy(FP_ONE.l, v, 32);
    }
    memcpy(FP_R2.l, v, 32); memset(&FP_ZERO, 0, sizeof FP_ZERO);
    memset(&F2_ZERO, 0, sizeof F2_ZERO); F2_ONE.c0 = FP_ONE; F2_ONE.c1 = FP_ZERO;
    memset(&F12_ONE, 0, sizeof F12_ONE); F12_ONE.c0.c0.c0 = FP_ONE;
    fp_from_u64(&XI.c0, 9); XI.c1 = FP_ONE;
    fp2 xi_inv, three; f2_inv(&xi_inv, &XI); fp_from_u64(&three.c0, 3); three.c1 = FP_ZERO; f2_mul(&TWIST_B, &three, &xi_inv);
    /* FROB_G[0][i] = xi^(i(p-1)/6); then g2[i] = g1[i]*conj(g1[i]) (norm trick: xi^((p^2-1)/6 i)), g3[i] = g1[i]*conj(g2[i])... computed directly by powering */
    uint64_t e[4]; /* (p-1)/6 */
    { u128 rem = 0; uint64_t pm1[4]; memcpy(pm1, FP_P, 32); pm1[0] -= 1; for (int i = 3; i >= 0; i--) { u128 cur = (rem << 64) | pm1[i]; e[i] = (uint64_t)(cur / 6); rem = cur % 6; } }
    fp2 g; f2_pow(&g, &XI, e, 4);
    FROB_G[0][0] = F2_ONE; for (int i = 1; i < 6; i++) f2_mul(&FROB_G[0][i], &FROB_G[0][i - 1], &g);
    /* xi^((p^2-1)/6) = g^(p+1) = conj(g)*g ; xi^((p^3-1)/6) = g^(p^2+p+1) = conj(g2)*g since g2 in Fp  */
    fp2 gc, g2, g3; f2_conj(&gc, &g); f2_mul(&g2, &gc, &g); f2_conj(&gc, &g2); f2_mul(&g3, &gc, &g);
    /* careful: g^(p^2) = g * (g^(p^2-1)) ; g^(p^2+p+1) = (g^(p+1))^p * g = conj(g2) * g */
    FROB_G[1][0] = F2_ONE; FROB_G[2][0] = F2_ONE;
    for (int i = 1; i < 6; i++) { f2_mul(&FROB_G[1][i], &FROB_G[1][i - 1], &g2); f2_mul(&FROB_G[2][i], &FROB_G[2][i - 1], &g3); }
    /* NAF of 6u+2 (66 digits) */
    u128 n = (u128)6 * BN_U + 2; int k = 0;
    while (n) { int d = 0; if (n & 1) { d = 2 - (int)(n & 3); n -= d; } ATE_NAF[k++] = (int8_t)d; n >>= 1; }
    ATE_NAF_LEN = k;
    done = 1;
}
#endif
