// BN254 arithmetic for the sm_100a verification kernels: Fp (8 x 32-bit Montgomery limbs, PTX carry
// chains from fp_ptx.cuh), the Fp2/Fp6/Fp12 tower, G1/G2 group law, optimal-ate line functions and
// the final exponentiation.  This is the arithmetic the reference obtains from the EVM precompiles
// ecAdd/ecMul/ecPairing (/root/reference/contracts/src/common/groth16.rs:12-14,54-55,121-125).
//
// The same source also compiles as plain C++ (tests/host_emu) with a portable Fp backend so the
// tower / curve / pairing logic can be checked on a CPU-only box; the library itself never takes
// that path: every exported entry point launches CUDA kernels.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define ZKV_HD __host__ __device__
#define ZKV_INLINE __forceinline__
#define ZKV_NOINLINE __noinline__
#define ZKV_CONST static __device__ __constant__ const
#define ZKV_TABLE static __device__ const          /* addressable per-thread operands: global memory through L1, not the constant bank */
#else
#define ZKV_HD
#define ZKV_INLINE inline
#define ZKV_NOINLINE
#define ZKV_CONST static const
#define ZKV_TABLE static const
#endif

// Block-wide rendezvous.  The heavy kernels are ~150 KB of straight-line code executed once per call site, i.e. pure streaming
// instruction fetch; warps of an SM that drift apart each need their own fetch stream and the kernels become
// instruction-fetch bound (ncu: stall_no_instruction 3.9 per issue with 2 warps per scheduler, profiles/).  All control flow of
// the Fp6-and-above routines is input independent, so a barrier at their entry keeps the warps of a block on the same cache lines.
// Only routines that EVERY thread of a block calls the same number of times may contain it (Fp2-level and curve routines,
// which the data-dependent group-law code also uses, do not).
#ifndef ZKV_RDV_LEVEL
#define ZKV_RDV_LEVEL 2
#endif
#if defined(__CUDA_ARCH__) && !defined(ZKV_NO_LOCKSTEP)
#define ZKV_RENDEZVOUS() __syncthreads()
#else
#define ZKV_RENDEZVOUS()
#endif
#if ZKV_RDV_LEVEL >= 1
#define ZKV_RENDEZVOUS1() ZKV_RENDEZVOUS()
#else
#define ZKV_RENDEZVOUS1()
#endif
#if ZKV_RDV_LEVEL >= 2
#define ZKV_RENDEZVOUS2() ZKV_RENDEZVOUS()
#else
#define ZKV_RENDEZVOUS2()
#endif

#include "bn254_consts.cuh"
#if defined(__CUDACC__)
#include "fp_ptx.cuh"
#endif

namespace zkv {

struct alignas(16) fp { uint32_t v[8]; };
struct fp2 { fp c0, c1; };
struct fp6 { fp2 c0, c1, c2; };
struct fp12 { fp6 c0, c1; };

// ------------------------------------------------------------------------------------------ Fp
ZKV_HD ZKV_INLINE fp fp_const(const uint32_t* c) { fp r; for (int i = 0; i < 8; i++) r.v[i] = c[i]; return r; }
ZKV_HD ZKV_INLINE fp fp_zero() { fp r; for (int i = 0; i < 8; i++) r.v[i] = 0; return r; }
ZKV_HD ZKV_INLINE fp fp_one() { return fp_const(C_ONE); }
ZKV_HD ZKV_INLINE bool fp_is_zero(const fp& a) { uint32_t t = 0; for (int i = 0; i < 8; i++) t |= a.v[i]; return t == 0; }
ZKV_HD ZKV_INLINE bool fp_eq(const fp& a, const fp& b) { uint32_t t = 0; for (int i = 0; i < 8; i++) t |= a.v[i] ^ b.v[i]; return t == 0; }
// raw (non-Montgomery) 256-bit compare a >= m
ZKV_HD ZKV_INLINE bool u256_geq(const uint32_t* a, const uint32_t* m) {
    uint32_t borrow = 0;
    for (int i = 0; i < 8; i++) { uint64_t t = (uint64_t)a[i] - m[i] - borrow; borrow = (uint32_t)(t >> 63); }
    return borrow == 0;
}

#if defined(__CUDA_ARCH__)
ZKV_HD ZKV_INLINE void fp_mul(fp& r, const fp& a, const fp& b) { fp_mul_ptx(r.v, a.v, b.v); }
ZKV_HD ZKV_INLINE void fp_add(fp& r, const fp& a, const fp& b) { fp_add_ptx(r.v, a.v, b.v); }
ZKV_HD ZKV_INLINE void fp_sub(fp& r, const fp& a, const fp& b) { fp_sub_ptx(r.v, a.v, b.v); }
#else
// portable backend (host emulation for tests only)
ZKV_HD inline void fp_mul(fp& r, const fp& a, const fp& b) {
    uint32_t t[10] = {0};
    for (int i = 0; i < 8; i++) {
        uint64_t c = 0;
        for (int j = 0; j < 8; j++) { c += (uint64_t)a.v[j] * b.v[i] + t[j]; t[j] = (uint32_t)c; c >>= 32; }
        c += t[8]; t[8] = (uint32_t)c; t[9] = (uint32_t)(c >> 32);
        uint32_t m = t[0] * 0xe4866389u;
        c = (uint64_t)m * C_P[0] + t[0]; c >>= 32;
        for (int j = 1; j < 8; j++) { c += (uint64_t)m * C_P[j] + t[j]; t[j - 1] = (uint32_t)c; c >>= 32; }
        c += t[8]; t[7] = (uint32_t)c; t[8] = t[9] + (uint32_t)(c >> 32);
    }
    if (t[8] || u256_geq(t, C_P)) { uint32_t bo = 0; for (int i = 0; i < 8; i++) { uint64_t d = (uint64_t)t[i] - C_P[i] - bo; r.v[i] = (uint32_t)d; bo = (uint32_t)(d >> 63); } }
    else for (int i = 0; i < 8; i++) r.v[i] = t[i];
}
ZKV_HD inline void fp_add(fp& r, const fp& a, const fp& b) {
    uint32_t t[8]; uint64_t c = 0;
    for (int i = 0; i < 8; i++) { c += (uint64_t)a.v[i] + b.v[i]; t[i] = (uint32_t)c; c >>= 32; }
    if (u256_geq(t, C_P)) { uint32_t bo = 0; for (int i = 0; i < 8; i++) { uint64_t d = (uint64_t)t[i] - C_P[i] - bo; r.v[i] = (uint32_t)d; bo = (uint32_t)(d >> 63); } }
    else for (int i = 0; i < 8; i++) r.v[i] = t[i];
}
ZKV_HD inline void fp_sub(fp& r, const fp& a, const fp& b) {
    uint32_t t[8]; uint32_t bo = 0;
    for (int i = 0; i < 8; i++) { uint64_t d = (uint64_t)a.v[i] - b.v[i] - bo; t[i] = (uint32_t)d; bo = (uint32_t)(d >> 63); }
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) { c += (uint64_t)t[i] + (bo ? C_P[i] : 0); r.v[i] = (uint32_t)c; c >>= 32; }
}
#endif
ZKV_HD ZKV_INLINE void fp_sqr(fp& r, const fp& a) { fp_mul(r, a, a); }
ZKV_HD ZKV_INLINE void fp_dbl(fp& r, const fp& a) { fp_add(r, a, a); }
ZKV_HD ZKV_INLINE void fp_neg(fp& r, const fp& a) { fp z = fp_zero(); fp_sub(r, z, a); }
ZKV_HD ZKV_INLINE void fp_half(fp& r, const fp& a) {
    uint32_t odd = 0u - (a.v[0] & 1u);
    uint32_t t[8]; uint64_t c = 0;
    for (int i = 0; i < 8; i++) { c += (uint64_t)a.v[i] + (C_P[i] & odd); t[i] = (uint32_t)c; c >>= 32; }
    for (int i = 0; i < 7; i++) r.v[i] = (t[i] >> 1) | (t[i + 1] << 31);
    r.v[7] = t[7] >> 1;   // a + p < 2^255: no carry out
}
ZKV_HD ZKV_INLINE void fp_to_mont(fp& r, const fp& a) { fp r2 = fp_const(C_R2); fp_mul(r, a, r2); }
ZKV_HD ZKV_INLINE void fp_from_mont(fp& r, const fp& a) { fp one = fp_zero(); one.v[0] = 1; fp_mul(r, a, one); }
// a^(p-2) by square-and-multiply (254 squarings + 127 products): the round-1 inversion, kept as the cross-check of fp_inv below
ZKV_HD ZKV_NOINLINE void fp_inv_fermat(fp& r, const fp& a) {
    fp acc = fp_one(), base = a;
    for (int i = 253; i >= 0; i--) {
        fp_sqr(acc, acc);
        if ((C_PM2[i >> 5] >> (i & 31)) & 1) fp_mul(acc, acc, base);
    }
    r = acc;
}
// 1 / a, inv(0) = 0.  Constant-time "safegcd" (Bernstein, Yang: "Fast constant-time gcd computation and modular inversion", 2019) in the
// 30-bit signed-limb form: 20 rounds of 30 division steps on the low words of (f, g) = (p, a), each round followed by one application of
// its 2 x 2 transition matrix to (f, g) and, modulo p, to (d, e) = (0, 1).  600 branch-free steps of ~25 ALU instructions and ~1 800
// multiplies replace the 381 Montgomery products (52 000 IMAD.WIDE) of the Fermat inversion: the inversions of a proof (affine vk_x,
// the slopes of the fixed pairs, the Fp12 inversion of the final exponentiation) leave the multiplier pipe to the pairing arithmetic.
// The result is THE inverse, so every value downstream is bit-identical to the round-1 tower and the oracle (tests/host_emu: fp_inv ==
// fp_inv_fermat == pow(a, -1, p)).  Operands are Montgomery residues x R: the plain inverse (x R)^-1 times R^3 through fp_mul is x^-1 R.
struct s30x9 { int32_t v[9]; };
ZKV_HD ZKV_INLINE void s30_divsteps(int32_t& zeta, uint32_t f0, uint32_t g0, int32_t t[4]) {
    uint32_t u = 1, v = 0, q = 0, r = 1, f = f0, g = g0;
    int32_t z = zeta;
#if defined(__CUDA_ARCH__)
#pragma unroll 6
#endif
    for (int i = 0; i < 30; i++) {
        uint32_t c1 = (uint32_t)(z >> 31), c2 = 0u - (g & 1u);
        uint32_t x = (f ^ c1) - c1, y = (u ^ c1) - c1, w = (v ^ c1) - c1;       // (f, u, v) negated while zeta < 0
        g += x & c2; q += y & c2; r += w & c2;
        c1 &= c2;                                                               // zeta < 0 and g odd: swap
        z = (int32_t)((uint32_t)z ^ c1) - 1;
        f += g & c1; u += q & c1; v += r & c1;
        g >>= 1; u <<= 1; v <<= 1;
    }
    zeta = z; t[0] = (int32_t)u; t[1] = (int32_t)v; t[2] = (int32_t)q; t[3] = (int32_t)r;
}
ZKV_HD ZKV_INLINE void s30_update_fg(s30x9& f, s30x9& g, const int32_t t[4]) {
    const int32_t M30 = 0x3FFFFFFF;
    const int64_t u = t[0], v = t[1], q = t[2], r = t[3];
    int64_t cf = u * f.v[0] + v * g.v[0], cg = q * f.v[0] + r * g.v[0];        // the low 30 bits are zero by construction
    cf >>= 30; cg >>= 30;
    for (int i = 1; i < 9; i++) {
        cf += u * f.v[i] + v * g.v[i]; cg += q * f.v[i] + r * g.v[i];
        f.v[i - 1] = (int32_t)cf & M30; cf >>= 30;
        g.v[i - 1] = (int32_t)cg & M30; cg >>= 30;
    }
    f.v[8] = (int32_t)cf; g.v[8] = (int32_t)cg;
}
ZKV_HD ZKV_INLINE void s30_update_de(s30x9& d, s30x9& e, const int32_t t[4]) {
    const int32_t M30 = 0x3FFFFFFF;
    const int64_t u = t[0], v = t[1], q = t[2], r = t[3];
    const int32_t sd = d.v[8] >> 31, se = e.v[8] >> 31;                        // negative d / e: one multiple of p is folded in
    int32_t md = (t[0] & sd) + (t[1] & se), me = (t[2] & sd) + (t[3] & se);
    int64_t cd = u * d.v[0] + v * e.v[0], ce = q * d.v[0] + r * e.v[0];
    md -= (int32_t)((ZKV_PINV30 * (uint32_t)cd + (uint32_t)md) & (uint32_t)M30);   // now t (d, e) + p (md, me) is divisible by 2^30
    me -= (int32_t)((ZKV_PINV30 * (uint32_t)ce + (uint32_t)me) & (uint32_t)M30);
    cd += (int64_t)C_P30[0] * md; ce += (int64_t)C_P30[0] * me;
    cd >>= 30; ce >>= 30;
    for (int i = 1; i < 9; i++) {
        cd += u * d.v[i] + v * e.v[i] + (int64_t)C_P30[i] * md;
        ce += q * d.v[i] + r * e.v[i] + (int64_t)C_P30[i] * me;
        d.v[i - 1] = (int32_t)cd & M30; cd >>= 30;
        e.v[i - 1] = (int32_t)ce & M30; ce >>= 30;
    }
    d.v[8] = (int32_t)cd; e.v[8] = (int32_t)ce;
}
ZKV_HD ZKV_NOINLINE void fp_inv(fp& r, const fp& a) {
    const int32_t M30 = 0x3FFFFFFF;
    s30x9 f, g, d, e;
    {   // g = a, f = p in 30-bit limbs; d = 0, e = 1
        uint64_t acc = 0; int bits = 0, k = 0;
        for (int i = 0; i < 8; i++) {
            acc |= (uint64_t)a.v[i] << bits; bits += 32;
            while (bits >= 30 && k < 8) { g.v[k++] = (int32_t)(acc & (uint64_t)M30); acc >>= 30; bits -= 30; }
        }
        g.v[8] = (int32_t)acc;
        for (int i = 0; i < 9; i++) { f.v[i] = C_P30[i]; d.v[i] = 0; e.v[i] = 0; }
        e.v[0] = 1;
    }
    int32_t zeta = -1;
    for (int it = 0; it < 20; it++) {
        int32_t t[4];
        s30_divsteps(zeta, (uint32_t)f.v[0] | ((uint32_t)f.v[1] << 30), (uint32_t)g.v[0] | ((uint32_t)g.v[1] << 30), t);
        s30_update_de(d, e, t);
        s30_update_fg(f, g, t);
    }
    // g = 0 and f = +-gcd: d = +- a^-1 in (-2p, p); normalise to [0, p) with the sign of f (a = 0: f = +-p, d = 0)
    {
        const int32_t neg = f.v[8] >> 31;
        int32_t add = d.v[8] >> 31;
        for (int i = 0; i < 9; i++) d.v[i] = ((d.v[i] + (C_P30[i] & add)) ^ neg) - neg;
        for (int i = 1; i < 9; i++) { d.v[i] += d.v[i - 1] >> 30; d.v[i - 1] &= M30; }
        add = d.v[8] >> 31;
        for (int i = 0; i < 9; i++) d.v[i] += C_P30[i] & add;
        for (int i = 1; i < 9; i++) { d.v[i] += d.v[i - 1] >> 30; d.v[i - 1] &= M30; }
    }
    fp x;
    {
        uint64_t acc = 0; int bits = 0, k = 0;
        for (int i = 0; i < 9 && k < 8; i++) {
            acc |= (uint64_t)(uint32_t)d.v[i] << bits; bits += 30;
            if (bits >= 32) { x.v[k++] = (uint32_t)acc; acc >>= 32; bits -= 32; }
        }
        if (k < 8) x.v[k] = (uint32_t)acc;
    }
    fp r3 = fp_const(C_R3);
    fp_mul(r, x, r3);
}

// ------------------------------------------------------------------------------------------ Fp2 = Fp[u]/(u^2+1)
ZKV_HD ZKV_INLINE fp2 f2_zero() { fp2 r; r.c0 = fp_zero(); r.c1 = fp_zero(); return r; }
ZKV_HD ZKV_INLINE fp2 f2_one() { fp2 r; r.c0 = fp_one(); r.c1 = fp_zero(); return r; }
ZKV_HD ZKV_INLINE fp2 f2_const(const uint32_t c[2][8]) { fp2 r; r.c0 = fp_const(c[0]); r.c1 = fp_const(c[1]); return r; }
ZKV_HD ZKV_INLINE bool f2_is_zero(const fp2& a) { return fp_is_zero(a.c0) & fp_is_zero(a.c1); }
ZKV_HD ZKV_INLINE bool f2_eq(const fp2& a, const fp2& b) { return fp_eq(a.c0, b.c0) & fp_eq(a.c1, b.c1); }
ZKV_HD ZKV_INLINE void f2_add(fp2& r, const fp2& a, const fp2& b) { fp_add(r.c0, a.c0, b.c0); fp_add(r.c1, a.c1, b.c1); }
ZKV_HD ZKV_INLINE void f2_sub(fp2& r, const fp2& a, const fp2& b) { fp_sub(r.c0, a.c0, b.c0); fp_sub(r.c1, a.c1, b.c1); }
ZKV_HD ZKV_INLINE void f2_neg(fp2& r, const fp2& a) { fp_neg(r.c0, a.c0); fp_neg(r.c1, a.c1); }
ZKV_HD ZKV_INLINE void f2_dbl(fp2& r, const fp2& a) { fp_dbl(r.c0, a.c0); fp_dbl(r.c1, a.c1); }
ZKV_HD ZKV_INLINE void f2_half(fp2& r, const fp2& a) { fp_half(r.c0, a.c0); fp_half(r.c1, a.c1); }
ZKV_HD ZKV_INLINE void f2_conj(fp2& r, const fp2& a) { r.c0 = a.c0; fp_neg(r.c1, a.c1); }
#if defined(__CUDA_ARCH__)
// Lazily reduced (fp_ptx.cuh): the Karatsuba products stay 512 bits wide and only the two result coefficients are reduced.
ZKV_HD ZKV_NOINLINE void f2_mul(fp2& r, const fp2& a, const fp2& b) {
    fp2 t; fp2_mul_ptx(t.c0.v, t.c1.v, a.c0.v, a.c1.v, b.c0.v, b.c1.v); r = t;
}
ZKV_HD ZKV_NOINLINE void f2_sqr(fp2& r, const fp2& a) {
    fp2 t; fp2_sqr_ptx(t.c0.v, t.c1.v, a.c0.v, a.c1.v); r = t;
}
#else
ZKV_HD ZKV_NOINLINE void f2_mul(fp2& r, const fp2& a, const fp2& b) {
    fp t0, t1, t2, s0, s1;
    fp_mul(t0, a.c0, b.c0); fp_mul(t1, a.c1, b.c1);
    fp_add(s0, a.c0, a.c1); fp_add(s1, b.c0, b.c1);
    fp_mul(t2, s0, s1);
    fp_sub(r.c0, t0, t1);
    fp_sub(t2, t2, t0); fp_sub(r.c1, t2, t1);
}
ZKV_HD ZKV_NOINLINE void f2_sqr(fp2& r, const fp2& a) {
    fp s, d, m;
    fp_add(s, a.c0, a.c1); fp_sub(d, a.c0, a.c1); fp_mul(m, a.c0, a.c1);
    fp_mul(r.c0, s, d); fp_dbl(r.c1, m);
}
#endif
ZKV_HD ZKV_NOINLINE void f2_mul_fp(fp2& r, const fp2& a, const fp& k) { fp_mul(r.c0, a.c0, k); fp_mul(r.c1, a.c1, k); }
// (9+u)(a0 + a1 u) = (9 a0 - a1) + (9 a1 + a0) u
ZKV_HD ZKV_NOINLINE void f2_mul_xi(fp2& r, const fp2& a) {
    fp t0, t1;
    fp_dbl(t0, a.c0); fp_dbl(t0, t0); fp_dbl(t0, t0); fp_add(t0, t0, a.c0);
    fp_dbl(t1, a.c1); fp_dbl(t1, t1); fp_dbl(t1, t1); fp_add(t1, t1, a.c1);
    fp n0, n1; fp_sub(n0, t0, a.c1); fp_add(n1, t1, a.c0);
    r.c0 = n0; r.c1 = n1;
}
ZKV_HD ZKV_NOINLINE void f2_inv(fp2& r, const fp2& a) {
    fp n, t;
    fp_sqr(n, a.c0); fp_sqr(t, a.c1); fp_add(n, n, t); fp_inv(n, n);
    fp_mul(r.c0, a.c0, n); fp_mul(t, a.c1, n); fp_neg(r.c1, t);
}

// ------------------------------------------------------------------------------------------ Fp6 = Fp2[v]/(v^3 - xi)
ZKV_HD ZKV_INLINE void f6_add(fp6& r, const fp6& a, const fp6& b) { f2_add(r.c0, a.c0, b.c0); f2_add(r.c1, a.c1, b.c1); f2_add(r.c2, a.c2, b.c2); }
ZKV_HD ZKV_INLINE void f6_sub(fp6& r, const fp6& a, const fp6& b) { f2_sub(r.c0, a.c0, b.c0); f2_sub(r.c1, a.c1, b.c1); f2_sub(r.c2, a.c2, b.c2); }
ZKV_HD ZKV_INLINE void f6_neg(fp6& r, const fp6& a) { f2_neg(r.c0, a.c0); f2_neg(r.c1, a.c1); f2_neg(r.c2, a.c2); }
ZKV_HD ZKV_INLINE void f6_mul_v(fp6& r, const fp6& a) { fp2 t; f2_mul_xi(t, a.c2); r.c2 = a.c1; r.c1 = a.c0; r.c0 = t; }
ZKV_HD ZKV_NOINLINE void f6_mul(fp6& r, const fp6& a, const fp6& b) {
    ZKV_RENDEZVOUS2();
    fp2 v0, v1, v2, t0, t1, t2, x0, x1;
    f2_mul(v0, a.c0, b.c0); f2_mul(v1, a.c1, b.c1); f2_mul(v2, a.c2, b.c2);
    f2_add(t0, a.c1, a.c2); f2_add(t1, b.c1, b.c2); f2_mul(t2, t0, t1);
    f2_sub(t2, t2, v1); f2_sub(t2, t2, v2); f2_mul_xi(t2, t2); f2_add(x0, t2, v0);
    f2_add(t0, a.c0, a.c1); f2_add(t1, b.c0, b.c1); f2_mul(t2, t0, t1);
    f2_sub(t2, t2, v0); f2_sub(t2, t2, v1); f2_mul_xi(t0, v2); f2_add(x1, t2, t0);
    f2_add(t0, a.c0, a.c2); f2_add(t1, b.c0, b.c2); f2_mul(t2, t0, t1);
    f2_sub(t2, t2, v0); f2_sub(t2, t2, v2); f2_add(r.c2, t2, v1);
    r.c0 = x0; r.c1 = x1;
}
// a * (b0 + b1 v)
ZKV_HD ZKV_NOINLINE void f6_mul_01(fp6& r, const fp6& a, const fp2& b0, const fp2& b1) {
    ZKV_RENDEZVOUS2();
    fp2 v0, v1, t0, t1, t2, x0, x2;
    f2_mul(v0, a.c0, b0); f2_mul(v1, a.c1, b1);
    f2_mul(t2, a.c2, b1); f2_mul_xi(t2, t2); f2_add(x0, t2, v0);          // c0 = a0 b0 + xi a2 b1
    f2_mul(t2, a.c2, b0); f2_add(x2, t2, v1);                             // c2 = a1 b1 + a2 b0
    f2_add(t0, a.c0, a.c1); f2_add(t1, b0, b1); f2_mul(t2, t0, t1);       // c1 = (a0+a1)(b0+b1) - v0 - v1
    f2_sub(t2, t2, v0); f2_sub(r.c1, t2, v1);
    r.c0 = x0; r.c2 = x2;
}
ZKV_HD ZKV_NOINLINE void f6_inv(fp6& r, const fp6& a) {
    ZKV_RENDEZVOUS2();
    fp2 A, B, C, t, F;
    f2_sqr(A, a.c0); f2_mul(t, a.c1, a.c2); f2_mul_xi(t, t); f2_sub(A, A, t);
    f2_sqr(B, a.c2); f2_mul_xi(B, B); f2_mul(t, a.c0, a.c1); f2_sub(B, B, t);
    f2_sqr(C, a.c1); f2_mul(t, a.c0, a.c2); f2_sub(C, C, t);
    f2_mul(F, a.c0, A);
    f2_mul(t, a.c2, B); f2_mul_xi(t, t); f2_add(F, F, t);
    f2_mul(t, a.c1, C); f2_mul_xi(t, t); f2_add(F, F, t);
    f2_inv(F, F);
    f2_mul(r.c0, A, F); f2_mul(r.c1, B, F); f2_mul(r.c2, C, F);
}

// ------------------------------------------------------------------------------------------ Fp12 = Fp6[w]/(w^2 - v)
ZKV_HD ZKV_INLINE fp12 f12_one() {
    fp12 r; fp2 z = f2_zero();
    r.c0.c0 = f2_one(); r.c0.c1 = z; r.c0.c2 = z; r.c1.c0 = z; r.c1.c1 = z; r.c1.c2 = z; return r;
}
ZKV_HD ZKV_INLINE bool f12_is_one(const fp12& a) {
    fp one = fp_one(); const fp* w = &a.c0.c0.c0; uint32_t t = 0;
    for (int i = 0; i < 8; i++) t |= w[0].v[i] ^ one.v[i];
    for (int k = 1; k < 12; k++) for (int i = 0; i < 8; i++) t |= w[k].v[i];
    return t == 0;
}
ZKV_HD ZKV_NOINLINE void f12_mul(fp12& r, const fp12& a, const fp12& b) {     // r may alias a or b
    fp6 m, t0, t1;
    f6_add(t0, a.c0, a.c1); f6_add(t1, b.c0, b.c1); f6_mul(m, t0, t1);
    f6_mul(t0, a.c0, b.c0); f6_mul(t1, a.c1, b.c1);                        // a, b are dead from here on
    f6_sub(m, m, t0); f6_sub(r.c1, m, t1);
    f6_mul_v(t1, t1); f6_add(r.c0, t0, t1);
}
// complex squaring: c0 = (a0+a1)(a0+v a1) - a0a1 - v a0a1 ; c1 = 2 a0a1
ZKV_HD ZKV_NOINLINE void f12_sqr(fp12& r, const fp12& a) {
    fp6 ab, s0, s1, t;
    f6_mul(ab, a.c0, a.c1);
    f6_add(s0, a.c0, a.c1); f6_mul_v(t, a.c1); f6_add(s1, a.c0, t);
    f6_mul(s0, s0, s1);
    f6_sub(s0, s0, ab); f6_mul_v(t, ab); f6_sub(r.c0, s0, t);
    f6_add(r.c1, ab, ab);
}
ZKV_HD ZKV_INLINE void f12_conj(fp12& r, const fp12& a) { r.c0 = a.c0; f6_neg(r.c1, a.c1); }
ZKV_HD ZKV_NOINLINE void f12_inv(fp12& r, const fp12& a) {
    fp6 t0, t1;
    f6_mul(t0, a.c0, a.c0); f6_mul(t1, a.c1, a.c1); f6_mul_v(t1, t1); f6_sub(t0, t0, t1);
    f6_inv(t0, t0);
    f6_mul(r.c0, a.c0, t0); f6_mul(t1, a.c1, t0); f6_neg(r.c1, t1);
}
// f *= l0 + (l3 + l4 v) w      (sparse "034" line product, 13 Fp2 multiplications)
ZKV_HD ZKV_NOINLINE void f12_mul_line(fp12& f, const fp2& l0, const fp2& l3, const fp2& l4) {
    ZKV_RENDEZVOUS1();
    fp6 t0, t1, s; fp2 l03;
    f2_mul(t0.c0, f.c0.c0, l0); f2_mul(t0.c1, f.c0.c1, l0); f2_mul(t0.c2, f.c0.c2, l0);
    f6_mul_01(t1, f.c1, l3, l4);
    f6_add(s, f.c0, f.c1); f2_add(l03, l0, l3);
    f6_mul_01(s, s, l03, l4);
    f6_sub(s, s, t0); f6_sub(f.c1, s, t1);
    f6_mul_v(t1, t1); f6_add(f.c0, t0, t1);
}
// f^(p^k), k in {1,2,3}
ZKV_HD ZKV_NOINLINE void f12_frob(fp12& r, const fp12& a, int k) {
    ZKV_RENDEZVOUS1();
    fp2 c[6] = {a.c0.c0, a.c1.c0, a.c0.c1, a.c1.c1, a.c0.c2, a.c1.c2};   // coefficient of w^i
    for (int i = 0; i < 6; i++) {
        if (k & 1) f2_conj(c[i], c[i]);
        if (i) {
            fp2 g = (k == 1) ? f2_const(C_FROB1[i]) : (k == 2) ? f2_const(C_FROB2[i]) : f2_const(C_FROB3[i]);
            f2_mul(c[i], c[i], g);
        }
    }
    r.c0.c0 = c[0]; r.c1.c0 = c[1]; r.c0.c1 = c[2]; r.c1.c1 = c[3]; r.c0.c2 = c[4]; r.c1.c2 = c[5];
}
// one Fp4 squaring (a + b s)^2, s^2 = xi: t0 = a^2 + xi b^2, t1 = 2ab
ZKV_HD ZKV_INLINE void fp4_sqr(fp2& t0, fp2& t1, const fp2& a, const fp2& b) {
    fp2 a2, b2, s;
    f2_sqr(a2, a); f2_sqr(b2, b);
    f2_add(s, a, b); f2_sqr(s, s); f2_sub(s, s, a2); f2_sub(t1, s, b2);
    f2_mul_xi(b2, b2); f2_add(t0, a2, b2);
}
// Granger-Scott squaring; valid only for elements of the cyclotomic subgroup
ZKV_HD ZKV_NOINLINE void f12_cyc_sqr(fp12& r, const fp12& a) {
    ZKV_RENDEZVOUS1();
    fp2 t0, t1, t2, t3, t4, t5, x;
    fp4_sqr(t0, t1, a.c0.c0, a.c1.c1);
    fp4_sqr(t2, t3, a.c1.c0, a.c0.c2);
    fp4_sqr(t4, t5, a.c0.c1, a.c1.c2);
    fp2 z0 = a.c0.c0, z4 = a.c0.c1, z3 = a.c0.c2, z2 = a.c1.c0, z1 = a.c1.c1, z5 = a.c1.c2;
    f2_sub(x, t0, z0); f2_dbl(x, x); f2_add(r.c0.c0, x, t0);     // 3 t0 - 2 z0
    f2_add(x, t1, z1); f2_dbl(x, x); f2_add(r.c1.c1, x, t1);     // 3 t1 + 2 z1
    f2_mul_xi(t5, t5);
    f2_add(x, t5, z2); f2_dbl(x, x); f2_add(r.c1.c0, x, t5);     // 3 xi t5 + 2 z2
    f2_sub(x, t4, z3); f2_dbl(x, x); f2_add(r.c0.c2, x, t4);     // 3 t4 - 2 z3
    f2_sub(x, t2, z4); f2_dbl(x, x); f2_add(r.c0.c1, x, t2);     // 3 t2 - 2 z4
    f2_add(x, t3, z5); f2_dbl(x, x); f2_add(r.c1.c2, x, t3);     // 3 t3 + 2 z5
}
// a^u for a in the cyclotomic subgroup, by the width-3 NAF of u (digits 0, +-1, +-3): one cyclotomic squaring per digit, one
// multiplication per non-zero digit (18 instead of the 27 of the binary expansion the oracle uses; same value).  A negative digit
// multiplies by the inverse, which for a unitary element is the conjugate: acc * conj(x) = conj(conj(acc) * x), so the table (a, a^3)
// is never modified and the input needs no copy.  r must not alias a.
ZKV_HD ZKV_NOINLINE void f12_pow_u(fp12& r, const fp12& a) {
    fp12 a3;
    f12_cyc_sqr(r, a); f12_mul(a3, r, a);
    if (C_U_WNAF3[ZKV_U_WNAF3_LEN - 1] == 1) r = a; else r = a3;
    for (int i = ZKV_U_WNAF3_LEN - 2; i >= 0; i--) {
        ZKV_RENDEZVOUS();
        f12_cyc_sqr(r, r);
        const int d = C_U_WNAF3[i];
        if (d) {
            if (d < 0) f12_conj(r, r);
            if (d == 1 || d == -1) f12_mul(r, r, a); else f12_mul(r, r, a3);
            if (d < 0) f12_conj(r, r);
        }
    }
}
// GT = m^((p^6-1)(p^2+1)(L0 + L1 p + L2 p^2 + L3 p^3)), L_i as in DESIGN.md section 3 (same value as the oracle's final_exp).
// Six Fp12 temporaries (the frame of this routine is the deepest of the path; every one of them is stack memory per thread).
ZKV_HD ZKV_NOINLINE void final_exp(fp12& out, const fp12& m) {
    fp12 f, t, t1, x, y, z;
    f12_conj(t, m); f12_inv(t1, m); f12_mul(f, t, t1);
    f12_frob(t, f, 2); f12_mul(f, t, f);                                   // f = m^((p^6-1)(p^2+1))
    f12_pow_u(t, f);                                                       // t = f^u
    f12_cyc_sqr(x, t); f12_cyc_sqr(t, x); f12_mul(y, t, x);                // x = f^(2u), y = f^(6u)
    f12_pow_u(z, y); f12_cyc_sqr(t, z); f12_pow_u(t1, t);                  // z = f^(6u^2), t1 = f^(12u^3)
    f12_mul(t, t1, z); f12_mul(t1, t, y);                                  // t1 = a = f^(12u^3 + 6u^2 + 6u)        (y is free now)
    f12_conj(t, x); f12_mul(y, t1, t);                                     // y = b = a * f^(-2u)                   (x is free now)
    f12_mul(t, t1, z); f12_mul(x, t, f);                                   // x = a * f^(6u^2) * f                  (z is free now)
    f12_frob(t, y, 1); f12_mul(z, x, t);                                   // z = x * b^p
    f12_frob(t, t1, 2); f12_mul(x, z, t);                                  // x = z * a^(p^2)
    f12_conj(t, f); f12_mul(t1, y, t); f12_frob(t, t1, 3);                 // t = (b / f)^(p^3)
    f12_mul(out, x, t);
}

// final_exp in four stages for the segmented kernels (same operations in the same order; the values named in final_exp are the state):
//   stage 0: m -> f, t = f^u          stage 1: t -> x = f^(2u), y = f^(6u), z = f^(6u^2)
//   stage 2: z -> t1 = f^(12u^3)      stage 3: f, x, y, z, t1 -> result
ZKV_HD ZKV_NOINLINE void final_exp_stage0(fp12& f, fp12& t, const fp12& m) {
    fp12 t1;
    f12_conj(t, m); f12_inv(t1, m); f12_mul(f, t, t1);
    f12_frob(t, f, 2); f12_mul(f, t, f);
    f12_pow_u(t, f);
}
ZKV_HD ZKV_NOINLINE void final_exp_stage1(fp12& x, fp12& y, fp12& z, const fp12& tin) {
    fp12 t;
    f12_cyc_sqr(x, tin); f12_cyc_sqr(t, x); f12_mul(y, t, x);
    f12_pow_u(z, y);
}
ZKV_HD ZKV_NOINLINE void final_exp_stage2(fp12& t1, const fp12& z) {
    fp12 t;
    f12_cyc_sqr(t, z); f12_pow_u(t1, t);
}
ZKV_HD ZKV_NOINLINE void final_exp_stage3(fp12& out, const fp12& f, fp12& x, fp12& y, fp12& z, fp12& t1) {   // x, y, z, t1 are consumed
    fp12 t;
    f12_mul(t, t1, z); f12_mul(t1, t, y);
    f12_conj(t, x); f12_mul(y, t1, t);
    f12_mul(t, t1, z); f12_mul(x, t, f);
    f12_frob(t, y, 1); f12_mul(z, x, t);
    f12_frob(t, t1, 2); f12_mul(x, z, t);
    f12_conj(t, f); f12_mul(t1, y, t); f12_frob(t, t1, 3);
    f12_mul(out, x, t);
}

// ------------------------------------------------------------------------------------------ G1: y^2 = x^3 + 3
struct g1j { fp x, y, z; };            // Jacobian; z == 0 is infinity
ZKV_HD ZKV_INLINE bool g1_on_curve(const fp& x, const fp& y) {
    fp l, r, three = fp_const(C_THREE); fp_sqr(l, y); fp_sqr(r, x); fp_mul(r, r, x); fp_add(r, r, three); return fp_eq(l, r);
}
ZKV_HD ZKV_NOINLINE void g1_dbl(g1j& r, const g1j& p) {   // infinity-safe: z=0 stays z=0
    fp A, B, C, D, E, F, t, x3, y3, z3;
    fp_sqr(A, p.x); fp_sqr(B, p.y); fp_sqr(C, B);
    fp_add(t, p.x, B); fp_sqr(t, t); fp_sub(t, t, A); fp_sub(t, t, C); fp_dbl(D, t);
    fp_dbl(E, A); fp_add(E, E, A); fp_sqr(F, E);
    fp_dbl(t, D); fp_sub(x3, F, t);
    fp_sub(t, D, x3); fp_mul(y3, E, t); fp_dbl(t, C); fp_dbl(t, t); fp_dbl(t, t); fp_sub(y3, y3, t);
    fp_mul(z3, p.y, p.z); fp_dbl(z3, z3);
    r.x = x3; r.y = y3; r.z = z3;
}
// acc += (x2,y2) affine, complete (handles acc = inf, equal and opposite points)
ZKV_HD ZKV_NOINLINE void g1_add_affine(g1j& acc, const fp& x2, const fp& y2) {
    if (fp_is_zero(acc.z)) { acc.x = x2; acc.y = y2; acc.z = fp_one(); return; }
    fp z1z1, u2, s2, h, rr, hh, hhh, v, t, x3, y3;
    fp_sqr(z1z1, acc.z); fp_mul(u2, x2, z1z1); fp_mul(s2, y2, acc.z); fp_mul(s2, s2, z1z1);
    fp_sub(h, u2, acc.x); fp_sub(rr, s2, acc.y);
    if (fp_is_zero(h)) {
        if (fp_is_zero(rr)) { g1j d; g1_dbl(d, acc); acc = d; }
        else { acc.x = fp_one(); acc.y = fp_one(); acc.z = fp_zero(); }
        return;
    }
    fp_sqr(hh, h); fp_mul(hhh, hh, h); fp_mul(v, acc.x, hh);
    fp_sqr(x3, rr); fp_sub(x3, x3, hhh); fp_dbl(t, v); fp_sub(x3, x3, t);
    fp_sub(t, v, x3); fp_mul(y3, rr, t); fp_mul(t, acc.y, hhh); fp_sub(y3, y3, t);
    fp_mul(acc.z, acc.z, h); acc.x = x3; acc.y = y3;
}
ZKV_HD ZKV_INLINE bool g1_to_affine(fp& x, fp& y, const g1j& p) {   // returns false for infinity (x=y=0)
    if (fp_is_zero(p.z)) { x = fp_zero(); y = fp_zero(); return false; }
    fp zi, zi2; fp_inv(zi, p.z); fp_sqr(zi2, zi); fp_mul(x, p.x, zi2); fp_mul(zi2, zi2, zi); fp_mul(y, p.y, zi2); return true;
}

// ------------------------------------------------------------------------------------------ G2 on the twist y^2 = x^3 + 3/xi
struct g2j { fp2 x, y, z; };           // Jacobian for the subgroup test; homogeneous projective in the Miller loop
ZKV_HD ZKV_INLINE bool g2_on_curve(const fp2& x, const fp2& y) {
    fp2 l, r, b = f2_const(C_TWIST_B); f2_sqr(l, y); f2_sqr(r, x); f2_mul(r, r, x); f2_add(r, r, b); return f2_eq(l, r);
}
ZKV_HD ZKV_NOINLINE void g2_dbl(g2j& r, const g2j& p) {
    fp2 A, B, C, D, E, F, t, x3, y3, z3;
    f2_sqr(A, p.x); f2_sqr(B, p.y); f2_sqr(C, B);
    f2_add(t, p.x, B); f2_sqr(t, t); f2_sub(t, t, A); f2_sub(t, t, C); f2_dbl(D, t);
    f2_dbl(E, A); f2_add(E, E, A); f2_sqr(F, E);
    f2_dbl(t, D); f2_sub(x3, F, t);
    f2_sub(t, D, x3); f2_mul(y3, E, t); f2_dbl(t, C); f2_dbl(t, t); f2_dbl(t, t); f2_sub(y3, y3, t);
    f2_mul(z3, p.y, p.z); f2_dbl(z3, z3);
    r.x = x3; r.y = y3; r.z = z3;
}
ZKV_HD ZKV_NOINLINE void g2_add(g2j& r, const g2j& p, const g2j& q) {   // complete
    if (f2_is_zero(p.z)) { r = q; return; }
    if (f2_is_zero(q.z)) { r = p; return; }
    fp2 z1z1, z2z2, u1, u2, s1, s2, h, rr, t, hh, hhh, v, x3, y3, z3;
    f2_sqr(z1z1, p.z); f2_sqr(z2z2, q.z);
    f2_mul(u1, p.x, z2z2); f2_mul(u2, q.x, z1z1);
    f2_mul(s1, p.y, q.z); f2_mul(s1, s1, z2z2);
    f2_mul(s2, q.y, p.z); f2_mul(s2, s2, z1z1);
    f2_sub(h, u2, u1); f2_sub(rr, s2, s1);
    if (f2_is_zero(h)) {
        if (f2_is_zero(rr)) { g2_dbl(r, p); }
        else { r.x = f2_one(); r.y = f2_one(); r.z = f2_zero(); }
        return;
    }
    f2_sqr(hh, h); f2_mul(hhh, hh, h); f2_mul(v, u1, hh);
    f2_sqr(x3, rr); f2_sub(x3, x3, hhh); f2_dbl(t, v); f2_sub(x3, x3, t);
    f2_sub(t, v, x3); f2_mul(y3, rr, t); f2_mul(t, s1, hhh); f2_sub(y3, y3, t);
    f2_mul(z3, p.z, q.z); f2_mul(z3, z3, h);
    r.x = x3; r.y = y3; r.z = z3;
}
// r = p + (qx, qy) with the second point affine (8 M + 3 S instead of 12 M + 4 S); complete like g2_add
ZKV_HD ZKV_NOINLINE void g2_add_affine(g2j& r, const g2j& p, const fp2& qx, const fp2& qy) {
    if (f2_is_zero(p.z)) { r.x = qx; r.y = qy; r.z = f2_one(); return; }
    fp2 z1z1, u2, s2, h, rr, t, hh, hhh, v, x3, y3, z3;
    f2_sqr(z1z1, p.z); f2_mul(u2, qx, z1z1);
    f2_mul(s2, qy, p.z); f2_mul(s2, s2, z1z1);
    f2_sub(h, u2, p.x); f2_sub(rr, s2, p.y);
    if (f2_is_zero(h)) {
        if (f2_is_zero(rr)) { g2_dbl(r, p); }
        else { r.x = f2_one(); r.y = f2_one(); r.z = f2_zero(); }
        return;
    }
    f2_sqr(hh, h); f2_mul(hhh, hh, h); f2_mul(v, p.x, hh);
    f2_sqr(x3, rr); f2_sub(x3, x3, hhh); f2_dbl(t, v); f2_sub(x3, x3, t);
    f2_sub(t, v, x3); f2_mul(y3, rr, t); f2_mul(t, p.y, hhh); f2_sub(y3, y3, t);
    f2_mul(z3, p.z, h);
    r.x = x3; r.y = y3; r.z = z3;
}
// psi^k = twist o Frobenius^k o untwist, on Jacobian coordinates
ZKV_HD ZKV_INLINE void g2_psi(g2j& r, const g2j& p, int k) {
    fp2 x = p.x, y = p.y, z = p.z;
    if (k & 1) { f2_conj(x, x); f2_conj(y, y); f2_conj(z, z); }
    fp2 gx = (k == 1) ? f2_const(C_FROB1[2]) : (k == 2) ? f2_const(C_FROB2[2]) : f2_const(C_FROB3[2]);
    fp2 gy = (k == 1) ? f2_const(C_FROB1[3]) : (k == 2) ? f2_const(C_FROB2[3]) : f2_const(C_FROB3[3]);
    f2_mul(r.x, x, gx); f2_mul(r.y, y, gy); r.z = z;
}
ZKV_HD ZKV_INLINE bool g2j_eq(const g2j& a, const g2j& b) {
    bool ia = f2_is_zero(a.z), ib = f2_is_zero(b.z);
    if (ia || ib) return ia && ib;
    fp2 za2, zb2, l, r; f2_sqr(za2, a.z); f2_sqr(zb2, b.z);
    f2_mul(l, a.x, zb2); f2_mul(r, b.x, za2); if (!f2_eq(l, r)) return false;
    f2_mul(za2, za2, a.z); f2_mul(zb2, zb2, b.z); f2_mul(l, a.y, zb2); f2_mul(r, b.y, za2); return f2_eq(l, r);
}
// Order-r membership for a point ON the twist: [u+1]Q + psi([u]Q) + psi^2([u]Q) == psi^3([2u]Q).
// (BN-curve test of Dai-Lin-Zhao-Zhou, eprint 2022/348 sec. 3.1.)  Same accept set as the oracle's [r]Q == inf,
// which is what tests/ check on subgroup, wrong-subgroup and small-order twist points.
ZKV_HD ZKV_NOINLINE bool g2_in_subgroup(const fp2& qx, const fp2& qy) {
    g2j q; q.x = qx; q.y = qy; q.z = f2_one();
    fp2 ax = qx, ay = qy, ny; f2_neg(ny, ay);
    g2j uq = q;                                      // [u]Q by the NAF of u with mixed additions of +-Q
    for (int i = ZKV_U_NAF_LEN - 2; i >= 0; i--) {
        g2j t; g2_dbl(t, uq); uq = t;
        const int d = C_U_NAF[i];
        if (d > 0) { g2_add_affine(t, uq, ax, ay); uq = t; }
        else if (d < 0) { g2_add_affine(t, uq, ax, ny); uq = t; }
    }
    g2j lhs, t, p1, p2, p3;
    g2_add(lhs, uq, q);
    g2_psi(p1, uq, 1); g2_add(t, lhs, p1); lhs = t;
    g2_psi(p2, uq, 2); g2_add(t, lhs, p2); lhs = t;
    g2_dbl(t, uq); g2_psi(p3, t, 3);
    return g2j_eq(lhs, p3);
}

// ------------------------------------------------------------------------------------------ Miller-loop steps
// R in homogeneous projective coordinates (x = X/Z, y = Y/Z); a line is (l0,l3,l4) meaning
// l0*yP + l3*xP*w + l4*v*w.  Formulas = oracle/bn254.h line_dbl/line_add (the shared convention).
struct line_t { fp2 l0, l3, l4; };
ZKV_HD ZKV_NOINLINE void line_dbl(g2j& R, line_t& l) {
    ZKV_RENDEZVOUS2();
    fp2 A, B, C, E, F, G, H, J, E2, t, tb = f2_const(C_TWIST_B);
    f2_mul(A, R.x, R.y); f2_half(A, A);
    f2_sqr(B, R.y); f2_sqr(C, R.z);
    f2_dbl(t, C); f2_add(t, t, C); f2_mul(E, tb, t);
    f2_dbl(F, E); f2_add(F, F, E);
    f2_add(G, B, F); f2_half(G, G);
    f2_add(H, R.y, R.z); f2_sqr(H, H); f2_add(t, B, C); f2_sub(H, H, t);
    f2_sub(l.l4, E, B);
    f2_sqr(J, R.x);
    f2_sqr(E2, E);
    f2_sub(t, B, F); f2_mul(R.x, A, t);
    f2_sqr(G, G); f2_dbl(t, E2); f2_add(t, t, E2); f2_sub(R.y, G, t);
    f2_mul(R.z, B, H);
    f2_neg(l.l0, H); f2_dbl(l.l3, J); f2_add(l.l3, l.l3, J);
}
ZKV_HD ZKV_NOINLINE void line_add(g2j& R, const fp2& qx, const fp2& qy, line_t& l) {
    ZKV_RENDEZVOUS2();
    fp2 th, la, C, D, E, F, G, H, t, t2;
    f2_mul(t, qy, R.z); f2_sub(th, R.y, t);
    f2_mul(t, qx, R.z); f2_sub(la, R.x, t);
    f2_sqr(C, th); f2_sqr(D, la); f2_mul(E, la, D); f2_mul(F, R.z, C); f2_mul(G, R.x, D);
    f2_add(H, E, F); f2_dbl(t, G); f2_sub(H, H, t);
    f2_mul(t, th, qx); f2_mul(t2, la, qy); f2_sub(l.l4, t, t2);
    l.l0 = la; f2_neg(l.l3, th);
    f2_sub(t, G, H); f2_mul(t, th, t); f2_mul(t2, E, R.y); f2_sub(R.y, t, t2);
    f2_mul(R.x, la, H);
    f2_mul(R.z, R.z, E);
}
ZKV_HD ZKV_NOINLINE void g2_frob_affine(fp2& x, fp2& y, int k) {   // pi^k on affine twist coordinates, k = 1, 2
    if (k & 1) { f2_conj(x, x); f2_conj(y, y); }
    fp2 gx = (k == 1) ? f2_const(C_FROB1[2]) : f2_const(C_FROB2[2]);
    fp2 gy = (k == 1) ? f2_const(C_FROB1[3]) : f2_const(C_FROB2[3]);
    f2_mul(x, x, gx); f2_mul(y, y, gy);
}
// f *= line evaluated at the G1 point (px, py); with off != 0 the factor is replaced by 1 (a pair with a member at
// infinity contributes 1, EIP-197): the evaluated coefficients are overwritten with (1, 0, 0) by word-wise selects, so every
// thread runs the same instruction stream and the block stays in lockstep.
// OUT OF LINE ON PURPOSE (as are the Miller loops below).  nvcc 12.9's optimiser (cicc -O1 and up; -O0 is fine) merged the stack
// slots of this routine's temporaries, when it was inlined into the Miller loop, with x2 / y2 of the loop's Frobenius tail, which are
// still live: the second Frobenius line was then computed from clobbered operands and the Miller value of the variable pair came out
// wrong, in some builds and not in others (DESIGN.md section 5).  Routines with sizeable temporaries are therefore never inlined into a
// frame that keeps its own values across the call, and the Frobenius operands are computed right before their single use.
ZKV_HD ZKV_NOINLINE void f12_mul_line_at(fp12& f, const line_t& l, const fp& px, const fp& py, bool off) {
    fp2 a, b, c;
    f2_mul_fp(a, l.l0, py); f2_mul_fp(b, l.l3, px); c = l.l4;
    const uint32_t keep = off ? 0u : 0xffffffffu;
    for (int k = 0; k < 8; k++) {
        a.c0.v[k] = (a.c0.v[k] & keep) | (C_ONE[k] & ~keep); a.c1.v[k] &= keep;
        b.c0.v[k] &= keep; b.c1.v[k] &= keep; c.c0.v[k] &= keep; c.c1.v[k] &= keep;
    }
    f12_mul_line(f, a, b, c);
}
// all ZKV_LINES_PER_G2 lines of a fixed G2 point, in the order the Miller loop consumes them
ZKV_HD ZKV_NOINLINE void g2_precompute_lines(line_t* out, const fp2& qx, const fp2& qy) {
    g2j R; R.x = qx; R.y = qy; R.z = f2_one();
    int n = 0;
    for (int d = ZKV_ATE_NAF_LEN - 2; d >= 0; d--) {
        line_dbl(R, out[n++]);
        int dg = C_ATE_NAF[d];
        if (dg) { fp2 y = qy; if (dg < 0) f2_neg(y, y); line_add(R, qx, y, out[n++]); }
    }
    { fp2 x1 = qx, y1 = qy; g2_frob_affine(x1, y1, 1); line_add(R, x1, y1, out[n++]); }
    { fp2 x2 = qx, y2 = qy; g2_frob_affine(x2, y2, 2); f2_neg(y2, y2); line_add(R, x2, y2, out[n++]); }
}

// Multi-Miller loop: one variable G2 (qx,qy; pair 0) + nfixed tabled G2 points (pairs 1..nfixed).
// skip bit j set => pair j contributes 1 (a member is infinity).  px/py: G1 points (Montgomery, affine).
// Every thread executes every step (skipped pairs multiply by 1), so the control flow is uniform across a block.
ZKV_HD ZKV_NOINLINE void miller_loop(fp12& f, const fp* px, const fp* py, const fp2& qx, const fp2& qy,
                               const line_t* const* tabs, int nfixed, uint32_t skip) {
    f = f12_one();
    g2j R; R.x = qx; R.y = qy; R.z = f2_one();
    line_t l; int li = 0;
    const bool var_off = (skip & 1u) != 0;
    for (int d = ZKV_ATE_NAF_LEN - 2; d >= 0; d--) {
        ZKV_RENDEZVOUS();
        if (d != ZKV_ATE_NAF_LEN - 2) f12_sqr(f, f);
        line_dbl(R, l); f12_mul_line_at(f, l, px[0], py[0], var_off);
        for (int j = 0; j < nfixed; j++) f12_mul_line_at(f, tabs[j][li], px[j + 1], py[j + 1], ((skip >> (j + 1)) & 1u) != 0);
        li++;
        int dg = C_ATE_NAF[d];
        if (dg) {
            fp2 y = qy; if (dg < 0) f2_neg(y, y);
            line_add(R, qx, y, l); f12_mul_line_at(f, l, px[0], py[0], var_off);
            for (int j = 0; j < nfixed; j++) f12_mul_line_at(f, tabs[j][li], px[j + 1], py[j + 1], ((skip >> (j + 1)) & 1u) != 0);
            li++;
        }
    }
    for (int s = 1; s <= 2; s++) {                      // the two Frobenius lines: Q1 = pi(Q), Q2 = -pi^2(Q), each computed right before its use
        fp2 xs = qx, ys = qy; g2_frob_affine(xs, ys, s);
        if (s == 2) f2_neg(ys, ys);
        line_add(R, xs, ys, l); f12_mul_line_at(f, l, px[0], py[0], var_off);
        for (int j = 0; j < nfixed; j++) f12_mul_line_at(f, tabs[j][li], px[j + 1], py[j + 1], ((skip >> (j + 1)) & 1u) != 0);
        li++;
    }
}

// ------------------------------------------------------------------------------------------ normalised lines (verify path)
// A line of a FIXED G2 point evaluated at P = (xP, yP) is  l0 yP + l3 xP w + l4 v w.  Dividing it by l0 yP (an element of Fp2: the final
// exponentiation maps every element of a proper subfield to 1) leaves  1 + n3 (xP/yP) w + n4 (1/yP) v w  with n3 = l3/l0, n4 = l4/l0
// tabulated per key.  The product of f with such a line needs 10 Fp2 multiplications instead of 13, and a pair that must contribute 1
// (a member at infinity) is obtained by zeroing xP/yP and 1/yP: same instruction stream, no special case.
// The Miller VALUE differs from the oracle's by subfield factors, the final exponentiation output (and so every accept / reject bit) does
// not; this path is therefore used by the verification entry points only, never by the pairing service that exposes Miller values.
struct nline_t { fp2 n3, n4; };
// f *= 1 + (c3 + c4 v) w
ZKV_HD ZKV_NOINLINE void f12_mul_line1(fp12& f, const fp2& c3, const fp2& c4) {
    ZKV_RENDEZVOUS1();
    fp6 a, b;
    f6_mul_01(a, f.c1, c3, c4); f6_mul_01(b, f.c0, c3, c4);
    f6_mul_v(a, a); f6_add(f.c0, f.c0, a); f6_add(f.c1, f.c1, b);
}
ZKV_HD ZKV_NOINLINE void f12_mul_nline_at(fp12& f, const nline_t& l, const fp& xy, const fp& iy) {
    fp2 c3, c4; f2_mul_fp(c3, l.n3, xy); f2_mul_fp(c4, l.n4, iy);
    f12_mul_line1(f, c3, c4);
}
// normalise a line table; returns false if some l0 is zero (degenerate key: the caller keeps the unscaled path)
ZKV_HD ZKV_NOINLINE bool g2_normalise_lines(nline_t* out, const line_t* in, int n) {
    // simultaneous inversion of all l0 (Montgomery's trick): out[i].n3 temporarily holds the prefix product l0_0 ... l0_i
    fp2 acc = f2_one(); bool ok = true;
    for (int i = 0; i < n; i++) { fp2 l0 = in[i].l0; if (f2_is_zero(l0)) ok = false; f2_mul(acc, acc, l0); out[i].n3 = acc; }
    if (!ok) return false;
    fp2 inv; f2_inv(inv, acc);
    for (int i = n - 1; i >= 0; i--) {
        fp2 li, l0 = in[i].l0, l3 = in[i].l3, l4 = in[i].l4, n3, n4;     // 1 / l0_i = inv(prefix_i) * prefix_{i-1}
        if (i) { fp2 prev = out[i - 1].n3; f2_mul(li, inv, prev); } else li = inv;
        f2_mul(inv, inv, l0);
        f2_mul(n3, l3, li); f2_mul(n4, l4, li);
        out[i].n3 = n3; out[i].n4 = n4;
    }
    return true;
}
// Verification-path Miller loop: pair 0 = (P0, variable Q), pairs 1, 2 = (P1, P2) against the normalised tables nt[0], nt[1].
// xy[j] = xPj / yPj, iy[j] = 1 / yPj for the two fixed pairs (both zero for a pair that must contribute 1).
// The loop can be run in SEGMENTS (digits d_hi down to d_lo of the NAF, the Frobenius lines with the last one): f and R are the state
// carried between segments (the caller keeps them in HBM), so that the kernels of several chunks can interleave at a granularity finer
// than one whole Miller loop.  miller_loop_norm is the single-segment form.
ZKV_HD ZKV_NOINLINE void miller_loop_norm_seg(fp12& f, g2j& R, const fp& px0, const fp& py0, const fp2& qx, const fp2& qy,
                                              const nline_t* const* nt, const fp* xy, const fp* iy, bool var_off, int d_hi, int d_lo, bool last) {
    line_t l; int li = 0;
    for (int d = ZKV_ATE_NAF_LEN - 2; d > d_hi; d--) li += 1 + (C_ATE_NAF[d] != 0);      // lines consumed by the earlier segments
    for (int d = d_hi; d >= d_lo; d--) {
        ZKV_RENDEZVOUS();
        if (d != ZKV_ATE_NAF_LEN - 2) f12_sqr(f, f);
        line_dbl(R, l); f12_mul_line_at(f, l, px0, py0, var_off);
        for (int j = 0; j < 2; j++) f12_mul_nline_at(f, nt[j][li], xy[j], iy[j]);
        li++;
        int dg = C_ATE_NAF[d];
        if (dg) {
            fp2 y = qy; if (dg < 0) f2_neg(y, y);
            line_add(R, qx, y, l); f12_mul_line_at(f, l, px0, py0, var_off);
            for (int j = 0; j < 2; j++) f12_mul_nline_at(f, nt[j][li], xy[j], iy[j]);
            li++;
        }
    }
    if (!last) return;
    for (int s = 1; s <= 2; s++) {
        fp2 xs = qx, ys = qy; g2_frob_affine(xs, ys, s);
        if (s == 2) f2_neg(ys, ys);
        line_add(R, xs, ys, l); f12_mul_line_at(f, l, px0, py0, var_off);
        for (int j = 0; j < 2; j++) f12_mul_nline_at(f, nt[j][li], xy[j], iy[j]);
        li++;
    }
}
// single-kernel form (own body: with compile-time loop bounds it is 3 % faster than the segment routine run over the whole range)
ZKV_HD ZKV_NOINLINE void miller_loop_norm(fp12& f, const fp& px0, const fp& py0, const fp2& qx, const fp2& qy,
                                          const nline_t* const* nt, const fp* xy, const fp* iy, bool var_off) {
    f = f12_one();
    g2j R; R.x = qx; R.y = qy; R.z = f2_one();
    line_t l; int li = 0;
    for (int d = ZKV_ATE_NAF_LEN - 2; d >= 0; d--) {
        ZKV_RENDEZVOUS();
        if (d != ZKV_ATE_NAF_LEN - 2) f12_sqr(f, f);
        line_dbl(R, l); f12_mul_line_at(f, l, px0, py0, var_off);
        for (int j = 0; j < 2; j++) f12_mul_nline_at(f, nt[j][li], xy[j], iy[j]);
        li++;
        int dg = C_ATE_NAF[d];
        if (dg) {
            fp2 y = qy; if (dg < 0) f2_neg(y, y);
            line_add(R, qx, y, l); f12_mul_line_at(f, l, px0, py0, var_off);
            for (int j = 0; j < 2; j++) f12_mul_nline_at(f, nt[j][li], xy[j], iy[j]);
            li++;
        }
    }
    for (int s = 1; s <= 2; s++) {
        fp2 xs = qx, ys = qy; g2_frob_affine(xs, ys, s);
        if (s == 2) f2_neg(ys, ys);
        line_add(R, xs, ys, l); f12_mul_line_at(f, l, px0, py0, var_off);
        for (int j = 0; j < 2; j++) f12_mul_nline_at(f, nt[j][li], xy[j], iy[j]);
        li++;
    }
}
// xy = x / y, iy = 1 / y for two affine G1 points with ONE inversion; a point with off set (or y == 0, which no point of the curve has)
// gets xy = iy = 0
ZKV_HD ZKV_NOINLINE void g1_slopes2(fp* xy, fp* iy, const fp* x, const fp* y, const bool* off) {
    const bool o0 = off[0] || fp_is_zero(y[0]), o1 = off[1] || fp_is_zero(y[1]);
    fp one = fp_one(), z = fp_zero(), y0 = o0 ? one : y[0], y1 = o1 ? one : y[1];
    fp t, inv; fp_mul(t, y0, y1); fp_inv(inv, t);
    fp i0, i1; fp_mul(i0, inv, y1); fp_mul(i1, inv, y0);
    fp a0, a1; fp_mul(a0, x[0], i0); fp_mul(a1, x[1], i1);
    xy[0] = o0 ? z : a0; xy[1] = o1 ? z : a1;
    iy[0] = o0 ? z : i0; iy[1] = o1 ? z : i1;
}

// ------------------------------------------------------------------------------------------ byte <-> field
ZKV_HD ZKV_INLINE void be32_to_raw(uint32_t* v, const uint8_t* b) {   // 32-byte big-endian -> 8 LE limbs (no reduction)
    for (int i = 0; i < 8; i++) { const uint8_t* q = b + 4 * (7 - i); v[i] = (uint32_t)q[0] << 24 | (uint32_t)q[1] << 16 | (uint32_t)q[2] << 8 | q[3]; }
}
ZKV_HD ZKV_INLINE void raw_to_be32(uint8_t* b, const uint32_t* v) {
    for (int i = 0; i < 8; i++) { uint8_t* q = b + 4 * (7 - i); q[0] = v[i] >> 24; q[1] = v[i] >> 16; q[2] = v[i] >> 8; q[3] = v[i]; }
}
ZKV_HD ZKV_INLINE void fp_to_be32(uint8_t* b, const fp& a) { fp t; fp_from_mont(t, a); raw_to_be32(b, t.v); }
// EIP-196 G1 decoding from raw limbs: returns 0 valid point (Montgomery x,y), 1 infinity, 2 invalid
ZKV_HD ZKV_INLINE int g1_decode_raw(fp& x, fp& y, const uint32_t* rx, const uint32_t* ry) {
    if (u256_geq(rx, C_P) || u256_geq(ry, C_P)) return 2;
    uint32_t any = 0;
    for (int i = 0; i < 8; i++) any |= rx[i] | ry[i];
    if (!any) { x = fp_zero(); y = fp_zero(); return 1; }
    fp t;
    for (int i = 0; i < 8; i++) t.v[i] = rx[i];
    fp_to_mont(x, t);
    for (int i = 0; i < 8; i++) t.v[i] = ry[i];
    fp_to_mont(y, t);
    return g1_on_curve(x, y) ? 0 : 2;
}
ZKV_HD inline void f12_to_bytes(uint8_t* out, const fp12& a) {   // 12 x BE-32, tower order c0.c0.c0, c0.c0.c1, c0.c1.c0, ...
    const fp* w = &a.c0.c0.c0;
    for (int i = 0; i < 12; i++) fp_to_be32(out + 32 * i, w[i]);
}

// ------------------------------------------------------------------------------------------ variable-base vk_x (keys passed as bytes)
// acc += q, both Jacobian, complete: either at infinity, equal points (doubling) and opposite points (infinity) included
ZKV_HD ZKV_NOINLINE void g1_add_jac(g1j& acc, const g1j& q) {
    if (fp_is_zero(q.z)) return;
    if (fp_is_zero(acc.z)) { acc = q; return; }
    fp z1z1, z2z2, u1, u2, s1, s2, h, rr, t;
    fp_sqr(z1z1, acc.z); fp_sqr(z2z2, q.z);
    fp_mul(u1, acc.x, z2z2); fp_mul(u2, q.x, z1z1);
    fp_mul(s1, acc.y, q.z); fp_mul(s1, s1, z2z2); fp_mul(s2, q.y, acc.z); fp_mul(s2, s2, z1z1);
    fp_sub(h, u2, u1); fp_sub(rr, s2, s1);
    if (fp_is_zero(h)) {
        if (fp_is_zero(rr)) { g1j d; g1_dbl(d, acc); acc = d; }
        else { acc.x = fp_one(); acc.y = fp_one(); acc.z = fp_zero(); }
        return;
    }
    fp hh, hhh, v, x3, y3;
    fp_sqr(hh, h); fp_mul(hhh, hh, h); fp_mul(v, u1, hh);
    fp_sqr(x3, rr); fp_sub(x3, x3, hhh); fp_dbl(t, v); fp_sub(x3, x3, t);
    fp_sub(t, v, x3); fp_mul(y3, rr, t); fp_mul(t, s1, hhh); fp_sub(y3, y3, t);
    fp_mul(t, acc.z, q.z); fp_mul(acc.z, t, h); acc.x = x3; acc.y = y3;
}
#define ZKV_VKX_MAX_SCALARS 15            /* n_ic <= 16 */
// width-4 NAF of k < 2^255 (odd digits -7..7, each non-zero digit followed by at least three zeros) as 256 nibbles, digit b in nibble b & 7 of
// w[b >> 3].  Scanned from bit 0 with the carry c of the negative digits: an even window value is a zero digit and leaves c as it is.
ZKV_HD ZKV_INLINE void g1_wnaf4(uint32_t* w, const uint32_t* k) {
    for (int q = 0; q < 32; q++) w[q] = 0;
    uint32_t c = 0;
    for (int b = 0; b < 256;) {
        const int q = b >> 5, sh = b & 31;
        uint32_t win = k[q] >> sh;
        if (sh > 28 && q < 7) win |= k[q + 1] << (32 - sh);
        win = (win & 15u) + c;
        if (!(win & 1u)) { b++; continue; }
        c = win >= 8u;
        w[b >> 3] |= (win & 15u) << (4 * (b & 7));         // win - 16 for a negative digit: the same low four bits
        b += 4;
    }
}
// vk_x = IC_0 + sum_j s_j IC_{j+1} (compute_vk_x, groth16.rs:51-58: the chain of ecMul / ecAdd precompile calls) for a key whose IC points
// arrive as bytes: ic = n_ic x 64 B (EVM words), s = n_ic - 1 scalars as 32-byte BE words.  Any 256-bit scalar is taken (ecMul reduces it:
// s P = (s mod r) P on G1).  Straus: one doubling chain shared by all scalars, each recoded as a width-4 NAF whose digits are added from a
// per-thread table of P, 3P, 5P, 7P (Jacobian).  Every addition is complete, so IC points or partial sums at infinity, and partial sums
// equal or opposite to a table entry, give the group's sum, which is what the chain computes; one inversion takes it to affine.
// Returns 0 (x, y) finite, 1 infinity (x = y = 0), 2 an IC point fails the EIP-196 checks (the chain's ecMul / ecAdd call fails; x = y = 0).
ZKV_HD ZKV_NOINLINE int g1_vkx_var(fp& x, fp& y, const uint8_t* ic, int n_ic, const uint8_t* s) {
    g1j tab[ZKV_VKX_MAX_SCALARS][4];
    uint32_t naf[ZKV_VKX_MAX_SCALARS][32];
    bool bad = false;
    g1j base; base.x = fp_one(); base.y = fp_one(); base.z = fp_zero();
    for (int j = 0; j < n_ic; j++) {
        uint32_t rx[8], ry[8];
        be32_to_raw(rx, ic + 64 * j); be32_to_raw(ry, ic + 64 * j + 32);
        fp px, py;
        const int r = g1_decode_raw(px, py, rx, ry);
        bad |= r == 2;
        if (j == 0) { if (r == 0) { base.x = px; base.y = py; base.z = fp_one(); } continue; }
        uint32_t k[8];
        be32_to_raw(k, s + 32 * (j - 1));
        while (u256_geq(k, C_R)) { uint32_t bo = 0; for (int t = 0; t < 8; t++) { uint64_t d = (uint64_t)k[t] - C_R[t] - bo; k[t] = (uint32_t)d; bo = (uint32_t)(d >> 63); } }
        if (r != 0) for (int t = 0; t < 8; t++) k[t] = 0;      // IC_j at infinity adds nothing
        g1_wnaf4(naf[j - 1], k);
        if (r != 0) continue;
        g1j* T = tab[j - 1];
        T[0].x = px; T[0].y = py; T[0].z = fp_one();
        g1j p2; g1_dbl(p2, T[0]);
        for (int m = 1; m < 4; m++) { T[m] = T[m - 1]; g1_add_jac(T[m], p2); }
    }
    if (bad) { x = fp_zero(); y = fp_zero(); return 2; }
    g1j acc; acc.x = fp_one(); acc.y = fp_one(); acc.z = fp_zero();
    for (int b = 255; b >= 0; b--) {
        if (!fp_is_zero(acc.z)) { g1j d; g1_dbl(d, acc); acc = d; }
        for (int j = 0; j + 1 < n_ic; j++) {
            const uint32_t nb = (naf[j][b >> 3] >> (4 * (b & 7))) & 15u;
            if (!nb) continue;
            const bool neg = nb >= 8u;
            g1j e = tab[j][((neg ? 16u - nb : nb) >> 1)];
            if (neg) fp_neg(e.y, e.y);
            g1_add_jac(acc, e);
        }
    }
    g1_add_jac(acc, base);
    return g1_to_affine(x, y, acc) ? 0 : 1;
}

}  // namespace zkv
