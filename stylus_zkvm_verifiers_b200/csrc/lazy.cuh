// Shared-memory-resident, lazily reduced Fp12 arithmetic for the two heavy kernels (multi-Miller loop, final exponentiation).
//
// Round 1 ran one proof per thread with every Fp2-and-above operand behind a pointer into the per-thread stack (3.3 - 4.5 KB per
// thread): 190 MB of stack for the resident threads of one wave against 126 MB of L2, 30 GB of DRAM traffic per Miller launch and a
// multiplier pipe that was busy 46 % of the time (VERDICT round 1).  Here the working set of a proof lives in SHARED MEMORY:
//   * every thread owns LZ_SLOTS "slots" of one Fp element (8 x u32) each, word-interleaved across the block as 128-bit vectors
//     (slot s, half h of thread t is lz_sm[(2 s + h) * LZ_NT + t]): a warp's LDS.128 / STS.128 touch 512 contiguous bytes, no bank conflict;
//   * the Fp6-level routines (csrc/lazy_gen.cuh, generated and bound-checked by tools/gen_lazy.py) take slot addresses, keep their
//     512-bit intermediate products in registers (255 registers, no spill, no stack) and reduce once per output coefficient;
//   * two blocks of LZ_NT = 128 threads per SM: 28 slots x 32 B x 128 threads = 112 KB per block.
// The arithmetic is the one behind the reference's ecPairing precompile call (/root/reference/contracts/src/common/groth16.rs:121-125);
// all values at rest are canonical Montgomery residues, so every result is bit-identical to the round-1 tower (bn254.cuh) and to the oracle.
#pragma once
#include "bn254.cuh"
#if !defined(__CUDACC__)
#include <cstdio>
#include <cstdlib>
#endif

#ifndef LZ_NT
#define LZ_NT 128
#endif
#define LZ_SLOT (2 * LZ_NT)
#define LZ_SLOTS 28

namespace zkv {

// Block-wide rendezvous at the entry of the Fp12-level routines (what ZKV_RENDEZVOUS is to the round-1 kernels).  OFF: measured on the
// Miller operation mix it buys nothing in this layout (61.7 % of the IMAD.WIDE issue rate without, 60.8 % with: profiles/r2_lzbench.json),
// and a build with the barriers inside these out-of-line routines faulted with an illegal address in k_miller_lz under cicc -O3 (not under
// -Xcicc -O1, not with the routines inlined, not with the barriers removed): no barrier, no exposure.
#ifdef LZ_LOCKSTEP
#define LZ_RDV() ZKV_RENDEZVOUS()
#else
#define LZ_RDV()
#endif

struct fp4 { fp2 c0, c1; };     // a + b s in Fp4 = Fp2[s] / (s^2 - xi) (the Granger-Scott squaring works on three such pairs)

#if defined(__CUDACC__)
#ifndef LZ_FN
#define LZ_FN __device__ __noinline__       /* the generated Fp6-level routines */
#endif
#ifndef LZ_FN2
#define LZ_FN2 __device__ __noinline__      /* the Fp12-level routines built on them */
#endif
#define LZ_INL __device__ __forceinline__
extern __shared__ uint4 lz_sm[];
LZ_INL uint32_t lz_tid() { return threadIdx.x; }
#ifdef ZKV_LZ_CHECK
#define LZ_CHK(idx) do { if ((idx) + LZ_NT >= LZ_SLOTS * LZ_SLOT) { printf("smem index out of range: %u (thread %u)\n", (unsigned)(idx), threadIdx.x); return; } } while (0)
#else
#define LZ_CHK(idx)
#endif
LZ_INL void lz_ld(uint32_t* r, uint32_t idx) {
    LZ_CHK(idx);
    uint4 a = lz_sm[idx], b = lz_sm[idx + LZ_NT];
    r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w; r[4] = b.x; r[5] = b.y; r[6] = b.z; r[7] = b.w;
}
LZ_INL void lz_st(uint32_t idx, const uint32_t* r) {
    LZ_CHK(idx);
    lz_sm[idx] = make_uint4(r[0], r[1], r[2], r[3]); lz_sm[idx + LZ_NT] = make_uint4(r[4], r[5], r[6], r[7]);
}
#else
// host emulation (tests/host_emu): one "thread", the slots are a plain array, the leaves are portable C with overflow checks
#include "../../tests/host_emu/lazy_leaf_host.h"
#endif

LZ_INL void lz_fp_neg(uint32_t* r, const uint32_t* a) { fp z = fp_zero(), x, y; for (int i = 0; i < 8; i++) x.v[i] = a[i]; fp_sub(y, z, x); for (int i = 0; i < 8; i++) r[i] = y.v[i]; }

#include "lazy_gen.cuh"

// ---------------------------------------------------------------------------------------------- slot <-> register helpers (canonical values)
LZ_INL fp lz_ldfp(uint32_t idx) { fp r; lz_ld(r.v, idx); return r; }
LZ_INL void lz_stfp(uint32_t idx, const fp& a) { lz_st(idx, a.v); }
LZ_INL fp2 lz_ld2(uint32_t idx) { fp2 r; lz_ld(r.c0.v, idx); lz_ld(r.c1.v, idx + LZ_SLOT); return r; }
LZ_INL void lz_st2(uint32_t idx, const fp2& a) { lz_st(idx, a.c0.v); lz_st(idx + LZ_SLOT, a.c1.v); }
LZ_INL void lz_st6(uint32_t idx, const fp6& a) { lz_st2(idx, a.c0); lz_st2(idx + 2 * LZ_SLOT, a.c1); lz_st2(idx + 4 * LZ_SLOT, a.c2); }
LZ_INL fp2 f2v_add(const fp2& a, const fp2& b) { fp2 r; f2_add(r, a, b); return r; }
LZ_INL fp2 f2v_sub(const fp2& a, const fp2& b) { fp2 r; f2_sub(r, a, b); return r; }
LZ_INL fp2 f2v_dbl(const fp2& a) { fp2 r; f2_dbl(r, a); return r; }
LZ_INL fp2 f2v_xi(const fp2& a) {       // (9 + u) a
    fp t0, t1; fp2 r;
    fp_dbl(t0, a.c0); fp_dbl(t0, t0); fp_dbl(t0, t0); fp_add(t0, t0, a.c0);
    fp_dbl(t1, a.c1); fp_dbl(t1, t1); fp_dbl(t1, t1); fp_add(t1, t1, a.c1);
    fp_sub(r.c0, t0, a.c1); fp_add(r.c1, t1, a.c0);
    return r;
}

// ---------------------------------------------------------------------------------------------- Fp12 on slots
// f (12 slots at `f`) <- f^2, complex squaring; `t` = a 6-slot temporary.  Two lz_f6mul, no other multiplication:
//   t = a0 a1;  (a0, a1) <- (a0 + a1, a0 + v a1) in place;  p = a0' a1';  c0 = p - t - v t,  c1 = 2 t.
LZ_FN2 void lz_f12sqr(uint32_t f, uint32_t t) {
    LZ_RDV();
    {
        fp6 ab = lz_f6mul(f, f + 6 * LZ_SLOT);
        lz_st6(t, ab);
    }
    {
        fp2 x0 = lz_ld2(f), x1 = lz_ld2(f + 2 * LZ_SLOT), x2 = lz_ld2(f + 4 * LZ_SLOT);
        fp2 y0 = lz_ld2(f + 6 * LZ_SLOT), y1 = lz_ld2(f + 8 * LZ_SLOT), y2 = lz_ld2(f + 10 * LZ_SLOT);
        lz_st2(f, f2v_add(x0, y0)); lz_st2(f + 2 * LZ_SLOT, f2v_add(x1, y1)); lz_st2(f + 4 * LZ_SLOT, f2v_add(x2, y2));
        lz_st2(f + 6 * LZ_SLOT, f2v_add(x0, f2v_xi(y2))); lz_st2(f + 8 * LZ_SLOT, f2v_add(x1, y0)); lz_st2(f + 10 * LZ_SLOT, f2v_add(x2, y1));
    }
    LZ_RDV();
    fp6 p = lz_f6mul(f, f + 6 * LZ_SLOT);
    fp2 t0 = lz_ld2(t), t1 = lz_ld2(t + 2 * LZ_SLOT), t2 = lz_ld2(t + 4 * LZ_SLOT);
    lz_st2(f, f2v_sub(f2v_sub(p.c0, t0), f2v_xi(t2)));
    lz_st2(f + 2 * LZ_SLOT, f2v_sub(f2v_sub(p.c1, t1), t0));
    lz_st2(f + 4 * LZ_SLOT, f2v_sub(f2v_sub(p.c2, t2), t1));
    lz_st2(f + 6 * LZ_SLOT, f2v_dbl(t0)); lz_st2(f + 8 * LZ_SLOT, f2v_dbl(t1)); lz_st2(f + 10 * LZ_SLOT, f2v_dbl(t2));
}

// f *= 1 + (c3 + c4 v) w   (a NORMALISED line of a fixed G2 point, bn254.cuh) with c3, c4 in the two Fp2 slots at `l`; `t` = 6-slot temporary.
//   a = f1 (c3 + c4 v) -> t;  b = f0 (c3 + c4 v);  f1 += b;  f0 += v a.        10 Fp2 products, 6 reductions (2 x lz_f6mul01)
LZ_FN2 void lz_mul_nline(uint32_t f, uint32_t t, uint32_t l) {
    LZ_RDV();
    { fp6 a = lz_f6mul01(f + 6 * LZ_SLOT, l); lz_st6(t, a); }
    fp6 b = lz_f6mul01(f, l);
    lz_st2(f + 6 * LZ_SLOT, f2v_add(lz_ld2(f + 6 * LZ_SLOT), b.c0));
    lz_st2(f + 8 * LZ_SLOT, f2v_add(lz_ld2(f + 8 * LZ_SLOT), b.c1));
    lz_st2(f + 10 * LZ_SLOT, f2v_add(lz_ld2(f + 10 * LZ_SLOT), b.c2));
    lz_st2(f, f2v_add(lz_ld2(f), f2v_xi(lz_ld2(t + 4 * LZ_SLOT))));
    lz_st2(f + 2 * LZ_SLOT, f2v_add(lz_ld2(f + 2 * LZ_SLOT), lz_ld2(t)));
    lz_st2(f + 4 * LZ_SLOT, f2v_add(lz_ld2(f + 4 * LZ_SLOT), lz_ld2(t + 2 * LZ_SLOT)));
}

// Fp2 helpers with operands and result BY VALUE: nvcc passes them in registers (no stack traffic, unlike the pointer forms of bn254.cuh),
// and one copy of the multiplier serves every call site of the curve arithmetic below (instruction-cache footprint).
LZ_FN fp2 f2v_mul(fp2 a, fp2 b) {
    fp2 r;
#if defined(__CUDA_ARCH__)
    fp2_mul_ptx(r.c0.v, r.c1.v, a.c0.v, a.c1.v, b.c0.v, b.c1.v);
#else
    f2_mul(r, a, b);
#endif
    return r;
}
LZ_FN fp2 f2v_sqr(fp2 a) {
    fp2 r;
#if defined(__CUDA_ARCH__)
    fp2_sqr_ptx(r.c0.v, r.c1.v, a.c0.v, a.c1.v);
#else
    f2_sqr(r, a);
#endif
    return r;
}
LZ_INL fp2 f2v_neg(const fp2& a) { fp2 r; f2_neg(r, a); return r; }
LZ_INL fp2 f2v_half(const fp2& a) { fp2 r; f2_half(r, a); return r; }
LZ_INL fp2 f2v_mul_fp(const fp2& a, const fp& k) { fp2 r; fp_mul(r.c0, a.c0, k); fp_mul(r.c1, a.c1, k); return r; }

// f *= a + (b + c v) w   (line of the VARIABLE G2 point evaluated at P: a = l0 yP, b = l3 xP, c = l4); b, c in the two Fp2 slots at `l`
// (clobbered), a by value; `t` = 6-slot temporary.  Karatsuba over Fp6:
//   t1 = f1 (b + c v) -> t;  f1 <- f0 + f1;  b <- a + b;  s = f1 (b + c v);  t0 = f0 a (coefficient-wise);  f0 = t0 + v t1;  f1 = s - t0 - t1.
LZ_FN2 void lz_mul_line(uint32_t f, uint32_t t, uint32_t l, fp2 a) {
    LZ_RDV();
    { fp6 t1 = lz_f6mul01(f + 6 * LZ_SLOT, l); lz_st6(t, t1); }
    for (int k = 0; k < 3; k++) lz_st2(f + (6 + 2 * k) * LZ_SLOT, f2v_add(lz_ld2(f + 2 * k * LZ_SLOT), lz_ld2(f + (6 + 2 * k) * LZ_SLOT)));
    lz_st2(l, f2v_add(lz_ld2(l), a));
    fp6 s = lz_f6mul01(f + 6 * LZ_SLOT, l);
    {
        fp2 t0 = f2v_mul(lz_ld2(f), a), t10 = lz_ld2(t), t12 = lz_ld2(t + 4 * LZ_SLOT);
        lz_st2(f, f2v_add(t0, f2v_xi(t12)));
        lz_st2(f + 6 * LZ_SLOT, f2v_sub(f2v_sub(s.c0, t0), t10));
        t0 = f2v_mul(lz_ld2(f + 2 * LZ_SLOT), a); fp2 t11 = lz_ld2(t + 2 * LZ_SLOT);
        lz_st2(f + 2 * LZ_SLOT, f2v_add(t0, t10));
        lz_st2(f + 8 * LZ_SLOT, f2v_sub(f2v_sub(s.c1, t0), t11));
        t0 = f2v_mul(lz_ld2(f + 4 * LZ_SLOT), a);
        lz_st2(f + 4 * LZ_SLOT, f2v_add(t0, t11));
        lz_st2(f + 10 * LZ_SLOT, f2v_sub(f2v_sub(s.c2, t0), t12));
    }
}

// ---------------------------------------------------------------------------------------------- Miller-loop steps on slots
// R = (X, Y, Z) in the three Fp2 slots at `r` (homogeneous projective, formulas of bn254.cuh line_dbl / line_add = oracle/bn254.h);
// the line l0 yP + l3 xP w + l4 v w is evaluated at P = (px, py) on the way out: b = l3 xP and c = l4 go to the two Fp2 slots at `l`,
// a = l0 yP is returned.  With off != 0 the line is replaced by 1 (a pair with a member at infinity), same instruction stream.
LZ_INL fp2 lz_line_out(uint32_t l, const fp2& l0, const fp2& l3, const fp2& l4, const fp& px, const fp& py, bool off) {
    fp2 a = f2v_mul_fp(l0, py), b = f2v_mul_fp(l3, px), c = l4;
    const uint32_t keep = off ? 0u : 0xffffffffu;
    for (int k = 0; k < 8; k++) {
        a.c0.v[k] = (a.c0.v[k] & keep) | (C_ONE[k] & ~keep); a.c1.v[k] &= keep;
        b.c0.v[k] &= keep; b.c1.v[k] &= keep; c.c0.v[k] &= keep; c.c1.v[k] &= keep;
    }
    lz_st2(l, b); lz_st2(l + 2 * LZ_SLOT, c);
    return a;
}
LZ_FN2 fp2 lz_line_dbl(uint32_t r, uint32_t l, const fp* px, const fp* py, bool off) {
    LZ_RDV();
    fp2 X = lz_ld2(r), Y = lz_ld2(r + 2 * LZ_SLOT), Z = lz_ld2(r + 4 * LZ_SLOT);
    fp2 A = f2v_half(f2v_mul(X, Y));
    fp2 B = f2v_sqr(Y), C = f2v_sqr(Z);
    fp2 E = f2v_mul(f2_const(C_TWIST_B), f2v_add(f2v_dbl(C), C));
    fp2 F = f2v_add(f2v_dbl(E), E);
    fp2 H = f2v_sub(f2v_sqr(f2v_add(Y, Z)), f2v_add(B, C));
    fp2 J = f2v_sqr(X);
    fp2 E2 = f2v_sqr(E);
    lz_st2(r, f2v_mul(A, f2v_sub(B, F)));
    fp2 G = f2v_sqr(f2v_half(f2v_add(B, F)));
    lz_st2(r + 2 * LZ_SLOT, f2v_sub(G, f2v_add(f2v_dbl(E2), E2)));
    lz_st2(r + 4 * LZ_SLOT, f2v_mul(B, H));
    return lz_line_out(l, f2v_neg(H), f2v_add(f2v_dbl(J), J), f2v_sub(E, B), *px, *py, off);
}
LZ_FN2 fp2 lz_line_add(uint32_t r, uint32_t l, fp2 qx, fp2 qy, const fp* px, const fp* py, bool off) {
    LZ_RDV();
    fp2 X = lz_ld2(r), Y = lz_ld2(r + 2 * LZ_SLOT), Z = lz_ld2(r + 4 * LZ_SLOT);
    fp2 th = f2v_sub(Y, f2v_mul(qy, Z)), la = f2v_sub(X, f2v_mul(qx, Z));
    fp2 C = f2v_sqr(th), D = f2v_sqr(la);
    fp2 E = f2v_mul(la, D), F = f2v_mul(Z, C), G = f2v_mul(X, D);
    fp2 H = f2v_sub(f2v_add(E, F), f2v_dbl(G));
    fp2 l4 = f2v_sub(f2v_mul(th, qx), f2v_mul(la, qy));
    lz_st2(r + 2 * LZ_SLOT, f2v_sub(f2v_mul(th, f2v_sub(G, H)), f2v_mul(E, Y)));
    lz_st2(r, f2v_mul(la, H));
    lz_st2(r + 4 * LZ_SLOT, f2v_mul(Z, E));
    return lz_line_out(l, la, f2v_neg(th), l4, *px, *py, off);
}

// Slot map of the verification Miller loop (per thread): f = slots 0..11, T = 12..17, R = 18..23, L = 24..27.
#define LZ_F 0
#define LZ_T 12
#define LZ_R 18
#define LZ_L 24
struct LzMillerIn {                 // everything a thread reads per step comes from global memory (L2-resident, 0.4 KB per proof), not from registers
    const fp *px0, *py0;            // G1 point of the variable pair
    const fp2 *qx, *qy;             // the variable G2 point
    const fp* sl;                   // xy0, xy1, iy0, iy1: slopes of the two fixed pairs (g1_slopes2)
    const nline_t* nt[2];           // normalised line tables of the two fixed G2 points
    bool var_off;
};
// The two fixed pairs' lines number li: f *= 1 + n3 (xP/yP) w + n4 (1/yP) v w for each.
// Their table entries (2 x 128 bytes per step, the same for every proof) are STAGED IN SHARED MEMORY, one 256-byte area per warp behind the
// slots (the kilobyte per block that 2 x 112 KB of slots leave of the SM's 228 KB): sixteen lanes fetch 16 bytes each of the NEXT step's
// entries at the start of a step, the loads are in flight during the step's two line products, and the values are parked in the staging
// area at its end, so the loop no longer waits for L2 (the long-scoreboard share of the loop body, DESIGN.md section 5).  Warp-private, so
// `__syncwarp` is all the ordering it needs.  `have` says whether the area already holds entry li (false at the start of a segment).
#define LZ_STAGE (LZ_SLOTS * LZ_SLOT)            /* uint4 index of the staging areas: 16 uint4 per warp */
#if defined(__CUDACC__)
LZ_INL uint32_t lz_stage_base() { return LZ_STAGE + (lz_tid() >> 5) * 16; }
LZ_INL uint4 lz_line_fetch(const nline_t* const nt[2], int li) {
    const uint32_t lane = lz_tid() & 31;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (lane < 16) v = ((const uint4*)(nt[lane >> 3] + li))[lane & 7];
    return v;
}
LZ_INL void lz_line_stage(uint4 v) {
    const uint32_t lane = lz_tid() & 31;
    __syncwarp();
    if (lane < 16) lz_sm[lz_stage_base() + lane] = v;
    __syncwarp();
}
LZ_INL nline_t lz_line_staged(int j) {
    nline_t nl; uint4* w = (uint4*)&nl;
    for (int k = 0; k < 8; k++) w[k] = lz_sm[lz_stage_base() + 8 * j + k];
    return nl;
}
#else
struct lz_stage_t { nline_t e[2]; };
static lz_stage_t lz_stage_host;
LZ_INL lz_stage_t lz_line_fetch(const nline_t* const nt[2], int li) { lz_stage_t v; v.e[0] = nt[0][li]; v.e[1] = nt[1][li]; return v; }
LZ_INL void lz_line_stage(const lz_stage_t& v) { lz_stage_host = v; }
LZ_INL nline_t lz_line_staged(int j) { return lz_stage_host.e[j]; }
#endif
LZ_INL void lz_fixed_lines(const LzMillerIn& in, int li, uint32_t tid, bool& have) {
    if (!have) lz_line_stage(lz_line_fetch(in.nt, li));
    const int nx = li + 1 < ZKV_LINES_PER_G2 ? li + 1 : li;
    auto next = lz_line_fetch(in.nt, nx);
    for (int j = 0; j < 2; j++) {
        nline_t nl = lz_line_staged(j);
        lz_st2(tid + LZ_L * LZ_SLOT, f2v_mul_fp(nl.n3, in.sl[j]));
        lz_st2(tid + (LZ_L + 2) * LZ_SLOT, f2v_mul_fp(nl.n4, in.sl[2 + j]));
        lz_mul_nline(tid + LZ_F * LZ_SLOT, tid + LZ_T * LZ_SLOT, tid + LZ_L * LZ_SLOT);
    }
    lz_line_stage(next); have = nx == li + 1;
}
// digits d_hi .. d_lo of the loop (the two Frobenius lines with the last segment); f and R must be in the slots (f = 1, R = Q before the first).
// OUT OF LINE, arguments by value: inlined into a kernel that also holds arrays for the slope computation, nvcc 12.9 merged stack slots of
// the (then address-taken) argument block with those arrays and the loop read clobbered pointers (the stack-slot merging bug of DESIGN.md
// section 5, seen again on the GPU as an illegal address); in its own frame the block lives in registers.
LZ_FN2 void lz_miller_norm_seg(LzMillerIn in, int d_hi, int d_lo, bool last) {
    const uint32_t tid = lz_tid(), F = tid + LZ_F * LZ_SLOT, T = tid + LZ_T * LZ_SLOT, RR = tid + LZ_R * LZ_SLOT, L = tid + LZ_L * LZ_SLOT;
    int li = 0; bool have = false;
    for (int d = ZKV_ATE_NAF_LEN - 2; d > d_hi; d--) li += 1 + (C_ATE_NAF[d] != 0);
    for (int d = d_hi; d >= d_lo; d--) {
        if (d != ZKV_ATE_NAF_LEN - 2) lz_f12sqr(F, T);
        { fp2 a = lz_line_dbl(RR, L, in.px0, in.py0, in.var_off); lz_mul_line(F, T, L, a); }
        lz_fixed_lines(in, li, tid, have);
        li++;
        const int dg = C_ATE_NAF[d];
        if (dg) {
            fp2 y = *in.qy; if (dg < 0) y = f2v_neg(y);
            { fp2 a = lz_line_add(RR, L, *in.qx, y, in.px0, in.py0, in.var_off); lz_mul_line(F, T, L, a); }
            lz_fixed_lines(in, li, tid, have);
            li++;
        }
    }
    if (!last) return;
    for (int s = 1; s <= 2; s++) {
        fp2 xs = *in.qx, ys = *in.qy; g2_frob_affine(xs, ys, s);
        if (s == 2) ys = f2v_neg(ys);
        { fp2 a = lz_line_add(RR, L, xs, ys, in.px0, in.py0, in.var_off); lz_mul_line(F, T, L, a); }
        lz_fixed_lines(in, li, tid, have);
        li++;
    }
}
// The order-r test of B, finished at the end of the verification Miller loop (DESIGN.md section 4).  The loop above leaves
// R = [6u+2]B + psi(B) - psi^2(B), and 6u+2 + p - p^2 + p^3 = 0 (mod r), so R = -psi^3(B) = T for B in G2 (psi acts as p there).  For B on
// the twist but outside G2 the sum is not T (the endomorphism 6u+2 + psi - psi^2 + psi^3 has no kernel in the cofactor group: its norm is
// prime to 2p - r), or an exceptional case of the homogeneous formulas (R = B or R = O before an addition) left Z_R = 0 for good.
// T in affine coordinates; B = (0, 0), the encoding of infinity, gives T = (0, 0).
LZ_INL void g2_neg_psi3(fp2& x, fp2& y) {
    f2_conj(x, x); f2_conj(y, y);
    x = f2v_mul(x, f2_const(C_FROB3[2])); y = f2v_neg(f2v_mul(y, f2_const(C_FROB3[3])));
}
// R (the three Fp2 slots at `r`) equals T: Z_R != 0, X_R = x_T Z_R, Y_R = y_T Z_R.  T = (0, 0) (B = infinity, a member) passes; no point
// of the twist has x = y = 0.
LZ_INL bool lz_r_is(uint32_t r, const fp2& tx, const fp2& ty) {
    const fp2 Z = lz_ld2(r + 4 * LZ_SLOT);
    const fp2 dx = f2v_sub(lz_ld2(r), f2v_mul(tx, Z)), dy = f2v_sub(lz_ld2(r + 2 * LZ_SLOT), f2v_mul(ty, Z));
    return (!f2_is_zero(Z) && f2_is_zero(dx) && f2_is_zero(dy)) || (f2_is_zero(tx) && f2_is_zero(ty));
}
// General multi-Miller loop on slots (pairing services): `nvar` pairs with their own variable G2 point, then `nfix` pairs whose G2 points
// have tabled (unscaled) lines; unscaled line products throughout, so the value is the oracle's Miller value bit for bit.  Arrays are
// pair-major (pair j of instance i at [j * stride + i]).  With more than one variable pair the accumulators R_j do not fit in the slots:
// R_j lives in global memory (`rst`, L2-resident) and visits the R slots for its own step; with one variable pair R stays in the slots.
struct LzGenIn {
    const fp *px, *py;              // G1 points, (nvar + nfix) x stride
    const fp2 *qx, *qy;             // variable G2 points, nvar x stride
    g2j* rst;                       // R_j between steps / segments, nvar x stride
    const line_t* tabs[3];          // line tables of the fixed G2 points
    const uint8_t* pskip;           // per pair: != 0 -> the pair contributes 1 (a member at infinity, or an instance that is not evaluated)
    size_t stride; int nvar, nfix;
};
LZ_FN2 void lz_miller_gen_seg(LzGenIn in, size_t i, int d_hi, int d_lo, bool first, bool last) {
    const uint32_t tid = lz_tid(), F = tid + LZ_F * LZ_SLOT, T = tid + LZ_T * LZ_SLOT, RR = tid + LZ_R * LZ_SLOT, L = tid + LZ_L * LZ_SLOT;
    const bool keep = in.nvar == 1;        // R stays in the slots for the whole segment
    int li = 0;
    for (int d = ZKV_ATE_NAF_LEN - 2; d > d_hi; d--) li += 1 + (C_ATE_NAF[d] != 0);
    if (keep) {
        if (first) { lz_st2(RR, in.qx[i]); lz_st2(RR + 2 * LZ_SLOT, in.qy[i]); lz_st2(RR + 4 * LZ_SLOT, f2_one()); }
        else { const g2j* R = in.rst + i; lz_st2(RR, R->x); lz_st2(RR + 2 * LZ_SLOT, R->y); lz_st2(RR + 4 * LZ_SLOT, R->z); }
    }
    const int nsteps = (d_hi - d_lo + 1) + (last ? 2 : 0);
    for (int step = 0; step < nsteps; step++) {
        const int d = d_hi - step;                          // d < d_lo: the two Frobenius steps
        const int frob = d < d_lo ? d_lo - d : 0;           // 1, 2
        if (!frob && d != ZKV_ATE_NAF_LEN - 2) lz_f12sqr(F, T);
        const int dg = frob ? 1 : C_ATE_NAF[d];
        for (int phase = frob ? 1 : 0; phase < 2; phase++) {                // phase 0: doubling lines, phase 1: addition lines (if the digit is non-zero)
            if (phase == 1 && !dg) break;
            for (int j = 0; j < in.nvar; j++) {
                const size_t ij = (size_t)j * in.stride + i;
                const bool off = in.pskip[ij] != 0;
                if (!keep) {
                    if (first && step == 0 && phase == 0) { lz_st2(RR, in.qx[ij]); lz_st2(RR + 2 * LZ_SLOT, in.qy[ij]); lz_st2(RR + 4 * LZ_SLOT, f2_one()); }
                    else { const g2j* R = in.rst + ij; lz_st2(RR, R->x); lz_st2(RR + 2 * LZ_SLOT, R->y); lz_st2(RR + 4 * LZ_SLOT, R->z); }
                }
                fp2 a;
                if (phase == 0) a = lz_line_dbl(RR, L, in.px + ij, in.py + ij, off);
                else {
                    fp2 x = in.qx[ij], y = in.qy[ij];
                    if (frob) { if (frob == 1) { f2_conj(x, x); f2_conj(y, y); } x = f2v_mul(x, f2_const(frob == 1 ? C_FROB1[2] : C_FROB2[2])); y = f2v_mul(y, f2_const(frob == 1 ? C_FROB1[3] : C_FROB2[3])); if (frob == 2) y = f2v_neg(y); }
                    else if (dg < 0) y = f2v_neg(y);
                    a = lz_line_add(RR, L, x, y, in.px + ij, in.py + ij, off);
                }
                lz_mul_line(F, T, L, a);
                if (!keep) { g2j* R = in.rst + ij; R->x = lz_ld2(RR); R->y = lz_ld2(RR + 2 * LZ_SLOT); R->z = lz_ld2(RR + 4 * LZ_SLOT); }
            }
            for (int j = 0; j < in.nfix; j++) {
                const size_t ij = (size_t)(in.nvar + j) * in.stride + i;
                const line_t ln = in.tabs[j][li];
                fp2 a = lz_line_out(L, ln.l0, ln.l3, ln.l4, in.px[ij], in.py[ij], in.pskip[ij] != 0);
                lz_mul_line(F, T, L, a);
            }
            li++;
        }
    }
    if (keep && !last) { g2j* R = in.rst + i; R->x = lz_ld2(RR); R->y = lz_ld2(RR + 2 * LZ_SLOT); R->z = lz_ld2(RR + 4 * LZ_SLOT); }
}
// After the last segment of a loop with nvar > 1 (R_j in in.rst): the order-r test of every variable G2 point, R_j against T_j = -psi^3(Q_j)
// (pair-major like the points).  The argument of lz_r_is holds per pair: each R_j ran through every doubling, addition and Frobenius step of
// its own Q_j, whatever its skip byte said.  Uses the R slots.
LZ_INL bool lz_gen_subgroup_ok(const LzGenIn& in, size_t i, const fp2* tx, const fp2* ty) {
    const uint32_t RR = lz_tid() + LZ_R * LZ_SLOT;
    bool ok = true;
    for (int j = 0; j < in.nvar; j++) {
        const size_t ij = (size_t)j * in.stride + i;
        const g2j* R = in.rst + ij;
        lz_st2(RR, R->x); lz_st2(RR + 2 * LZ_SLOT, R->y); lz_st2(RR + 4 * LZ_SLOT, R->z);
        ok &= lz_r_is(RR, tx[ij], ty[ij]);
    }
    return ok;
}
LZ_INL void lz_miller_init(const fp2& qx, const fp2& qy) {       // f = 1, R = (qx, qy, 1)
    const uint32_t tid = lz_tid();
    fp2 one = f2_one(), z = f2_zero();
    lz_st2(tid + LZ_F * LZ_SLOT, one);
    for (int k = 1; k < 6; k++) lz_st2(tid + (LZ_F + 2 * k) * LZ_SLOT, z);
    lz_st2(tid + LZ_R * LZ_SLOT, qx); lz_st2(tid + (LZ_R + 2) * LZ_SLOT, qy); lz_st2(tid + (LZ_R + 4) * LZ_SLOT, one);
}

// ---------------------------------------------------------------------------------------------- final exponentiation on slots
// Slot map: A = slots 0..11 (the accumulator), X = 12..17, Y = 18..23 (two Fp6 temporaries), L = 24..27 (two Fp2).  Operands other than
// the accumulator are read from GLOBAL memory (they are cold: one 384-byte read per use), so one proof needs 24 + 4 slots, not 36.
LZ_INL void lz_ldg6(uint32_t dst, const fp6* src, bool neg) {             // global Fp6 -> 6 slots, optionally negated
    const fp* w = &src->c0.c0;
    for (int k = 0; k < 6; k++) { fp t = w[k]; if (neg) fp_neg(t, t); lz_stfp(dst + k * LZ_SLOT, t); }
}
LZ_INL void lz_ldg12(uint32_t dst, const fp12* src) { lz_ldg6(dst, &src->c0, false); lz_ldg6(dst + 6 * LZ_SLOT, &src->c1, false); }
LZ_INL void lz_stg12(fp12* dst, uint32_t src) { fp* w = &dst->c0.c0.c0; for (int k = 0; k < 12; k++) w[k] = lz_ldfp(src + k * LZ_SLOT); }
LZ_INL void lz_conj(uint32_t a) { for (int k = 6; k < 12; k++) { fp t = lz_ldfp(a + k * LZ_SLOT); fp_neg(t, t); lz_stfp(a + k * LZ_SLOT, t); } }
// A <- A * b (b in global memory; conjb: multiply by conj(b), the inverse of a unitary b).  Karatsuba over Fp6 with everything in place:
//   X <- b0, Y <- t0 = A0 X;  A0 <- A0 + A1;  X <- b1, A1 <- t1 = A1 X;  X <- b0 + b1;  m = A0 X;  A1 <- m - t0 - t1,  A0 <- t0 + v t1.
LZ_FN2 void lz_f12mul_g(uint32_t a, uint32_t x, uint32_t y, const fp12* b, bool conjb) {
    LZ_RDV();
    lz_ldg6(x, &b->c0, false);
    { fp6 t0 = lz_f6mul(a, x); lz_st6(y, t0); }
    for (int k = 0; k < 3; k++) lz_st2(a + 2 * k * LZ_SLOT, f2v_add(lz_ld2(a + 2 * k * LZ_SLOT), lz_ld2(a + (6 + 2 * k) * LZ_SLOT)));
    lz_ldg6(x, &b->c1, conjb);
    { fp6 t1 = lz_f6mul(a + 6 * LZ_SLOT, x); lz_st6(a + 6 * LZ_SLOT, t1); }
    { const fp* w = &b->c0.c0.c0; for (int k = 0; k < 6; k++) { fp t; fp_add(t, lz_ldfp(x + k * LZ_SLOT), w[k]); lz_stfp(x + k * LZ_SLOT, t); } }
    LZ_RDV();
    fp6 m = lz_f6mul(a, x);
    fp2 t10 = lz_ld2(a + 6 * LZ_SLOT), t11 = lz_ld2(a + 8 * LZ_SLOT), t12 = lz_ld2(a + 10 * LZ_SLOT);
    fp2 t00 = lz_ld2(y), t01 = lz_ld2(y + 2 * LZ_SLOT), t02 = lz_ld2(y + 4 * LZ_SLOT);
    lz_st2(a + 6 * LZ_SLOT, f2v_sub(f2v_sub(m.c0, t00), t10));
    lz_st2(a + 8 * LZ_SLOT, f2v_sub(f2v_sub(m.c1, t01), t11));
    lz_st2(a + 10 * LZ_SLOT, f2v_sub(f2v_sub(m.c2, t02), t12));
    lz_st2(a, f2v_add(t00, f2v_xi(t12)));
    lz_st2(a + 2 * LZ_SLOT, f2v_add(t01, t10));
    lz_st2(a + 4 * LZ_SLOT, f2v_add(t02, t11));
}
// Granger-Scott squaring of a cyclotomic-subgroup element in place (bn254.cuh f12_cyc_sqr); `l` = two spare Fp2 slots.
// Fp2 coefficient k of the element sits at slots 2k, 2k+1 (k: c0.c0, c0.c1, c0.c2, c1.c0, c1.c1, c1.c2).
LZ_FN2 void lz_cyc_sqr(uint32_t a, uint32_t l) {
    LZ_RDV();
    const uint32_t z0 = a, z4 = a + 2 * LZ_SLOT, z3 = a + 4 * LZ_SLOT, z2 = a + 6 * LZ_SLOT, z1 = a + 8 * LZ_SLOT, z5 = a + 10 * LZ_SLOT;
    {
        fp4 t = lz_f4sqr(z0, z1);                                       // (t0, t1)
        fp2 x = f2v_dbl(f2v_sub(t.c0, lz_ld2(z0))); lz_st2(z0, f2v_add(x, t.c0));      // 3 t0 - 2 z0
        x = f2v_dbl(f2v_add(t.c1, lz_ld2(z1))); lz_st2(z1, f2v_add(x, t.c1));          // 3 t1 + 2 z1
    }
    { fp4 t = lz_f4sqr(z2, z3); lz_st2(l, t.c0); lz_st2(l + 2 * LZ_SLOT, t.c1); }      // (t2, t3) parked: their targets z4, z5 are inputs of the next squaring
    {
        fp4 t = lz_f4sqr(z4, z5);                                       // (t4, t5)
        fp2 t5 = f2v_xi(t.c1);
        fp2 x = f2v_dbl(f2v_add(t5, lz_ld2(z2))); lz_st2(z2, f2v_add(x, t5));          // 3 xi t5 + 2 z2
        x = f2v_dbl(f2v_sub(t.c0, lz_ld2(z3))); lz_st2(z3, f2v_add(x, t.c0));          // 3 t4 - 2 z3
        fp2 t2 = lz_ld2(l), t3 = lz_ld2(l + 2 * LZ_SLOT);
        x = f2v_dbl(f2v_sub(t2, lz_ld2(z4))); lz_st2(z4, f2v_add(x, t2));              // 3 t2 - 2 z4
        x = f2v_dbl(f2v_add(t3, lz_ld2(z5))); lz_st2(z5, f2v_add(x, t3));              // 3 t3 + 2 z5
    }
}
// A <- A^(p^k), k = 1, 2, 3, in place
LZ_FN2 void lz_frob(uint32_t a, int k) {
    LZ_RDV();
    const int slot_of_w[6] = {0, 3, 1, 4, 2, 5};                        // coefficient of w^i is Fp2 number slot_of_w[i]
    for (int i = 0; i < 6; i++) {
        const uint32_t s = a + 2 * slot_of_w[i] * LZ_SLOT;
        fp2 c = lz_ld2(s);
        if (k & 1) f2_conj(c, c);
        if (i) c = f2v_mul(c, (k == 1) ? f2_const(C_FROB1[i]) : (k == 2) ? f2_const(C_FROB2[i]) : f2_const(C_FROB3[i]));
        if (i || (k & 1)) lz_st2(s, c);
    }
}
LZ_INL fp fpv_inv(fp a) { fp r; fp_inv(r, a); return r; }            // safegcd inversion of bn254.cuh; inv(0) = 0
// A <- 1 / A in place (bn254.cuh f12_inv / f6_inv); x, y = Fp6 temporaries
LZ_FN2 void lz_f12inv(uint32_t a, uint32_t x, uint32_t y) {
    LZ_RDV();
    { fp6 s0 = lz_f6mul(a, a); lz_st6(y, s0); }
    {
        fp6 s1 = lz_f6mul(a + 6 * LZ_SLOT, a + 6 * LZ_SLOT);            // t = a0^2 - v a1^2
        lz_st2(x, f2v_sub(lz_ld2(y), f2v_xi(s1.c2)));
        lz_st2(x + 2 * LZ_SLOT, f2v_sub(lz_ld2(y + 2 * LZ_SLOT), s1.c0));
        lz_st2(x + 4 * LZ_SLOT, f2v_sub(lz_ld2(y + 4 * LZ_SLOT), s1.c1));
    }
    {                                                                   // x <- 1 / x in Fp6
        fp2 c0 = lz_ld2(x), c1 = lz_ld2(x + 2 * LZ_SLOT), c2 = lz_ld2(x + 4 * LZ_SLOT);
        fp2 A = f2v_sub(f2v_sqr(c0), f2v_xi(f2v_mul(c1, c2)));
        fp2 B = f2v_sub(f2v_xi(f2v_sqr(c2)), f2v_mul(c0, c1));
        fp2 C = f2v_sub(f2v_sqr(c1), f2v_mul(c0, c2));
        fp2 F = f2v_add(f2v_add(f2v_mul(c0, A), f2v_xi(f2v_mul(c2, B))), f2v_xi(f2v_mul(c1, C)));
        fp n, t; fp_sqr(n, F.c0); fp_sqr(t, F.c1); fp_add(n, n, t); n = fpv_inv(n);
        fp2 Fi; fp_mul(Fi.c0, F.c0, n); fp_mul(t, F.c1, n); fp_neg(Fi.c1, t);
        lz_st2(x, f2v_mul(A, Fi)); lz_st2(x + 2 * LZ_SLOT, f2v_mul(B, Fi)); lz_st2(x + 4 * LZ_SLOT, f2v_mul(C, Fi));
    }
    LZ_RDV();
    { fp6 r0 = lz_f6mul(a, x); lz_st6(a, r0); }
    {
        fp6 r1 = lz_f6mul(a + 6 * LZ_SLOT, x);
        lz_st2(a + 6 * LZ_SLOT, f2v_neg(r1.c0)); lz_st2(a + 8 * LZ_SLOT, f2v_neg(r1.c1)); lz_st2(a + 10 * LZ_SLOT, f2v_neg(r1.c2));
    }
}
#define LZ_A 0
#define LZ_X 12
#define LZ_Y 18
// A <- g^u for the cyclotomic element g = *ga (global), by the width-3 NAF of u (bn254.cuh f12_pow_u: same products in the same order);
// *ga3 (global scratch) receives g^3.
LZ_INL void lz_pow_u(const fp12* ga, fp12* ga3) {
    const uint32_t tid = lz_tid(), A = tid + LZ_A * LZ_SLOT, X = tid + LZ_X * LZ_SLOT, Y = tid + LZ_Y * LZ_SLOT, L = tid + LZ_L * LZ_SLOT;
    lz_ldg12(A, ga);
    lz_cyc_sqr(A, L); lz_f12mul_g(A, X, Y, ga, false);
    lz_stg12(ga3, A);
    if (C_U_WNAF3[ZKV_U_WNAF3_LEN - 1] == 1) lz_ldg12(A, ga);
    for (int i = ZKV_U_WNAF3_LEN - 2; i >= 0; i--) {
        lz_cyc_sqr(A, L);
        const int d = C_U_WNAF3[i];
        if (d) lz_f12mul_g(A, X, Y, (d == 1 || d == -1) ? ga : ga3, d < 0);
    }
}
// The final exponentiation of bn254.cuh final_exp in the same four stages as final_exp_stage0..3, on slots; st[0..5] = six Fp12 of global
// state per proof (f, scratch, x, y, z, t).  Stage 0 reads the Miller value *m, stage 3 leaves the result in the accumulator slots.
LZ_INL void lz_final_exp_stage(int stage, const fp12* m, fp12* st) {
    const uint32_t tid = lz_tid(), A = tid + LZ_A * LZ_SLOT, X = tid + LZ_X * LZ_SLOT, Y = tid + LZ_Y * LZ_SLOT, L = tid + LZ_L * LZ_SLOT;
    fp12 *f = st, *s1 = st + 1, *x = st + 2, *y = st + 3, *z = st + 4, *t = st + 5;
    if (stage == 0) {
        lz_ldg12(A, m); lz_f12inv(A, X, Y); lz_f12mul_g(A, X, Y, m, true);       // m^(p^6 - 1) = conj(m) / m
        lz_stg12(f, A); lz_frob(A, 2); lz_f12mul_g(A, X, Y, f, false);           // f = that^(p^2 + 1)
        lz_stg12(f, A);
        lz_pow_u(f, s1);                                                         // f^u
        lz_stg12(t, A);
    } else if (stage == 1) {
        lz_ldg12(A, t);
        lz_cyc_sqr(A, L); lz_stg12(x, A);                                        // x = f^(2u)
        lz_cyc_sqr(A, L); lz_f12mul_g(A, X, Y, x, false); lz_stg12(y, A);        // y = f^(6u)
        lz_pow_u(y, s1); lz_stg12(z, A);                                         // z = f^(6u^2)
    } else if (stage == 2) {
        lz_ldg12(A, z);
        lz_cyc_sqr(A, L); lz_stg12(t, A);
        lz_pow_u(t, s1);                                                         // f^(12u^3)
        lz_stg12(t, A);
    } else {
        lz_ldg12(A, t);
        lz_f12mul_g(A, X, Y, z, false); lz_f12mul_g(A, X, Y, y, false); lz_stg12(t, A);       // t = a = f^(12u^3 + 6u^2 + 6u)
        lz_f12mul_g(A, X, Y, x, true); lz_stg12(s1, A);                                        // s1 = b = a f^(-2u)
        lz_frob(A, 1); lz_stg12(x, A);                                                         // x = b^p
        lz_ldg12(A, s1); lz_f12mul_g(A, X, Y, f, true); lz_frob(A, 3); lz_stg12(s1, A);        // s1 = (b / f)^(p^3)
        lz_ldg12(A, t); lz_frob(A, 2); lz_stg12(y, A);                                         // y = a^(p^2)
        lz_ldg12(A, t); lz_f12mul_g(A, X, Y, z, false); lz_f12mul_g(A, X, Y, f, false);        // a f^(6u^2) f
        lz_f12mul_g(A, X, Y, x, false); lz_f12mul_g(A, X, Y, y, false); lz_f12mul_g(A, X, Y, s1, false);
    }
}

}  // namespace zkv
