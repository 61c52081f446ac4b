// sm_100a kernels of the batched Groth16 verification pipeline, one proof per thread.
// Stage map (SURVEY.md section 2.1a): K1 decode/validate, K3/K4 public-input hashing, K5 vk_x,
// K2 G2 membership, K6 multi-Miller loop, K7 final exponentiation + K8 status.
// Reference control flow being reproduced: /root/reference/contracts/src/common/groth16.rs:23-128,
// risc0/verifier.rs:146-197, sp1/verifier.rs:58-111; precompile semantics per EIP-196/197.
#pragma once
#include "bn254.cuh"
#include "lazy.cuh"
#include "sha256.cuh"

namespace zkv {

enum : uint8_t { F_INVALID = 1, F_SKIP0 = 2, F_SKIPC = 4, F_SKIPX = 8, F_SELMIS = 16, F_BADDATA = 32 };   // (the pairing service reuses 0x20..0x80 as its own skip bits)
enum : uint8_t { ST_OK = 0, ST_INVALID_INITIALIZATION = 1, ST_INVALID_PROOF_DATA = 2, ST_SELECTOR_MISMATCH = 3, ST_VERIFICATION_FAILED = 4 };

// rejection status of a verification-path proof from its flags: the order of risc0/verifier.rs:151-170 and sp1/verifier.rs:64-83
// (length < 4 -> InvalidProofData, selector, length != 260 -> InvalidProofData; k_decode sets exactly one of F_BADDATA / F_SELMIS)
__device__ __forceinline__ uint8_t reject_status(uint8_t fl) { return (fl & F_BADDATA) ? ST_INVALID_PROOF_DATA : (fl & F_SELMIS) ? ST_SELECTOR_MISMATCH : ST_VERIFICATION_FAILED; }
#define F_REJECT (F_INVALID | F_SELMIS | F_BADDATA)

#define ZKV_WIN_BITS 4
#define ZKV_WIN_PER_SCALAR 64          /* 256 / 4 */
#define ZKV_WIN_ENTRIES 15             /* d = 1..15 */

struct g1aff { fp x, y; };             // (0,0) encodes infinity (not on the curve, so unambiguous)

// ---------------------------------------------------------------------------- decode helpers
// EIP-196 G1 decoding from raw limbs: returns 0 valid point (Montgomery x,y), 1 infinity, 2 invalid
__device__ __forceinline__ int g1_decode_raw(fp& x, fp& y, const uint32_t* rx, const uint32_t* ry) {
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
// EIP-197 G2 decoding (wire order x_im, x_re, y_im, y_re), WITHOUT the subgroup test
__device__ __forceinline__ int g2_decode_bytes(fp2& x, fp2& y, const uint8_t* b) {
    uint32_t r[4][8]; uint32_t any = 0; bool big = false;
    for (int k = 0; k < 4; k++) { be32_to_raw(r[k], b + 32 * k); big |= u256_geq(r[k], C_P); for (int i = 0; i < 8; i++) any |= r[k][i]; }
    if (big) return 2;
    if (!any) { x = f2_zero(); y = f2_zero(); return 1; }
    fp t;
    for (int i = 0; i < 8; i++) t.v[i] = r[0][i]; fp_to_mont(x.c1, t);
    for (int i = 0; i < 8; i++) t.v[i] = r[1][i]; fp_to_mont(x.c0, t);
    for (int i = 0; i < 8; i++) t.v[i] = r[2][i]; fp_to_mont(y.c1, t);
    for (int i = 0; i < 8; i++) t.v[i] = r[3][i]; fp_to_mont(y.c0, t);
    return g2_on_curve(x, y) ? 0 : 2;
}

// K1: decode (a, b, c) of one proof record.  Fixed-stride records: rec i at recs + i * stride.  Variable records (rec_off != nullptr: the
// caller's concatenated seals / proofs uploaded as they are): rec i = recs + rec_off[i] - rec_base, length rec_off[i+1] - rec_off[i], and
// the front checks of risc0/verifier.rs:151-170 / sp1/verifier.rs:64-83 happen HERE, in the reference's order: length < 4 ->
// InvalidProofData, selector mismatch, length - 4 != 256 -> InvalidProofData (strict abi_decode of 8 x uint256).  rec + off points at
// 8 x BE-32.  vm == RISC0 applies negate_g1 exactly as groth16.rs:75-84 does: on the raw 256-bit words, BEFORE any range check.
// a record that never reaches the Groth16 stage: harmless operands for the uniform kernels behind, and its reject flag
__device__ __forceinline__ void decode_reject(int i, uint8_t fl, fp* ax, fp* ay, fp2* bx, fp2* by, fp* cx, fp* cy, uint8_t* flags) {
    ax[i] = fp_zero(); ay[i] = fp_zero(); cx[i] = fp_zero(); cy[i] = fp_zero(); bx[i] = f2_zero(); by[i] = f2_zero();
    flags[i] = fl | F_SKIP0 | F_SKIPC;
}
// (a, b, c) of the 8 x BE-32 words at p into slot i (k_decode and k_decode_keys)
__device__ __forceinline__ void decode_points(int i, const uint8_t* p, int vm, fp* ax, fp* ay, fp2* bx, fp2* by, fp* cx, fp* cy, uint8_t* flags) {
    uint8_t fl = 0;
    uint32_t rx[8], ry[8];
    be32_to_raw(rx, p); be32_to_raw(ry, p + 32);
    if (vm == 0) {
        uint32_t any = 0;
        for (int k = 0; k < 8; k++) any |= rx[k] | ry[k];
        if (any) {   // y = Q.wrapping_sub(y)  (mod 2^256)
            uint32_t bo = 0;
            for (int k = 0; k < 8; k++) { uint64_t d = (uint64_t)C_P[k] - ry[k] - bo; ry[k] = (uint32_t)d; bo = (uint32_t)(d >> 63); }
        }
    }
    fp x, y;
    int ra = g1_decode_raw(x, y, rx, ry);
    ax[i] = x; ay[i] = y;
    be32_to_raw(rx, p + 192); be32_to_raw(ry, p + 224);
    int rc = g1_decode_raw(x, y, rx, ry);
    cx[i] = x; cy[i] = y;
    fp2 qx, qy;
    int rb = g2_decode_bytes(qx, qy, p + 64);
    bx[i] = qx; by[i] = qy;
    if (ra == 2 || rb == 2 || rc == 2) fl |= F_INVALID;
    if (ra == 1 || rb == 1) fl |= F_SKIP0;
    if (rc == 1) fl |= F_SKIPC;
    flags[i] = fl;
}
__global__ void k_decode(int n, const uint8_t* recs, size_t stride, size_t off, uint32_t selector_le, int check_selector, int vm,
                         const uint64_t* rec_off, uint64_t rec_base,
                         fp* ax, fp* ay, fp2* bx, fp2* by, fp* cx, fp* cy, uint8_t* flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t* rec = rec_off ? recs + (size_t)(rec_off[i] - rec_base) : recs + (size_t)i * stride;
    const uint64_t len = rec_off ? rec_off[i + 1] - rec_off[i] : (uint64_t)stride;
    uint8_t fl = 0;
    if (rec_off && len < 4) fl = F_BADDATA;
    else if (check_selector) {
        uint32_t s = (uint32_t)rec[0] | (uint32_t)rec[1] << 8 | (uint32_t)rec[2] << 16 | (uint32_t)rec[3] << 24;
        if (s != selector_le) fl = F_SELMIS;
    }
    if (rec_off && !fl && len != off + 256) fl = F_BADDATA;
    if (fl) { decode_reject(i, fl, ax, ay, bx, by, cx, cy, flags); return; }
    decode_points(i, rec + off, vm, ax, ay, bx, by, cx, cy, flags);
}

// K3: RISC Zero public signals 2 and 3 (risc0/verifier.rs:172-179 + crypto.rs:103-110 split_digest):
// claim_lo / claim_hi are the little-endian readings of claim[0..16) / claim[16..32).
// mode 0: claim = ReceiptClaim::ok(image_id, journal).digest(); mode 1: claim digest supplied (verify_integrity).
struct Risc0HashConsts { uint32_t tag_out[8], claim_mid[8], sys0[8]; };
__global__ void k_risc0_signals(int n, const uint8_t* image_ids, const uint8_t* journals, const uint8_t* claims, int mode,
                                Risc0HashConsts hc, uint32_t* scal /* [n][2][8] */) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t claim[8];
    if (mode == 0) {
        uint32_t im[8], jr[8];
        for (int k = 0; k < 8; k++) { im[k] = load_be32(image_ids + 32 * (size_t)i + 4 * k); jr[k] = load_be32(journals + 32 * (size_t)i + 4 * k); }
        risc0_claim_digest(claim, im, jr, hc.tag_out, hc.claim_mid, hc.sys0);
    } else {
        for (int k = 0; k < 8; k++) claim[k] = load_be32(claims + 32 * (size_t)i + 4 * k);
    }
    uint32_t* o = scal + (size_t)i * 16;
    for (int k = 0; k < 4; k++) { o[k] = __byte_perm(claim[k], 0, 0x0123); o[8 + k] = __byte_perm(claim[4 + k], 0, 0x0123); o[4 + k] = 0; o[12 + k] = 0; }
}

// K4: SP1 public signals (sp1/types.rs:21-38): s0 = U256_be(program_vkey), s1 = SHA256(pv) & (2^253 - 1).
// A signal >= R makes the proof fail (groth16.rs:32-34); only s0 can be.
__global__ void k_sp1_signals(int n, const uint8_t* vkeys, const uint8_t* pv, const uint64_t* pv_off, uint64_t pv_base, size_t pv_stride,
                              uint32_t* scal /* [n][2][8] */, uint8_t* flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t* o = scal + (size_t)i * 16;
    uint32_t s0[8];
    be32_to_raw(s0, vkeys + 32 * (size_t)i);
    if (u256_geq(s0, C_R)) flags[i] |= F_INVALID;
    for (int k = 0; k < 8; k++) o[k] = s0[k];
    const uint8_t* msg; size_t len;
    if (pv_off) { msg = pv + (size_t)(pv_off[i] - pv_base); len = (size_t)(pv_off[i + 1] - pv_off[i]); } else { msg = pv + (size_t)i * pv_stride; len = pv_stride; }
    uint32_t h[8];
    sha256_msg(h, msg, len);
    h[0] &= 0x1fffffffu;
    for (int k = 0; k < 8; k++) o[8 + k] = h[7 - k];
}

// generic signals: n x k x BE-32 -> limbs; any signal >= R invalidates the proof (groth16.rs:32-34)
__global__ void k_generic_signals(int n, int k, const uint8_t* sig, uint32_t* scal, uint8_t* flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool bad = false;
    for (int j = 0; j < k; j++) {
        uint32_t s[8];
        be32_to_raw(s, sig + ((size_t)i * k + j) * 32);
        bad |= u256_geq(s, C_R);
        for (int t = 0; t < 8; t++) scal[((size_t)i * k + j) * 8 + t] = s[t];
    }
    if (bad) flags[i] |= F_INVALID;
}

// K5: vk_x = base + sum_t s_t * IC_t from 4-bit fixed-base window tables (compute_vk_x, groth16.rs:51-58,
// i.e. the k ecMul + k ecAdd precompile calls).  tab[t][w][d-1] = d * 16^w * IC_t (affine, Montgomery).
// vk_x of slot i: its `ns` scalars start at scal + i * stride * 8 (k_vkx: stride = ns; k_vkx_keys: the set's widest key)
__device__ __forceinline__ void vkx_one(int i, const uint32_t* scal, int stride, int ns, int nwin, const g1aff* tab, const g1aff& base, fp* vx, fp* vy, uint8_t* flags) {
    g1j acc;
    if (fp_is_zero(base.x) && fp_is_zero(base.y)) { acc.x = fp_one(); acc.y = fp_one(); acc.z = fp_zero(); }
    else { acc.x = base.x; acc.y = base.y; acc.z = fp_one(); }
    for (int t = 0; t < ns; t++) {
        const uint32_t* s = scal + ((size_t)i * stride + t) * 8;
        const g1aff* tt = tab + (size_t)t * ZKV_WIN_PER_SCALAR * ZKV_WIN_ENTRIES;
        for (int w = 0; w < nwin; w++) {
            uint32_t d = (s[w >> 3] >> ((w & 7) * 4)) & 15u;
            if (d) {
                const g1aff* e = tt + w * ZKV_WIN_ENTRIES + (d - 1);
                fp ex = e->x, ey = e->y;
                if (!(fp_is_zero(ex) && fp_is_zero(ey))) g1_add_affine(acc, ex, ey);
            }
        }
    }
    fp x, y;
    bool fin = g1_to_affine(x, y, acc);
    vx[i] = x; vy[i] = y;
    if (!fin && flags) flags[i] |= F_SKIPX;
}
__global__ void k_vkx(int n, const uint32_t* scal, int ns, int nwin, const g1aff* tab, g1aff base, fp* vx, fp* vy, uint8_t* flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    vkx_one(i, scal, ns, ns, nwin, tab, base, vx, vy, flags);
}

// K2: order-r membership of B (EIP-197; the reference reaches it through ecPairing, groth16.rs:121-125)
// g2_in_subgroup of bn254.cuh with the running point in REGISTERS and the Fp2 products through the by-value multiplier of lazy.cuh
// (f2v_mul / f2v_sqr: operands and results in registers, one copy of the code): the pointer-passing form keeps every Fp2 value in a
// 2.9 KB per-thread stack frame.  Same formulas in the same order (g2_dbl, g2_add_affine with its special cases), so the same accept set
// and the same intermediate values; the tail ([u+1]Q + psi + psi^2 against psi^3 of [2u]Q) runs through the bn254.cuh routines.
#if defined(__CUDACC__)
__device__ __noinline__ bool g2v_in_subgroup(fp2 qx, fp2 qy) {
    fp2 X = qx, Y = qy, Z = f2_one();
    const fp2 ny = f2v_neg(qy);
    for (int i = ZKV_U_NAF_LEN - 2; i >= 0; i--) {
        {   // doubling (g2_dbl)
            fp2 A = f2v_sqr(X), B = f2v_sqr(Y), C = f2v_sqr(B);
            fp2 D = f2v_dbl(f2v_sub(f2v_sub(f2v_sqr(f2v_add(X, B)), A), C));
            fp2 E = f2v_add(f2v_dbl(A), A), F = f2v_sqr(E);
            fp2 X3 = f2v_sub(F, f2v_dbl(D));
            fp2 Y3 = f2v_sub(f2v_mul(E, f2v_sub(D, X3)), f2v_dbl(f2v_dbl(f2v_dbl(C))));
            Z = f2v_dbl(f2v_mul(Y, Z)); X = X3; Y = Y3;
        }
        const int d = C_U_NAF[i];
        if (d) {    // mixed addition of +-Q (g2_add_affine)
            const fp2 ay = d > 0 ? qy : ny;
            if (f2_is_zero(Z)) { X = qx; Y = ay; Z = f2_one(); continue; }
            fp2 z1z1 = f2v_sqr(Z), u2 = f2v_mul(qx, z1z1), s2 = f2v_mul(f2v_mul(ay, Z), z1z1);
            fp2 h = f2v_sub(u2, X), rr = f2v_sub(s2, Y);
            if (f2_is_zero(h)) {
                if (f2_is_zero(rr)) { g2j p, r; p.x = X; p.y = Y; p.z = Z; g2_dbl(r, p); X = r.x; Y = r.y; Z = r.z; }
                else { X = f2_one(); Y = f2_one(); Z = f2_zero(); }
                continue;
            }
            fp2 hh = f2v_sqr(h), hhh = f2v_mul(hh, h), v = f2v_mul(X, hh);
            fp2 X3 = f2v_sub(f2v_sub(f2v_sqr(rr), hhh), f2v_dbl(v));
            fp2 Y3 = f2v_sub(f2v_mul(rr, f2v_sub(v, X3)), f2v_mul(Y, hhh));
            Z = f2v_mul(Z, h); X = X3; Y = Y3;
        }
    }
    g2j q, uq, lhs, t, p1, p2, p3;
    q.x = qx; q.y = qy; q.z = f2_one(); uq.x = X; uq.y = Y; uq.z = Z;
    g2_add(lhs, uq, q);
    g2_psi(p1, uq, 1); g2_add(t, lhs, p1); lhs = t;
    g2_psi(p2, uq, 2); g2_add(t, lhs, p2); lhs = t;
    g2_dbl(t, uq); g2_psi(p3, t, 3);
    return g2j_eq(lhs, p3);
}
#else
static inline bool g2v_in_subgroup(fp2 qx, fp2 qy) { return g2_in_subgroup(qx, qy); }
#endif
// (four blocks per SM at 128 registers were measured: the spills cost more than the second wave they save, 2.80 against 2.59 ms per 2^16)
__global__ void k_g2_check(int n, const fp2* bx, const fp2* by, uint8_t* flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t fl = flags[i];
    if (fl & F_REJECT) return;
    fp2 x = bx[i], y = by[i];
    if (f2_is_zero(x) && f2_is_zero(y)) return;      // infinity is a member
    if (!g2v_in_subgroup(x, y)) flags[i] = fl | F_INVALID;
}
// K2 of the shared-memory verification path (k_miller_lz, k_miller_lz_keys): T = -psi^3(B), against which the last Miller segment compares
// its R (lz_r_is), so the subgroup test costs a Frobenius map here and two Fp2 products there instead of k_g2_check's ~1 800 Fp products
__global__ void k_g2_target(int n, const fp2* bx, const fp2* by, fp2* tx, fp2* ty) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fp2 x = bx[i], y = by[i];
    g2_neg_psi3(x, y);
    tx[i] = x; ty[i] = y;
}

// flags[i] |= extra[i] (vk_x's flag bits when it ran beside the G2 check on a scratch array)
__global__ void k_or_flags(int n, uint8_t* flags, const uint8_t* extra) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && extra[i]) flags[i] |= extra[i];
}

// K6: multi-Miller loop.  Pair 0 = (px[0], variable G2); pairs 1..nfixed = (px[j], fixed G2 with line table tabs[j-1]).
// If pre != nullptr the result is multiplied by that constant (Miller(alpha, beta), precomputed per vk).
struct MillerArgs {
    const fp* px[4]; const fp* py[4];
    const fp2* qx; const fp2* qy;
    const line_t* tabs[3];
    int nfixed;
    const nline_t* ntabs[2];  // verification path: normalised tables of gamma and delta (bn254.cuh), used by k_miller_norm
    const fp12* pre;
    uint8_t skip_bit[4];      // which flag bit disables pair j (0 = never)
    uint8_t vk_skip;          // pairs disabled for the whole batch (a vk G2 point at infinity)
};
// Launch shape of the two heavy kernels: blocks whose warps start together, run the same instruction stream and meet at the
// rendezvous points of bn254.cuh, so they share instruction-cache lines; two such blocks per SM run out of phase with each
// other, which lets one block's integer-multiply bursts overlap the other's carry / load phases.
#ifndef ZKV_HTPB
#define ZKV_HTPB 128
#endif
#ifndef ZKV_MINBLOCKS
#define ZKV_MINBLOCKS 2
#endif
// The verification Miller-loop kernels (k_miller_norm, k_miller_norm_seg) run three blocks per SM (168 registers): measured on whole
// waves, -4 % per proof against two blocks; the final exponentiation (more live Fp12 values) is 6 % slower at three and stays at two.
#ifndef ZKV_MINBLOCKS_MILLER
#define ZKV_MINBLOCKS_MILLER 3
#endif
#ifndef ZKV_HTPB_MILLER
#define ZKV_HTPB_MILLER ZKV_HTPB
#endif
#ifndef ZKV_HTPB_FE
#define ZKV_HTPB_FE ZKV_HTPB
#endif
#ifndef ZKV_MINBLOCKS_FE
#define ZKV_MINBLOCKS_FE ZKV_MINBLOCKS
#endif
__global__ void __launch_bounds__(ZKV_HTPB, ZKV_MINBLOCKS) k_miller(int n, MillerArgs a, const uint8_t* flags, fp12* out) {
    int i0 = blockIdx.x * blockDim.x + threadIdx.x;
    int i = i0 < n ? i0 : n - 1;                      // surplus threads redo the last proof (every thread reaches every rendezvous)
    uint8_t fl = flags[i];
    uint32_t skip = a.vk_skip;
    for (int j = 0; j <= a.nfixed; j++) if (fl & a.skip_bit[j]) skip |= 1u << j;
    if (fl & (F_INVALID | F_SELMIS)) skip = 0xF;      // result is never used: every factor is replaced by 1 (the work is still done: uniform control flow)
    fp px[4], py[4];
    for (int j = 0; j <= a.nfixed; j++) { px[j] = a.px[j][i]; py[j] = a.py[j][i]; }
    fp2 qx = a.qx[i], qy = a.qy[i];
    fp12 f;
    miller_loop(f, px, py, qx, qy, a.tabs, a.nfixed, skip);
    if (a.pre) { fp12 p = *a.pre; f12_mul(f, f, p); }
    if (i0 < n) out[i] = f;
}

// K6 for the verification entry points: pairs (A', B), (vk_x, gamma), (C, delta) with the NORMALISED gamma / delta tables (bn254.cuh),
// times the per-key constant Miller(alpha, beta).  Same launch shape and flag conventions as k_miller.
__global__ void __launch_bounds__(ZKV_HTPB_MILLER, ZKV_MINBLOCKS_MILLER) k_miller_norm(int n, MillerArgs a, const uint8_t* flags, fp12* out) {
    int i0 = blockIdx.x * blockDim.x + threadIdx.x;
    int i = i0 < n ? i0 : n - 1;
    uint8_t fl = flags[i];
    uint32_t skip = a.vk_skip;
    for (int j = 0; j < 3; j++) if (fl & a.skip_bit[j]) skip |= 1u << j;
    if (fl & F_REJECT) skip = 0xF;
    fp x12[2] = {a.px[1][i], a.px[2][i]}, y12[2] = {a.py[1][i], a.py[2][i]}, xy[2], iy[2];
    bool off[2] = {(skip & 2u) != 0, (skip & 4u) != 0};
    g1_slopes2(xy, iy, x12, y12, off);
    fp px0 = a.px[0][i], py0 = a.py[0][i];
    fp2 qx = a.qx[i], qy = a.qy[i];
    fp12 f;
    miller_loop_norm(f, px0, py0, qx, qy, a.ntabs, xy, iy, (skip & 1u) != 0);
    if (a.pre) { fp12 p = *a.pre; f12_mul(f, f, p); }
    if (i0 < n) out[i] = f;
}

// Segment form of k_miller_norm: digits d_hi .. d_lo of the loop; f (in `fio`) and R (in `rst`) are carried in HBM between segments, the
// slopes of the two fixed pairs are computed by the first segment and kept in `sl` (4 Fp per proof).
__global__ void __launch_bounds__(ZKV_HTPB_MILLER, ZKV_MINBLOCKS_MILLER) k_miller_norm_seg(int n, MillerArgs a, const uint8_t* flags, fp12* fio, g2j* rst, fp* sl,
                                                                              int d_hi, int d_lo, int first, int last) {
    int i0 = blockIdx.x * blockDim.x + threadIdx.x;
    int i = i0 < n ? i0 : n - 1;
    uint8_t fl = flags[i];
    uint32_t skip = a.vk_skip;
    for (int j = 0; j < 3; j++) if (fl & a.skip_bit[j]) skip |= 1u << j;
    if (fl & F_REJECT) skip = 0xF;
    fp xy[2], iy[2];
    if (first) {
        fp x12[2] = {a.px[1][i], a.px[2][i]}, y12[2] = {a.py[1][i], a.py[2][i]};
        bool off[2] = {(skip & 2u) != 0, (skip & 4u) != 0};
        g1_slopes2(xy, iy, x12, y12, off);
        if (i0 < n && !last) { sl[4 * (size_t)i] = xy[0]; sl[4 * (size_t)i + 1] = xy[1]; sl[4 * (size_t)i + 2] = iy[0]; sl[4 * (size_t)i + 3] = iy[1]; }
    } else {
        xy[0] = sl[4 * (size_t)i]; xy[1] = sl[4 * (size_t)i + 1]; iy[0] = sl[4 * (size_t)i + 2]; iy[1] = sl[4 * (size_t)i + 3];
    }
    fp px0 = a.px[0][i], py0 = a.py[0][i];
    fp2 qx = a.qx[i], qy = a.qy[i];
    fp12 f; g2j R;
    if (first) { f = f12_one(); R.x = qx; R.y = qy; R.z = f2_one(); }
    else { f = fio[i]; R = rst[i]; }
    miller_loop_norm_seg(f, R, px0, py0, qx, qy, a.ntabs, xy, iy, (skip & 1u) != 0, d_hi, d_lo, last != 0);
    if (last) { if (a.pre) { fp12 p = *a.pre; f12_mul(f, f, p); } }
    else if (i0 < n) rst[i] = R;
    if (i0 < n) fio[i] = f;
}

// K7 + K8: final exponentiation, is-one test and status byte
__global__ void __launch_bounds__(ZKV_HTPB_FE, ZKV_MINBLOCKS_FE) k_final_exp(int n, const fp12* in, const uint8_t* flags, uint8_t* status, uint8_t* gt_out, int pairing_mode) {
    int i0 = blockIdx.x * blockDim.x + threadIdx.x;
    int i = i0 < n ? i0 : n - 1;
    uint8_t fl = flags[i];
    fp12 m = in[i], gt;
    final_exp(gt, m);                                 // every thread runs it (k_miller left a harmless value for rejected inputs): uniform control flow
    if (i0 >= n) return;
    if (fl & (pairing_mode ? (F_INVALID | F_SELMIS) : F_REJECT)) {
        status[i] = pairing_mode ? 2 : reject_status(fl);
        if (gt_out) for (int k = 0; k < 384; k++) gt_out[(size_t)i * 384 + k] = 0;
        return;
    }
    bool one = f12_is_one(gt);
    status[i] = pairing_mode ? (one ? 1 : 0) : (one ? ST_OK : ST_VERIFICATION_FAILED);
    if (gt_out) f12_to_bytes(gt_out + (size_t)i * 384, gt);
}
// Staged form of k_final_exp (bn254.cuh final_exp_stage0..3): the state (f, x, y, z, t1; slot 1 first holds t = f^u) lives in `st`, five
// Fp12 per proof, so that the three exponentiations by u of different chunks can interleave.  Stage 3 writes the status like k_final_exp.
__global__ void __launch_bounds__(ZKV_HTPB_FE, ZKV_MINBLOCKS_FE) k_final_exp_stage(int n, int stage, const fp12* in, fp12* st, const uint8_t* flags, uint8_t* status) {
    int i0 = blockIdx.x * blockDim.x + threadIdx.x;
    int i = i0 < n ? i0 : n - 1;
    const bool w = i0 < n;
    fp12* s = st + 5 * (size_t)i;
    if (stage == 0) {
        fp12 m = in[i], f, t;
        final_exp_stage0(f, t, m);
        if (w) { s[0] = f; s[1] = t; }
    } else if (stage == 1) {
        fp12 t = s[1], x, y, z;
        final_exp_stage1(x, y, z, t);
        if (w) { s[1] = x; s[2] = y; s[3] = z; }
    } else if (stage == 2) {
        fp12 z = s[3], t1;
        final_exp_stage2(t1, z);
        if (w) s[4] = t1;
    } else {
        fp12 f = s[0], x = s[1], y = s[2], z = s[3], t1 = s[4], gt;
        final_exp_stage3(gt, f, x, y, z, t1);
        if (!w) return;
        uint8_t fl = flags[i];
        if (fl & F_REJECT) { status[i] = reject_status(fl); return; }
        status[i] = f12_is_one(gt) ? ST_OK : ST_VERIFICATION_FAILED;
    }
}
// ---------------------------------------------------------------------------- shared-memory-resident forms of K6 / K7 (csrc/lazy.cuh)
// Same inputs, outputs and flag conventions as k_miller_norm_seg / k_final_exp_stage; the working set of a proof (f, R, temporaries: 28 Fp
// slots = 896 B) lives in shared memory, two blocks of LZ_NT = 128 threads per SM, the Fp6-level products are lazily reduced.  The state
// between segments / stages travels through HBM exactly as in the round-1 kernels.  `sl` must have room for 4 Fp per LAUNCHED thread
// (surplus threads of the last block park their slopes behind the batch).
#define LZ_SMEM_BYTES (LZ_SLOTS * 32 * LZ_NT)
#define LZ_SMEM_MILLER (LZ_SMEM_BYTES + 1024)      /* + the per-warp line staging areas of lz_fixed_lines: 2 x (112 KB + 1 KB + 1 KB reserved) = the SM's 228 KB */
// slopes of the two fixed pairs (g1_slopes2) written to sl[0..3] = xy0, xy1, iy0, iy1; out of line so that its arrays have a frame of their own
__device__ __noinline__ void lz_slopes_to(fp* sl, const fp* x1, const fp* y1, const fp* x2, const fp* y2, bool off1, bool off2) {
    fp x12[2] = {*x1, *x2}, y12[2] = {*y1, *y2}, xy[2], iy[2];
    bool off[2] = {off1, off2};
    g1_slopes2(xy, iy, x12, y12, off);
    sl[0] = xy[0]; sl[1] = xy[1]; sl[2] = iy[0]; sl[3] = iy[1];
}
// body of k_miller_lz / k_miller_lz_keys; the key's tables (nt0, nt1: normalised gamma / delta lines, pre = Miller(alpha, beta)) and its
// disabled pairs come in separately, the rest from `a`.  The last segment also finishes the subgroup test of B against T = (tx, ty)
// (k_g2_target) and ORs F_INVALID into the proof's flag byte when it fails; R runs through every step whatever the skip bits say.
__device__ __forceinline__ void miller_lz(int n, const MillerArgs& a, const nline_t* nt0, const nline_t* nt1, const fp12* pre, uint8_t vk_skip,
                                          uint8_t* flags, const fp2* tx, const fp2* ty, fp12* fio, g2j* rst, fp* sl, int d_hi, int d_lo, int first, int last) {
    const int i0 = blockIdx.x * LZ_NT + threadIdx.x, i = i0 < n ? i0 : n - 1;
    const uint8_t fl = flags[i];
    uint32_t skip = vk_skip;
    for (int j = 0; j < 3; j++) if (fl & a.skip_bit[j]) skip |= 1u << j;
    if (fl & F_REJECT) skip = 0xF;
    fp* mysl = sl + 4 * (size_t)i0;
    if (first) lz_slopes_to(mysl, a.px[1] + i, a.py[1] + i, a.px[2] + i, a.py[2] + i, (skip & 2u) != 0, (skip & 4u) != 0);
    LzMillerIn in;
    in.px0 = a.px[0] + i; in.py0 = a.py[0] + i; in.qx = a.qx + i; in.qy = a.qy + i; in.sl = mysl; in.nt[0] = nt0; in.nt[1] = nt1; in.var_off = (skip & 1u) != 0;
    const uint32_t tid = lz_tid();
    if (first) lz_miller_init(a.qx[i], a.qy[i]);
    else {
        lz_ldg12(tid + LZ_F * LZ_SLOT, fio + i);
        const g2j* R = rst + i;
        lz_st2(tid + LZ_R * LZ_SLOT, R->x); lz_st2(tid + (LZ_R + 2) * LZ_SLOT, R->y); lz_st2(tid + (LZ_R + 4) * LZ_SLOT, R->z);
    }
    lz_miller_norm_seg(in, d_hi, d_lo, last != 0);
    if (last && !lz_r_is(tid + LZ_R * LZ_SLOT, tx[i], ty[i]) && i0 < n) flags[i] = fl | F_INVALID;
    if (last) { if (pre) lz_f12mul_g(tid + LZ_F * LZ_SLOT, tid + LZ_T * LZ_SLOT, tid + LZ_R * LZ_SLOT, pre, false); }      // x Miller(alpha, beta); T and R are free now
    else if (i0 < n) { g2j* R = rst + i; R->x = lz_ld2(tid + LZ_R * LZ_SLOT); R->y = lz_ld2(tid + (LZ_R + 2) * LZ_SLOT); R->z = lz_ld2(tid + (LZ_R + 4) * LZ_SLOT); }
    if (i0 < n) lz_stg12(fio + i, tid + LZ_F * LZ_SLOT);
}
__global__ void __launch_bounds__(LZ_NT, 2) k_miller_lz(int n, MillerArgs a, uint8_t* flags, const fp2* tx, const fp2* ty, fp12* fio, g2j* rst, fp* sl, int d_hi, int d_lo, int first, int last) {
    miller_lz(n, a, a.ntabs[0], a.ntabs[1], a.pre, a.vk_skip, flags, tx, ty, fio, rst, sl, d_hi, d_lo, first, last);
}
// stages s_lo .. s_hi of the final exponentiation (0..3 = all of it in one launch); st = 6 Fp12 of state per LAUNCHED thread; the last stage writes the
// status (pairing_mode: 1 product is one / 0 it is not / 2 the call reverts) and, if gt_out is set, the value (12 x BE-32, zeroed for rejected inputs)
__device__ __forceinline__ void final_exp_lz(int n, int s_lo, int s_hi, const fp12* in, fp12* st, const uint8_t* flags, uint8_t* status, uint8_t* gt_out, int pairing_mode) {
    const int i0 = blockIdx.x * LZ_NT + threadIdx.x, i = i0 < n ? i0 : n - 1;
    for (int s = s_lo; s <= s_hi; s++) lz_final_exp_stage(s, in + i, st + 6 * (size_t)i0);
    if (s_hi < 3 || i0 >= n) return;
    const uint8_t fl = flags[i];
    if (fl & (pairing_mode ? (F_INVALID | F_SELMIS) : F_REJECT)) {
        status[i] = pairing_mode ? 2 : reject_status(fl);
        if (gt_out) for (int k = 0; k < 384; k++) gt_out[(size_t)i * 384 + k] = 0;
        return;
    }
    const uint32_t tid = lz_tid();
    fp one = fp_one(); uint32_t t = 0;
    for (int k = 0; k < 12; k++) {
        fp w = lz_ldfp(tid + (LZ_A + k) * LZ_SLOT);
        for (int j = 0; j < 8; j++) t |= w.v[j] ^ (k == 0 ? one.v[j] : 0u);
        if (gt_out) fp_to_be32(gt_out + (size_t)i * 384 + 32 * k, w);
    }
    status[i] = pairing_mode ? (t == 0 ? 1 : 0) : (t == 0 ? ST_OK : ST_VERIFICATION_FAILED);
}
__global__ void __launch_bounds__(LZ_NT, 2) k_final_exp_lz(int n, int s_lo, int s_hi, const fp12* in, fp12* st, const uint8_t* flags, uint8_t* status, uint8_t* gt_out, int pairing_mode) {
    final_exp_lz(n, s_lo, s_hi, in, st, flags, status, gt_out, pairing_mode);
}
// General multi-Miller loop (lz_miller_gen_seg): nvar variable pairs + nfix tabled pairs per instance, pair-major arrays of `in.stride`
// entries each (stride >= launched threads: surplus threads work on the padding, whose pskip bytes are 1).  iskip[i] != 0: the instance is
// not evaluated (invalid input): all its pairs are treated as skipped.
__global__ void __launch_bounds__(LZ_NT, 2) k_pairing_lz(int n, LzGenIn in, fp12* fio, int d_hi, int d_lo, int first, int last) {
    const size_t i = (size_t)blockIdx.x * LZ_NT + threadIdx.x;
    const uint32_t tid = lz_tid();
    if (first) { fp2 z = f2_zero(); lz_st2(tid + LZ_F * LZ_SLOT, f2_one()); for (int k = 1; k < 6; k++) lz_st2(tid + (LZ_F + 2 * k) * LZ_SLOT, z); }
    else lz_ldg12(tid + LZ_F * LZ_SLOT, fio + i);
    lz_miller_gen_seg(in, i, d_hi, d_lo, first != 0, last != 0);
    lz_stg12(fio + i, tid + LZ_F * LZ_SLOT);
    (void)n;
}
// pairing4 service: per-pair skip bytes for k_pairing_lz from the decode flags (pair 0: F_SKIP0, pairs 1..3: 0x20, 0x40, 0x80), the key's own
// points at infinity (vk_skip) and invalid instances (nothing is evaluated)
__global__ void k_pairing4_skip(int n, size_t stride, const uint8_t* flags, uint8_t vk_skip, uint8_t* pskip) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t fl = flags[i], bits[4] = {F_SKIP0, 0x20, 0x40, 0x80};
    const bool bad = (fl & (F_INVALID | F_SELMIS)) != 0;
    for (int j = 0; j < 4; j++) pskip[(size_t)j * stride + i] = (bad || (fl & bits[j]) || ((vk_skip >> j) & 1)) ? 1 : 0;
}
// decode for the general pairing service: one thread per (instance, pair); input record = G1 (64 B) || G2 (128 B) (EIP-197), instance-major
// in the input, pair-major in the outputs.  pst: 0 usable pair, F_SKIP0 a member is infinity (the pair contributes 1), F_INVALID bad encoding /
// off curve / off twist (the subgroup test comes after, k_g2_check on the same flags)
__global__ void k_pairing_decode(int n, int k, size_t stride, const uint8_t* in, fp* px, fp* py, fp2* qx, fp2* qy, uint8_t* pst) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)n * k) return;
    const size_t i = t / k; const int j = (int)(t % k);
    const uint8_t* p = in + (i * k + j) * 192;
    uint32_t rx[8], ry[8];
    be32_to_raw(rx, p); be32_to_raw(ry, p + 32);
    fp x, y; int r1 = g1_decode_raw(x, y, rx, ry);
    fp2 x2, y2; int r2 = g2_decode_bytes(x2, y2, p + 64);
    const size_t o = (size_t)j * stride + i;
    px[o] = x; py[o] = y; qx[o] = x2; qy[o] = y2;
    pst[o] = (r1 == 2 || r2 == 2) ? F_INVALID : (r1 == 1 || r2 == 1) ? F_SKIP0 : 0;
}
// per instance: invalid if any pair is; per pair: skip byte for the Miller kernel (every pair of an invalid instance is skipped)
__global__ void k_pairing_flags(int n, int k, size_t stride, const uint8_t* pst, uint8_t* pskip, uint8_t* iflags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t bad = 0;
    for (int j = 0; j < k; j++) bad |= pst[(size_t)j * stride + i] & F_INVALID;
    for (int j = 0; j < k; j++) pskip[(size_t)j * stride + i] = (bad || (pst[(size_t)j * stride + i] & F_SKIP0)) ? 1 : 0;
    iflags[i] = bad ? F_INVALID : 0;
}
// parity hook: one Fp12 tower operation per thread on byte operands (12 x BE-32 each, tower order).
// op 0: a*b  1: a^2  2: a * line(b.c0.c0, b.c0.c1, b.c0.c2)  3: cyclotomic square  4: 1/a  5..7: Frobenius^(op-4)  8: final exponentiation  9: single-pair Miller loop
__global__ void __launch_bounds__(ZKV_HTPB, ZKV_MINBLOCKS) k_fp12_op(int n, int op, const uint8_t* a, const uint8_t* b, uint8_t* out) {
    int i0 = blockIdx.x * blockDim.x + threadIdx.x;
    int i = i0 < n ? i0 : n - 1;                      // every thread runs the operation: the tower routines contain block-wide rendezvous
    fp12 x, y, z; fp* xw = &x.c0.c0.c0; fp* yw = &y.c0.c0.c0;
    for (int k = 0; k < 12; k++) {
        fp t; be32_to_raw(t.v, a + (size_t)i * 384 + 32 * k); fp_to_mont(xw[k], t);
        if (b) { be32_to_raw(t.v, b + (size_t)i * 384 + 32 * k); fp_to_mont(yw[k], t); } else yw[k] = fp_zero();
    }
    switch (op) {
        case 0: f12_mul(z, x, y); break;
        case 1: f12_sqr(z, x); break;
        case 2: z = x; f12_mul_line(z, y.c0.c0, y.c0.c1, y.c0.c2); break;
        case 3: f12_cyc_sqr(z, x); break;
        case 4: f12_inv(z, x); break;
        case 5: case 6: case 7: f12_frob(z, x, op - 4); break;
        case 8: final_exp(z, x); break;
        default: {                                    // op 9: Miller loop of one pair (P, Q) with a variable Q; b holds P.x, P.y, Q in wire order (x_im, x_re, y_im, y_re)
            fp px[1] = {yw[0]}, py[1] = {yw[1]}; fp2 qx, qy; qx.c1 = yw[2]; qx.c0 = yw[3]; qy.c1 = yw[4]; qy.c0 = yw[5];
            miller_loop(z, px, py, qx, qy, nullptr, 0, n > (1 << 30) ? 1u : 0u); break; }
    }
    if (i0 < n) f12_to_bytes(out + (size_t)i * 384, z);
}
// parity hook for the shared-memory-resident tower (lazy.cuh): the same operations as k_fp12_op (op 0..8) on slots, plus
// op 9: a * (1 + (c3 + c4 v) w) with c3, c4 = b's first two Fp2 (the normalised line product of the verification loop);
// op 10: the verification Miller loop (lz_miller_norm_seg, in three segments) of the single pair (P, Q) held in b like k_fp12_op's op 9, the
// two fixed pairs switched off (zero slopes, all-zero line tables `ztab`): the value must equal k_fp12_op's op 9 bit for bit.
__global__ void __launch_bounds__(LZ_NT, 2) k_lz_fp12_op(int n, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, fp12* scratch /* 7 Fp12 per launched thread */, const nline_t* ztab) {
    const int i0 = blockIdx.x * LZ_NT + threadIdx.x, i = i0 < n ? i0 : n - 1;
    const uint32_t tid = lz_tid(), A = tid + LZ_A * LZ_SLOT, X = tid + LZ_X * LZ_SLOT, Y = tid + LZ_Y * LZ_SLOT, L = tid + LZ_L * LZ_SLOT;
    fp12* my = scratch + 7 * (size_t)i0;
    {
        fp12 y; fp* yw = &y.c0.c0.c0;
        for (int k = 0; k < 12; k++) {
            fp t; be32_to_raw(t.v, a + (size_t)i * 384 + 32 * k); fp_to_mont(t, t); lz_stfp(A + k * LZ_SLOT, t);
            if (b) { be32_to_raw(t.v, b + (size_t)i * 384 + 32 * k); fp_to_mont(yw[k], t); } else yw[k] = fp_zero();
        }
        my[6] = y;
    }
    switch (op) {
        case 0: lz_f12mul_g(A, X, Y, my + 6, false); break;
        case 1: lz_f12sqr(A, X); break;
        case 2: { fp2 l0 = my[6].c0.c0; lz_st2(L, my[6].c0.c1); lz_st2(L + 2 * LZ_SLOT, my[6].c0.c2); lz_mul_line(A, X, L, l0); break; }
        case 3: lz_cyc_sqr(A, L); break;
        case 4: lz_f12inv(A, X, Y); break;
        case 5: case 6: case 7: lz_frob(A, op - 4); break;
        case 8: { lz_stg12(my + 6, A); for (int s = 0; s < 4; s++) lz_final_exp_stage(s, my + 6, my); break; }
        case 9: lz_st2(L, my[6].c0.c0); lz_st2(L + 2 * LZ_SLOT, my[6].c0.c1); lz_mul_nline(A, X, L); break;
        default: {
            const fp* yw = &my[6].c0.c0.c0;
            fp* g = &my[0].c0.c0.c0;                        // per-thread global scratch: px, py, slopes (4 x 0), qx, qy
            g[0] = yw[0]; g[1] = yw[1]; for (int k = 2; k < 6; k++) g[k] = fp_zero();
            fp2 qx, qy; qx.c1 = yw[2]; qx.c0 = yw[3]; qy.c1 = yw[4]; qy.c0 = yw[5];
            fp2* gq = (fp2*)(g + 6); gq[0] = qx; gq[1] = qy;
            LzMillerIn in; in.px0 = g; in.py0 = g + 1; in.sl = g + 2; in.qx = gq; in.qy = gq + 1; in.nt[0] = ztab; in.nt[1] = ztab; in.var_off = false;
            lz_miller_init(qx, qy);
            const int top = ZKV_ATE_NAF_LEN - 2;
            for (int k = 0; k < 3; k++) lz_miller_norm_seg(in, top - (top + 1) * k / 3, top - (top + 1) * (k + 1) / 3 + 1, k == 2);
            break; }
    }
    if (i0 < n) for (int k = 0; k < 12; k++) fp_to_be32(out + (size_t)i * 384 + 32 * k, lz_ldfp(A + k * LZ_SLOT));
}
__global__ void k_f12_to_bytes(int n, const fp12* in, uint8_t* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { fp12 t = in[i]; f12_to_bytes(out + (size_t)i * 384, t); }
}

// ---------------------------------------------------------------------------- per-vk setup (runs once per key per device)
struct VkDev {                 // device-resident, Montgomery form
    fp2 g2x[3], g2y[3];        // beta, gamma, delta
    fp alpha_x, alpha_y;
    int valid;                 // all key points decode under EIP-196/197 rules (else every verify fails)
    int g2_inf[3]; int alpha_inf;
    int norm_ok;               // the normalised gamma / delta line tables exist (no vanishing l0)
};
// block j<3 (one thread each) validates + tabulates G2 point j; block 3 validates alpha
__global__ void k_vk_setup(const uint8_t* alpha, const uint8_t* g2bytes /* 3 x 128 */, VkDev* vk, line_t* lines /* 3 x LINES */, nline_t* nlines /* 2 x LINES: gamma, delta */) {
    int j = blockIdx.x;
    if (j < 3) {
        fp2 x, y;
        int r = g2_decode_bytes(x, y, g2bytes + 128 * j);
        if (r == 0 && !g2_in_subgroup(x, y)) r = 2;
        vk->g2x[j] = x; vk->g2y[j] = y; vk->g2_inf[j] = (r == 1);
        if (r == 2) atomicAnd(&vk->valid, 0);
        if (r == 0) g2_precompute_lines(lines + (size_t)j * ZKV_LINES_PER_G2, x, y);
        if (j >= 1 && (r != 0 || !g2_normalise_lines(nlines + (size_t)(j - 1) * ZKV_LINES_PER_G2, lines + (size_t)j * ZKV_LINES_PER_G2, ZKV_LINES_PER_G2))) atomicAnd(&vk->norm_ok, 0);
    } else if (j == 3) {
        uint32_t rx[8], ry[8]; be32_to_raw(rx, alpha); be32_to_raw(ry, alpha + 32);
        fp x, y; int r = g1_decode_raw(x, y, rx, ry);
        vk->alpha_x = x; vk->alpha_y = y; vk->alpha_inf = (r == 1);
        if (r == 2) atomicAnd(&vk->valid, 0);
    }
}
// Miller(alpha, beta) with beta's line table
__global__ void k_vk_miller_ab(const VkDev* vk, const line_t* lines, fp12* out) {
    fp12 f;
    if (vk->alpha_inf || vk->g2_inf[0] || !vk->valid) { f = f12_one(); }
    else {
        fp px[2], py[2]; px[1] = vk->alpha_x; py[1] = vk->alpha_y; px[0] = fp_zero(); py[0] = fp_zero();
        const line_t* tabs[1] = {lines};
        fp2 z = f2_zero();
        miller_loop(f, px, py, z, z, tabs, 1, 1u);
    }
    *out = f;
}
// window tables: block t = IC point t+1 (ic bytes start at IC_1), thread w = window.  Also validates the points.
__global__ void k_ic_tables(const uint8_t* ic /* n_ic x 64, IC_0 first */, g1aff* tab, g1aff* ic0, VkDev* vk) {
    int t = blockIdx.x, w = threadIdx.x;
    uint32_t rx[8], ry[8];
    if (t == 0 && w == 0) {
        be32_to_raw(rx, ic); be32_to_raw(ry, ic + 32);
        fp x, y; int r = g1_decode_raw(x, y, rx, ry);
        if (r == 2) atomicAnd(&vk->valid, 0);
        ic0->x = x; ic0->y = y;
    }
    be32_to_raw(rx, ic + 64 * (t + 1)); be32_to_raw(ry, ic + 64 * (t + 1) + 32);
    fp x, y; int r = g1_decode_raw(x, y, rx, ry);
    if (r == 2 && w == 0) atomicAnd(&vk->valid, 0);
    g1aff* o = tab + ((size_t)t * ZKV_WIN_PER_SCALAR + w) * ZKV_WIN_ENTRIES;
    if (r != 0) { for (int d = 0; d < ZKV_WIN_ENTRIES; d++) { o[d].x = fp_zero(); o[d].y = fp_zero(); } return; }
    g1j b; b.x = x; b.y = y; b.z = fp_one();
    for (int k = 0; k < ZKV_WIN_BITS * w; k++) { g1j d; g1_dbl(d, b); b = d; }
    fp bx, by; g1_to_affine(bx, by, b);
    g1j acc; acc.x = fp_one(); acc.y = fp_one(); acc.z = fp_zero();
    for (int d = 0; d < ZKV_WIN_ENTRIES; d++) {
        g1_add_affine(acc, bx, by);
        fp ex, ey; g1_to_affine(ex, ey, acc);
        o[d].x = ex; o[d].y = ey;
    }
}

// ---------------------------------------------------------------------------- key sets (zkv_groth16_verify_batch_keys)
// A batch whose proofs name their own key is first GROUPED: slot s of the workspace holds caller record perm[s] of key slot_key[s], the
// proofs of one key occupy consecutive slots in caller order, and each key's group is padded to a multiple of 32 slots, so every warp of
// the Miller kernel works on ONE key (lz_fixed_lines stages a step's gamma / delta line entries once per warp).  Padding slots hold
// ZKV_SLOT_EMPTY and their group's key; slots behind the last group (the host sizes the workspace for the bound n + 31 x keys present)
// hold ZKV_SLOT_EMPTY and key 0, and the heavy kernels do not run them (the slot total is read on the device).
#define ZKV_MAX_KEYS 256
#define ZKV_GROUP_TILE 4096            /* caller records per block of the grouping kernels: 8 warps x 16 rounds of 32 */
#define ZKV_SLOT_EMPTY 0xffffffffu
struct KeyDesc {                       // one key of a set on one device (device memory)
    g1aff base;                        // IC0
    const g1aff* tab;                  // window tables of IC1..
    const nline_t* nt[2];              // normalised gamma / delta line tables
    const fp12* pre;                   // Miller(alpha, beta)
    int ns, vm, reject;                // signals per proof (n_ic - 1), ZKV_VM_*, every proof fails (a key point is invalid)
    uint8_t vk_skip;                   // pairs 1 / 2 disabled for every proof (gamma / delta at infinity), as MillerArgs::vk_skip
};
__device__ __forceinline__ uint32_t group_of(uint32_t k, int nk) { return k < (uint32_t)nk ? k : 0u; }   // out-of-range keys fail in group 0
// per tile t of ZKV_GROUP_TILE records: cnt[t * nk + k] = records of key k
__global__ void __launch_bounds__(256) k_group_count(int n, int nk, const uint32_t* key_idx, uint32_t* cnt) {
    __shared__ uint32_t h[ZKV_MAX_KEYS];
    for (int k = threadIdx.x; k < nk; k += blockDim.x) h[k] = 0;
    __syncthreads();
    const size_t t0 = (size_t)blockIdx.x * ZKV_GROUP_TILE;
    for (int j = threadIdx.x; j < ZKV_GROUP_TILE; j += blockDim.x)
        if (t0 + j < (size_t)n) atomicAdd(&h[group_of(key_idx[t0 + j], nk)], 1u);
    __syncthreads();
    for (int k = threadIdx.x; k < nk; k += blockDim.x) cnt[(size_t)blockIdx.x * nk + k] = h[k];
}
// one block of ZKV_MAX_KEYS threads, thread k = key k: group k starts at the exclusive sum of the padded group sizes before it;
// cnt[t * nk + k] becomes the first slot of tile t's records of key k; the padding slots get their key; *total = slots in all groups
__global__ void __launch_bounds__(ZKV_MAX_KEYS) k_group_scan(int ntiles, int nk, uint32_t* cnt, uint8_t* slot_key, uint32_t* total) {
    __shared__ uint32_t sc[ZKV_MAX_KEYS];
    const int k = threadIdx.x;
    uint32_t c = 0;
    if (k < nk) for (int t = 0; t < ntiles; t++) c += cnt[(size_t)t * nk + k];
    const uint32_t padded = (c + 31u) & ~31u;
    sc[k] = k < nk ? padded : 0u;
    __syncthreads();
    for (int d = 1; d < ZKV_MAX_KEYS; d <<= 1) {
        const uint32_t v = k >= d ? sc[k - d] : 0u;
        __syncthreads();
        sc[k] += v;
        __syncthreads();
    }
    if (k == ZKV_MAX_KEYS - 1) *total = sc[k];
    if (k >= nk) return;
    uint32_t s = sc[k] - padded;
    for (uint32_t p = s + c; p < s + padded; p++) slot_key[p] = (uint8_t)k;
    for (int t = 0; t < ntiles; t++) { const uint32_t v = cnt[(size_t)t * nk + k]; cnt[(size_t)t * nk + k] = s; s += v; }
}
// perm[slot] / slot_key[slot] of every record: warp w of a block takes records [w * 512, w * 512 + 512) of the block's tile in rounds of 32;
// the rank of a record among its key's records is (tile base) + (that key's records in the tile's earlier warps) + (earlier rounds) + (earlier
// lanes of its round, __match_any_sync): caller order inside every group, and the same slots on every run
__global__ void __launch_bounds__(256) k_group_scatter(int n, int nk, const uint32_t* key_idx, const uint32_t* base, uint32_t* perm, uint8_t* slot_key) {
    __shared__ uint32_t wc[8][ZKV_MAX_KEYS];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int k = lane; k < nk; k += 32) wc[w][k] = 0;
    __syncwarp();
    const size_t r0 = (size_t)blockIdx.x * ZKV_GROUP_TILE + (size_t)w * (ZKV_GROUP_TILE / 8);
    const unsigned lt = (1u << lane) - 1u;
    for (int r = 0; r < ZKV_GROUP_TILE / 8; r += 32) {
        const size_t i = r0 + r + lane;
        const uint32_t k = i < (size_t)n ? group_of(key_idx[i], nk) : ZKV_SLOT_EMPTY;
        const unsigned peers = __match_any_sync(0xffffffffu, k);
        if (k != ZKV_SLOT_EMPTY && (peers & lt) == 0) wc[w][k] += __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    for (int k = threadIdx.x; k < nk; k += blockDim.x) {
        uint32_t run = base[(size_t)blockIdx.x * nk + k];
        for (int v = 0; v < 8; v++) { const uint32_t c = wc[v][k]; wc[v][k] = run; run += c; }
    }
    __syncthreads();
    for (int r = 0; r < ZKV_GROUP_TILE / 8; r += 32) {
        const size_t i = r0 + r + lane;
        const uint32_t k = i < (size_t)n ? group_of(key_idx[i], nk) : ZKV_SLOT_EMPTY;
        const unsigned peers = __match_any_sync(0xffffffffu, k);
        if (k != ZKV_SLOT_EMPTY) { const uint32_t s = wc[w][k] + __popc(peers & lt); perm[s] = (uint32_t)i; slot_key[s] = (uint8_t)k; }
        __syncwarp();
        if (k != ZKV_SLOT_EMPTY && (peers & lt) == 0) wc[w][k] += __popc(peers);
        __syncwarp();
    }
}
// k_decode in slot order: record perm[s] of the 256-byte proofs, the vm of the slot's key; empty slots, out-of-range key indices and keys
// with an invalid point get the reject flags of a malformed record
__global__ void k_decode_keys(int n, const uint32_t* perm, const uint8_t* slot_key, const KeyDesc* keys, int nk, const uint32_t* key_idx, const uint8_t* proofs,
                              fp* ax, fp* ay, fp2* bx, fp2* by, fp* cx, fp* cy, uint8_t* flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = perm[i];
    const KeyDesc* kd = keys + slot_key[i];
    if (p == ZKV_SLOT_EMPTY || key_idx[p] >= (uint32_t)nk || kd->reject) { decode_reject(i, F_INVALID, ax, ay, bx, by, cx, cy, flags); return; }
    decode_points(i, proofs + (size_t)p * 256, kd->vm, ax, ay, bx, by, cx, cy, flags);
}
// signals of record perm[s]: words sig_off[p] .. sig_off[p + 1] of `sig` (offsets relative to sig_base); a count other than the key's
// n_ic - 1 (groth16.rs:32) or a signal >= R (groth16.rs:32-34) fails the proof.  Scalars at a stride of `stride` (the widest key) per slot.
__global__ void k_signals_keys(int n, const uint32_t* perm, const uint8_t* slot_key, const KeyDesc* keys, const uint8_t* sig, const uint64_t* sig_off, uint64_t sig_base,
                               int stride, uint32_t* scal, uint8_t* flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = perm[i];
    if (p == ZKV_SLOT_EMPTY) return;
    const int k = keys[slot_key[i]].ns;
    const uint64_t a = sig_off[p], b = sig_off[p + 1];
    if (b < a || b - a != (uint64_t)k) { flags[i] |= F_INVALID; return; }
    bool bad = false;
    for (int j = 0; j < k; j++) {
        uint32_t s[8];
        be32_to_raw(s, sig + (a - sig_base + j) * 32);
        bad |= u256_geq(s, C_R);
        for (int t = 0; t < 8; t++) scal[((size_t)i * stride + j) * 8 + t] = s[t];
    }
    if (bad) flags[i] |= F_INVALID;
}
// k_vkx with the slot's key: its IC0, window tables and scalar count; empty slots get the point at infinity's encoding and no work
__global__ void k_vkx_keys(int n, const uint32_t* perm, const uint8_t* slot_key, const KeyDesc* keys, const uint32_t* scal, int stride, fp* vx, fp* vy, uint8_t* flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (perm[i] == ZKV_SLOT_EMPTY) { vx[i] = fp_zero(); vy[i] = fp_zero(); return; }
    const KeyDesc* kd = keys + slot_key[i];
    const g1aff base = kd->base;
    vkx_one(i, scal, stride, kd->ns, ZKV_WIN_PER_SCALAR, kd->tab, base, vx, vy, flags);
}
// slots of a chunk [o, o + m) that lie in a group: the rest of the chunk is not run (whole blocks return; the last block's surplus threads
// redo the chunk's last grouped slot, whose warp is of a single key since group sizes are multiples of 32)
__device__ __forceinline__ int grouped_in_chunk(const uint32_t* total, size_t o, int m) {
    const size_t t = *total;
    return t <= o ? 0 : (int)(t - o < (size_t)m ? t - o : (size_t)m);
}
// k_miller_lz over slots: each warp reads its key's tables (one key per warp, see above)
__global__ void __launch_bounds__(LZ_NT, 2) k_miller_lz_keys(const uint32_t* total, size_t o, int m, MillerArgs a, const uint8_t* slot_key, const KeyDesc* keys,
                                                            uint8_t* flags, const fp2* tx, const fp2* ty, fp12* fio, g2j* rst, fp* sl, int d_hi, int d_lo, int first, int last) {
    const int n = grouped_in_chunk(total, o, m);
    if ((int)blockIdx.x * LZ_NT >= n) return;
    const int i0 = blockIdx.x * LZ_NT + threadIdx.x;
    const KeyDesc* kd = keys + slot_key[i0 < n ? i0 : n - 1];
    miller_lz(n, a, kd->nt[0], kd->nt[1], kd->pre, kd->vk_skip, flags, tx, ty, fio, rst, sl, d_hi, d_lo, first, last);
}
__global__ void __launch_bounds__(LZ_NT, 2) k_final_exp_lz_keys(const uint32_t* total, size_t o, int m, int s_lo, int s_hi, const fp12* in, fp12* st, const uint8_t* flags, uint8_t* status) {
    const int n = grouped_in_chunk(total, o, m);
    if ((int)blockIdx.x * LZ_NT >= n) return;
    final_exp_lz(n, s_lo, s_hi, in, st, flags, status, nullptr, 0);
}
// slot statuses back to caller order
__global__ void k_status_to_caller(int n, const uint32_t* total, const uint32_t* perm, const uint8_t* slot_status, uint8_t* status) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || (uint32_t)i >= *total) return;
    const uint32_t p = perm[i];
    if (p != ZKV_SLOT_EMPTY) status[p] = slot_status[i];
}

// ---------------------------------------------------------------------------- small services
// pairing service input decode: 4 G1 points + 1 G2 point per instance.  Infinity bits: pair0 -> F_SKIP0, pairs 1..3 -> 0x20,0x40,0x80
__global__ void k_g1_decode4(int n, const uint8_t* g1s /* n x 4 x 64 */, const uint8_t* g2s /* n x 128 */,
                             fp* px0, fp* py0, fp* px1, fp* py1, fp* px2, fp* py2, fp* px3, fp* py3, fp2* qx, fp2* qy, uint8_t* flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fp* xs[4] = {px0, px1, px2, px3}; fp* ys[4] = {py0, py1, py2, py3};
    const uint8_t bits[4] = {F_SKIP0, 0x20, 0x40, 0x80};
    uint8_t fl = 0;
    for (int j = 0; j < 4; j++) {
        uint32_t rx[8], ry[8];
        const uint8_t* p = g1s + ((size_t)i * 4 + j) * 64;
        be32_to_raw(rx, p); be32_to_raw(ry, p + 32);
        fp x, y; int r = g1_decode_raw(x, y, rx, ry);
        xs[j][i] = x; ys[j][i] = y;
        if (r == 2) fl |= F_INVALID;
        if (r == 1) fl |= bits[j];
    }
    fp2 x2, y2; int rb = g2_decode_bytes(x2, y2, g2s + (size_t)i * 128);
    qx[i] = x2; qy[i] = y2;
    if (rb == 2) fl |= F_INVALID;
    if (rb == 1) fl |= F_SKIP0;
    flags[i] = fl;
}
__global__ void k_fp_mul_bytes(int n, const uint8_t* a, const uint8_t* b, uint8_t* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fp x, y, z;
    be32_to_raw(x.v, a + 32 * (size_t)i); be32_to_raw(y.v, b + 32 * (size_t)i);
    fp_to_mont(x, x); fp_to_mont(y, y); fp_mul(z, x, y);
    fp_to_be32(out + 32 * (size_t)i, z);
}
__global__ void k_g2_check_bytes(int n, const uint8_t* g2s, uint8_t* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fp2 x, y; int r = g2_decode_bytes(x, y, g2s + 128 * (size_t)i);
    if (r == 2) { out[i] = 2; return; }
    if (r == 1) { out[i] = 1; return; }
    out[i] = g2_in_subgroup(x, y) ? 1 : 0;
}
__global__ void k_points_to_bytes(int n, const fp* x, const fp* y, uint8_t* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fp_to_be32(out + 64 * (size_t)i, x[i]); fp_to_be32(out + 64 * (size_t)i + 32, y[i]);
}


// ---------------------------------------------------------------------------- precompile-shaped services (groth16.rs:60-73)
// 0x06 ecAdd: in n x 128 B (x1,y1,x2,y2), out n x 64 B, ok[i] = 0 ok / 1 "call reverted" (output zeroed)
__global__ void k_ec_add(int n, const uint8_t* in, uint8_t* out, uint8_t* ok) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t* p = in + 128 * (size_t)i;
    uint32_t rx[8], ry[8];
    fp x1, y1, x2, y2;
    be32_to_raw(rx, p); be32_to_raw(ry, p + 32);
    int r1 = g1_decode_raw(x1, y1, rx, ry);
    be32_to_raw(rx, p + 64); be32_to_raw(ry, p + 96);
    int r2 = g1_decode_raw(x2, y2, rx, ry);
    uint8_t* o = out + 64 * (size_t)i;
    if (r1 == 2 || r2 == 2) { ok[i] = 1; for (int k = 0; k < 64; k++) o[k] = 0; return; }
    g1j acc;
    if (r1 == 1) { acc.x = fp_one(); acc.y = fp_one(); acc.z = fp_zero(); } else { acc.x = x1; acc.y = y1; acc.z = fp_one(); }
    if (r2 == 0) g1_add_affine(acc, x2, y2);
    fp x, y; g1_to_affine(x, y, acc);
    fp_to_be32(o, x); fp_to_be32(o + 32, y); ok[i] = 0;
}
// 0x07 ecMul: in n x 96 B (x,y,s), s any 256-bit integer
__global__ void k_ec_mul(int n, const uint8_t* in, uint8_t* out, uint8_t* ok) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t* p = in + 96 * (size_t)i;
    uint32_t rx[8], ry[8], s[8];
    fp x1, y1;
    be32_to_raw(rx, p); be32_to_raw(ry, p + 32); be32_to_raw(s, p + 64);
    int r1 = g1_decode_raw(x1, y1, rx, ry);
    uint8_t* o = out + 64 * (size_t)i;
    if (r1 == 2) { ok[i] = 1; for (int k = 0; k < 64; k++) o[k] = 0; return; }
    g1j acc; acc.x = fp_one(); acc.y = fp_one(); acc.z = fp_zero();
    if (r1 == 0) {
        for (int b = 255; b >= 0; b--) {
            g1j d; g1_dbl(d, acc); acc = d;
            if ((s[b >> 5] >> (b & 31)) & 1u) g1_add_affine(acc, x1, y1);
        }
    }
    fp x, y; g1_to_affine(x, y, acc);
    fp_to_be32(o, x); fp_to_be32(o + 32, y); ok[i] = 0;
}
// [s]Q for a point on the twist (no subgroup requirement): test-vector / synthetic-proof generation hook
__global__ void k_g2_mul(int n, const uint8_t* pts /* n x 128 or 1 x 128 if bcast */, int bcast, const uint8_t* scalars, uint8_t* out, uint8_t* ok) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fp2 qx, qy; uint32_t s[8];
    int r = g2_decode_bytes(qx, qy, pts + (bcast ? 0 : 128 * (size_t)i));
    be32_to_raw(s, scalars + 32 * (size_t)i);
    uint8_t* o = out + 128 * (size_t)i;
    if (r == 2) { ok[i] = 1; for (int k = 0; k < 128; k++) o[k] = 0; return; }
    g2j acc; acc.x = f2_one(); acc.y = f2_one(); acc.z = f2_zero();
    if (r == 0) {
        g2j q; q.x = qx; q.y = qy; q.z = f2_one();
        for (int b = 255; b >= 0; b--) {
            g2j d; g2_dbl(d, acc); acc = d;
            if ((s[b >> 5] >> (b & 31)) & 1u) { g2_add(d, acc, q); acc = d; }
        }
    }
    ok[i] = 0;
    if (f2_is_zero(acc.z)) { for (int k = 0; k < 128; k++) o[k] = 0; return; }
    fp2 zi, zi2, x, y; f2_inv(zi, acc.z); f2_sqr(zi2, zi); f2_mul(x, acc.x, zi2); f2_mul(zi2, zi2, zi); f2_mul(y, acc.y, zi2);
    fp_to_be32(o, x.c1); fp_to_be32(o + 32, x.c0); fp_to_be32(o + 64, y.c1); fp_to_be32(o + 96, y.c0);
}

// ---------------------------------------------------------------------------- K0: integer-pipe microbenchmarks
// IMAD.WIDE.U32 issue rate: two 8-limb accumulators per thread, each row = a 4-product mad.lo.cc / madc.hi.cc chain (the
// instruction mix of one multiplier row).  The carry flags make every product loop-variant, so ptxas can neither hoist the
// multiplies out of the loop nor split them into IMAD + IADD (a plain `c += a * b` microbenchmark is silently reduced to
// 64-bit adds; see DESIGN.md section 6).  64 IMAD.WIDE per loop iteration.
__global__ void k_imad_wide(uint32_t* out, uint32_t a0, uint32_t b0, int iters) {
    uint32_t a1 = a0 + threadIdx.x, a2 = a1 * 3, a3 = a1 * 5, a4 = a1 * 7, b = b0 ^ blockIdx.x;
    uint32_t e0 = 1, e1 = 2, e2 = 3, e3 = 4, e4 = 5, e5 = 6, e6 = 7, e7 = 8, o0 = 9, o1 = 10, o2 = 11, o3 = 12, o4 = 13, o5 = 14, o6 = 15, o7 = 16;
    for (int k = 0; k < iters; k++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            asm volatile("mad.lo.cc.u32 %0, %16, %20, %0;\n\tmadc.hi.cc.u32 %1, %16, %20, %1;\n\tmadc.lo.cc.u32 %2, %17, %20, %2;\n\tmadc.hi.cc.u32 %3, %17, %20, %3;\n\t"
                         "madc.lo.cc.u32 %4, %18, %20, %4;\n\tmadc.hi.cc.u32 %5, %18, %20, %5;\n\tmadc.lo.cc.u32 %6, %19, %20, %6;\n\tmadc.hi.u32 %7, %19, %20, %7;\n\t"
                         "mad.lo.cc.u32 %8, %17, %20, %8;\n\tmadc.hi.cc.u32 %9, %17, %20, %9;\n\tmadc.lo.cc.u32 %10, %18, %20, %10;\n\tmadc.hi.cc.u32 %11, %18, %20, %11;\n\t"
                         "madc.lo.cc.u32 %12, %19, %20, %12;\n\tmadc.hi.cc.u32 %13, %19, %20, %13;\n\tmadc.lo.cc.u32 %14, %16, %20, %14;\n\tmadc.hi.u32 %15, %16, %20, %15;"
                         : "+r"(e0), "+r"(e1), "+r"(e2), "+r"(e3), "+r"(e4), "+r"(e5), "+r"(e6), "+r"(e7), "+r"(o0), "+r"(o1), "+r"(o2), "+r"(o3), "+r"(o4), "+r"(o5), "+r"(o6), "+r"(o7)
                         : "r"(a1), "r"(a2), "r"(a3), "r"(a4), "r"(b));
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = e0 ^ e1 ^ e2 ^ e3 ^ e4 ^ e5 ^ e6 ^ e7 ^ o0 ^ o1 ^ o2 ^ o3 ^ o4 ^ o5 ^ o6 ^ o7;
}
// dependent chain of Montgomery multiplications per thread (throughput across many threads)
__global__ void k_fpmul_chain(fp* out, int iters) {
    fp x = fp_one(), y = fp_const(C_R2);
    x.v[0] ^= threadIdx.x; y.v[1] ^= blockIdx.x;
    x.v[7] &= 0x0fffffff; y.v[7] &= 0x0fffffff;
    for (int k = 0; k < iters; k++) { fp_mul(x, x, y); fp_mul(y, y, x); }
    fp_add(x, x, y);
    out[blockIdx.x * blockDim.x + threadIdx.x] = x;
}

}  // namespace zkv
