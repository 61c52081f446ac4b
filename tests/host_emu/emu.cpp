// TEST INFRASTRUCTURE: compiles csrc/bn254.cuh as plain C++ (portable Fp backend) so the tower / curve /
// pairing logic the kernels use can be compared with the oracle on a CPU-only box.  Never shipped.
#include <cstring>
#include "../../stylus_zkvm_verifiers_b200/csrc/bn254.cuh"
#include "../../stylus_zkvm_verifiers_b200/csrc/lazy.cuh"
using namespace zkv;

static bool dec_fp(fp& r, const uint8_t* b) { fp t; be32_to_raw(t.v, b); if (u256_geq(t.v, C_P)) return false; fp_to_mont(r, t); return true; }
static bool dec_g2(fp2& x, fp2& y, const uint8_t* b) { return dec_fp(x.c1, b) && dec_fp(x.c0, b + 32) && dec_fp(y.c1, b + 64) && dec_fp(y.c0, b + 96); }
static void dec_f12(fp12& a, const uint8_t* in) { fp* w = &a.c0.c0.c0; for (int i = 0; i < 12; i++) dec_fp(w[i], in + 32 * i); }

extern "C" {
int emu_fp_mul(const uint8_t* a, const uint8_t* b, uint8_t* out) { fp x, y, z; dec_fp(x, a); dec_fp(y, b); fp_mul(z, x, y); fp_to_be32(out, z); return 0; }
int emu_fp_inv(const uint8_t* a, uint8_t* out) { fp x, z; dec_fp(x, a); fp_inv(z, x); fp_to_be32(out, z); return 0; }
int emu_fp_inv_fermat(const uint8_t* a, uint8_t* out) { fp x, z; dec_fp(x, a); fp_inv_fermat(z, x); fp_to_be32(out, z); return 0; }
int emu_f12_mul(const uint8_t* a, const uint8_t* b, uint8_t* out) { fp12 x, y, z; dec_f12(x, a); dec_f12(y, b); f12_mul(z, x, y); f12_to_bytes(out, z); return 0; }
int emu_f12_sqr(const uint8_t* a, uint8_t* out) { fp12 x, z; dec_f12(x, a); f12_sqr(z, x); f12_to_bytes(out, z); return 0; }
int emu_f12_cyc_sqr(const uint8_t* a, uint8_t* out) { fp12 x, z; dec_f12(x, a); f12_cyc_sqr(z, x); f12_to_bytes(out, z); return 0; }
int emu_f12_inv(const uint8_t* a, uint8_t* out) { fp12 x, z; dec_f12(x, a); f12_inv(z, x); f12_to_bytes(out, z); return 0; }
int emu_final_exp(const uint8_t* a, uint8_t* out) { fp12 x, z; dec_f12(x, a); final_exp(z, x); f12_to_bytes(out, z); return 0; }
int emu_final_exp_staged(const uint8_t* a, uint8_t* out) {
    fp12 m, f, x, y, z, t1, r; dec_f12(m, a);
    final_exp_stage0(f, x, m); { fp12 t = x; final_exp_stage1(x, y, z, t); } final_exp_stage2(t1, z); final_exp_stage3(r, f, x, y, z, t1);
    f12_to_bytes(out, r); return 0;
}
// 1 = in G2, 0 = on twist but not in G2, 2 = not on twist / bad encoding
int emu_g2_check(const uint8_t* q) { fp2 x, y; if (!dec_g2(x, y, q)) return 2; if (!g2_on_curve(x, y)) return 2; return g2_in_subgroup(x, y) ? 1 : 0; }
// 4-pair Miller loop + final exp with bn254.cuh's thread-stack routines: pair 0 variable G2, pairs 1..3 from line tables of the three fixed points
int emu_pairing4(const uint8_t* g1s /*4x64*/, const uint8_t* g2 /*128*/, const uint8_t* fixed /*3x128*/, uint8_t* miller_out, uint8_t* gt_out) {
    static line_t tabs_store[3][ZKV_LINES_PER_G2];
    fp px[4], py[4];
    for (int j = 0; j < 4; j++) { dec_fp(px[j], g1s + 64 * j); dec_fp(py[j], g1s + 64 * j + 32); }
    fp2 qx, qy; dec_g2(qx, qy, g2);
    const line_t* tabs[3];
    for (int j = 0; j < 3; j++) { fp2 x, y; dec_g2(x, y, fixed + 128 * j); g2_precompute_lines(tabs_store[j], x, y); tabs[j] = tabs_store[j]; }
    fp12 f, gt;
    miller_loop(f, px, py, qx, qy, tabs, 3, 0);
    final_exp(gt, f);
    f12_to_bytes(miller_out, f); f12_to_bytes(gt_out, gt);
    return f12_is_one(gt) ? 1 : 0;
}
// 3-pair loop times a precomputed Miller(alpha, beta), as run_verify does
int emu_pairing3_pre(const uint8_t* g1s /*4x64: A, alpha, vkx, C*/, const uint8_t* g2, const uint8_t* fixed, uint8_t* miller_out) {
    static line_t tabs_store[3][ZKV_LINES_PER_G2];
    fp px[4], py[4];
    for (int j = 0; j < 4; j++) { dec_fp(px[j], g1s + 64 * j); dec_fp(py[j], g1s + 64 * j + 32); }
    fp2 qx, qy; dec_g2(qx, qy, g2);
    for (int j = 0; j < 3; j++) { fp2 x, y; dec_g2(x, y, fixed + 128 * j); g2_precompute_lines(tabs_store[j], x, y); }
    fp12 pre, f;
    { fp ax[2] = {fp_zero(), px[1]}, ay[2] = {fp_zero(), py[1]}; const line_t* t1[1] = {tabs_store[0]}; fp2 z = f2_zero(); miller_loop(pre, ax, ay, z, z, t1, 1, 1u);   /* pair 0 switched off: only the tabled (alpha, beta) pair contributes */ }
    fp bx[3] = {px[0], px[2], px[3]}, by[3] = {py[0], py[2], py[3]};
    const line_t* t2[2] = {tabs_store[1], tabs_store[2]};
    miller_loop(f, bx, by, qx, qy, t2, 2, 0);
    f12_mul(f, f, pre);
    f12_to_bytes(miller_out, f);
    return 0;
}
// the verification path as run_verify does it: normalised gamma / delta tables, 3-pair loop, times Miller(alpha, beta), final exponentiation
int emu_verify_norm_gt(const uint8_t* g1s /*4x64: A, alpha, vkx, C*/, const uint8_t* g2, const uint8_t* fixed, int skip_mask, uint8_t* gt_out) {
    static line_t tabs_store[3][ZKV_LINES_PER_G2];
    static nline_t ntabs[2][ZKV_LINES_PER_G2];
    fp px[4], py[4];
    for (int j = 0; j < 4; j++) { dec_fp(px[j], g1s + 64 * j); dec_fp(py[j], g1s + 64 * j + 32); }
    fp2 qx, qy; dec_g2(qx, qy, g2);
    for (int j = 0; j < 3; j++) { fp2 x, y; dec_g2(x, y, fixed + 128 * j); g2_precompute_lines(tabs_store[j], x, y); }
    for (int j = 0; j < 2; j++) if (!g2_normalise_lines(ntabs[j], tabs_store[j + 1], ZKV_LINES_PER_G2)) return -1;
    fp12 pre, f, gt;
    { fp ax[2] = {fp_zero(), px[1]}, ay[2] = {fp_zero(), py[1]}; const line_t* t1[1] = {tabs_store[0]}; fp2 z = f2_zero(); miller_loop(pre, ax, ay, z, z, t1, 1, 1u); }
    fp x2[2] = {px[2], px[3]}, y2[2] = {py[2], py[3]}, xy[2], iy[2];
    bool off[2] = {(skip_mask & 2) != 0, (skip_mask & 4) != 0};
    g1_slopes2(xy, iy, x2, y2, off);
    const nline_t* nt[2] = {ntabs[0], ntabs[1]};
    miller_loop_norm(f, px[0], py[0], qx, qy, nt, xy, iy, (skip_mask & 1) != 0);
    f12_mul(f, f, pre);
    final_exp(gt, f);
    f12_to_bytes(gt_out, gt);
    return f12_is_one(gt) ? 1 : 0;
}
// scalar multiple by double-and-add with the complete mixed addition used by k_vkx / k_ec_mul
int emu_g1_mul(const uint8_t* pt, const uint8_t* k, uint8_t* out) {
    fp x, y; dec_fp(x, pt); dec_fp(y, pt + 32);
    uint32_t s[8]; be32_to_raw(s, k);
    g1j acc; acc.x = fp_one(); acc.y = fp_one(); acc.z = fp_zero();
    for (int b = 255; b >= 0; b--) { g1j d; g1_dbl(d, acc); acc = d; if ((s[b >> 5] >> (b & 31)) & 1u) g1_add_affine(acc, x, y); }
    fp ox, oy; g1_to_affine(ox, oy, acc); fp_to_be32(out, ox); fp_to_be32(out + 32, oy); return 0;
}

// ---- shared-memory-resident lazily reduced tower (csrc/lazy.cuh) on the one-thread slot emulation
static void slots_from_bytes(int slot, const uint8_t* in, int nfp) { for (int i = 0; i < nfp; i++) { fp t; dec_fp(t, in + 32 * i); lz_stfp((slot + i) * LZ_SLOT, t); } }
static void slots_to_bytes(uint8_t* out, int slot, int nfp) { for (int i = 0; i < nfp; i++) fp_to_be32(out + 32 * i, lz_ldfp((slot + i) * LZ_SLOT)); }
static void fp6_to_bytes(uint8_t* out, const fp6& r) { const fp* w = &r.c0.c0; for (int i = 0; i < 6; i++) fp_to_be32(out + 32 * i, w[i]); }
// a, b: 6 x BE-32 (tower order c0.c0, c0.c1, c1.c0, ...); sparse != 0: b = b0 + b1 v (4 x BE-32)
int emu_lz_f6mul(const uint8_t* a, const uint8_t* b, int sparse, uint8_t* out, uint8_t* out_ref) {
    slots_from_bytes(0, a, 6); slots_from_bytes(6, b, sparse ? 4 : 6);
    fp6 r = sparse ? lz_f6mul01(0, 6 * LZ_SLOT) : lz_f6mul(0, 6 * LZ_SLOT);
    fp6_to_bytes(out, r);
    fp6 x, y, z; fp* xw = &x.c0.c0; fp* yw = &y.c0.c0;
    for (int i = 0; i < 6; i++) { dec_fp(xw[i], a + 32 * i); if (!sparse || i < 4) dec_fp(yw[i], b + 32 * i); else yw[i] = fp_zero(); }
    f6_mul(z, x, y); fp6_to_bytes(out_ref, z);
    return 0;
}
int emu_lz_f12sqr(const uint8_t* a, uint8_t* out) { slots_from_bytes(0, a, 12); lz_f12sqr(0, 12 * LZ_SLOT); slots_to_bytes(out, 0, 12); return 0; }
// the verification Miller loop on slots (lz_miller_norm_seg, in `nseg` segments with the state carried between them) against miller_loop_norm
int emu_lz_miller_norm(const uint8_t* g1s /*4x64: A, alpha(unused), vkx, C*/, const uint8_t* g2, const uint8_t* fixed, int skip_mask, int nseg, uint8_t* out_lz, uint8_t* out_ref) {
    static line_t tabs_store[3][ZKV_LINES_PER_G2];
    static nline_t ntabs[2][ZKV_LINES_PER_G2];
    fp px[4], py[4];
    for (int j = 0; j < 4; j++) { dec_fp(px[j], g1s + 64 * j); dec_fp(py[j], g1s + 64 * j + 32); }
    fp2 qx, qy; dec_g2(qx, qy, g2);
    for (int j = 0; j < 3; j++) { fp2 x, y; dec_g2(x, y, fixed + 128 * j); g2_precompute_lines(tabs_store[j], x, y); }
    for (int j = 0; j < 2; j++) if (!g2_normalise_lines(ntabs[j], tabs_store[j + 1], ZKV_LINES_PER_G2)) return -1;
    fp x2[2] = {px[2], px[3]}, y2[2] = {py[2], py[3]}, xy[2], iy[2];
    bool off[2] = {(skip_mask & 2) != 0, (skip_mask & 4) != 0};
    g1_slopes2(xy, iy, x2, y2, off);
    const nline_t* nt[2] = {ntabs[0], ntabs[1]};
    fp12 f;
    miller_loop_norm(f, px[0], py[0], qx, qy, nt, xy, iy, (skip_mask & 1) != 0);
    f12_to_bytes(out_ref, f);
    fp sl[4] = {xy[0], xy[1], iy[0], iy[1]};
    LzMillerIn in; in.px0 = &px[0]; in.py0 = &py[0]; in.qx = &qx; in.qy = &qy; in.sl = sl; in.nt[0] = ntabs[0]; in.nt[1] = ntabs[1]; in.var_off = (skip_mask & 1) != 0;
    lz_miller_init(qx, qy);
    const int top = ZKV_ATE_NAF_LEN - 2;
    for (int k = 0; k < nseg; k++) {
        int hi = top - (top + 1) * k / nseg, lo = top - (top + 1) * (k + 1) / nseg + 1;
        lz_miller_norm_seg(in, hi, lo, k == nseg - 1);
    }
    slots_to_bytes(out_lz, LZ_F, 12);
    return 0;
}
// the final exponentiation on slots, stage by stage with the state in "global" memory, against final_exp
int emu_lz_final_exp(const uint8_t* a, uint8_t* out) {
    fp12 m; dec_f12(m, a);
    static fp12 st[6];
    for (int s = 0; s < 4; s++) lz_final_exp_stage(s, &m, st);
    slots_to_bytes(out, LZ_A, 12);
    return 0;
}
int emu_lz_f12_ops(const uint8_t* a, const uint8_t* b, uint8_t* mul, uint8_t* mulc, uint8_t* inv, uint8_t* csq, uint8_t* fr /*3x384*/) {
    fp12 y; dec_f12(y, b);
    const uint32_t A = LZ_A * LZ_SLOT, X = LZ_X * LZ_SLOT, Y = LZ_Y * LZ_SLOT, L = LZ_L * LZ_SLOT;
    slots_from_bytes(0, a, 12); lz_f12mul_g(A, X, Y, &y, false); slots_to_bytes(mul, 0, 12);
    slots_from_bytes(0, a, 12); lz_f12mul_g(A, X, Y, &y, true); slots_to_bytes(mulc, 0, 12);
    slots_from_bytes(0, a, 12); lz_f12inv(A, X, Y); slots_to_bytes(inv, 0, 12);
    slots_from_bytes(0, a, 12); lz_cyc_sqr(A, L); slots_to_bytes(csq, 0, 12);
    for (int k = 1; k <= 3; k++) { slots_from_bytes(0, a, 12); lz_frob(A, k); slots_to_bytes(fr + 384 * (k - 1), 0, 12); }
    return 0;
}
int emu_f12_misc(const uint8_t* a, const uint8_t* b, uint8_t* mulc, uint8_t* fr /*3x384*/) {      // round-1 tower counterparts
    fp12 x, y, z; dec_f12(x, a); dec_f12(y, b);
    f12_conj(z, y); f12_mul(z, x, z); f12_to_bytes(mulc, z);
    for (int k = 1; k <= 3; k++) { f12_frob(z, x, k); f12_to_bytes(fr + 384 * (k - 1), z); }
    return 0;
}
}
