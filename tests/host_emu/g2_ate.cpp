// TEST INFRASTRUCTURE: the G2 subgroup test that the verification Miller loop finishes (csrc/lazy.cuh lz_miller_norm_seg, g2_neg_psi3,
// lz_r_is), compiled as plain C++ so that tests/test_g2_ate_check.py can compare its accept set with the oracle's on a CPU-only box.
#include <cstring>
#include "../../stylus_zkvm_verifiers_b200/csrc/bn254.cuh"
#include "../../stylus_zkvm_verifiers_b200/csrc/lazy.cuh"
using namespace zkv;

static bool dec_fp(fp& r, const uint8_t* b) { fp t; be32_to_raw(t.v, b); if (u256_geq(t.v, C_P)) return false; fp_to_mont(r, t); return true; }
static bool dec_g2(fp2& x, fp2& y, const uint8_t* b) { return dec_fp(x.c1, b) && dec_fp(x.c0, b + 32) && dec_fp(y.c1, b + 64) && dec_fp(y.c0, b + 96); }

extern "C" {
// B (EIP-197 encoding, on the twist or infinity) through the Miller loop the way k_miller_lz runs it: `nseg` segments, the variable pair
// switched off or not (R is advanced either way), the fixed pairs' tables zero (they do not touch R).  r_out receives R's X, Y, Z
// (6 x BE-32, wire order im / re per Fp2).  Returns 1 if R equals -psi^3(B) (the kernel accepts B), 0 if not, 2 for a bad encoding.
int emu_ate_g2_check(const uint8_t* g2, int nseg, int var_off, uint8_t* r_out) {
    static nline_t zt[ZKV_LINES_PER_G2];
    fp2 qx, qy;
    if (!dec_g2(qx, qy, g2)) return 2;
    fp px = fp_one(), py = fp_one(), sl[4] = {fp_zero(), fp_zero(), fp_zero(), fp_zero()};
    LzMillerIn in; in.px0 = &px; in.py0 = &py; in.qx = &qx; in.qy = &qy; in.sl = sl; in.nt[0] = zt; in.nt[1] = zt; in.var_off = var_off != 0;
    lz_miller_init(qx, qy);
    const int top = ZKV_ATE_NAF_LEN - 2;
    for (int k = 0; k < nseg; k++) lz_miller_norm_seg(in, top - (top + 1) * k / nseg, top - (top + 1) * (k + 1) / nseg + 1, k == nseg - 1);
    for (int c = 0; c < 3; c++) {
        const fp2 v = lz_ld2((LZ_R + 2 * c) * LZ_SLOT);
        fp_to_be32(r_out + 64 * c, v.c1); fp_to_be32(r_out + 64 * c + 32, v.c0);
    }
    fp2 tx = qx, ty = qy;
    g2_neg_psi3(tx, ty);
    return lz_r_is(LZ_R * LZ_SLOT, tx, ty) ? 1 : 0;
}
}
