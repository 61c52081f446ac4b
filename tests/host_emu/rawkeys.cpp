// TEST INFRASTRUCTURE: the raw-key verification path's own arithmetic (csrc/bn254.cuh g1_vkx_var, csrc/lazy.cuh lz_miller_gen_seg with four
// variable pairs and lz_gen_subgroup_ok) compiled as plain C++, so that tests/test_rawkeys_emu.py can compare it with the oracle on a CPU-only box.
#include <cstring>
#include "../../stylus_zkvm_verifiers_b200/csrc/bn254.cuh"
#include "../../stylus_zkvm_verifiers_b200/csrc/lazy.cuh"
using namespace zkv;

static bool dec_fp(fp& r, const uint8_t* b) { fp t; be32_to_raw(t.v, b); if (u256_geq(t.v, C_P)) return false; fp_to_mont(r, t); return true; }
static bool dec_g2(fp2& x, fp2& y, const uint8_t* b) { return dec_fp(x.c1, b) && dec_fp(x.c0, b + 32) && dec_fp(y.c1, b + 64) && dec_fp(y.c0, b + 96); }

extern "C" {
// vk_x of n_ic IC points (64 B each) and n_ic - 1 scalars (32 B each) as k_vkx_rawkeys computes it: 0 finite, 1 infinity, 2 an IC point fails
int emu_vkx_var(const uint8_t* ic, int n_ic, const uint8_t* s, uint8_t* out) {
    fp x, y;
    const int r = g1_vkx_var(x, y, ic, n_ic, s);
    fp_to_be32(out, x); fp_to_be32(out + 32, y);
    return r;
}
// Four pairs (G1 64 B || G2 128 B each, on their curves or infinity) through the Miller loop of k_miller_rawkeys: `nseg` segments with f and R_j
// carried between them, a pair with a member at infinity switched off.  miller_out receives f; returns 1 if every G2 point passes the fused
// order-r test (lz_gen_subgroup_ok against -psi^3(Q_j)), 0 if one fails, 2 for a bad encoding.
int emu_rawkeys_miller4(const uint8_t* pairs, int nseg, uint8_t* miller_out) {
    fp px[4], py[4]; fp2 qx[4], qy[4], tx[4], ty[4]; g2j rst[4]; uint8_t pskip[4];
    for (int j = 0; j < 4; j++) {
        const uint8_t* p = pairs + 192 * j;
        if (!dec_fp(px[j], p) || !dec_fp(py[j], p + 32) || !dec_g2(qx[j], qy[j], p + 64)) return 2;
        pskip[j] = (fp_is_zero(px[j]) && fp_is_zero(py[j])) || (f2_is_zero(qx[j]) && f2_is_zero(qy[j]));
        tx[j] = qx[j]; ty[j] = qy[j]; g2_neg_psi3(tx[j], ty[j]);
    }
    LzGenIn in; memset(&in, 0, sizeof in);
    in.px = px; in.py = py; in.qx = qx; in.qy = qy; in.rst = rst; in.pskip = pskip; in.stride = 1; in.nvar = 4; in.nfix = 0;
    lz_st2(LZ_F * LZ_SLOT, f2_one());
    for (int k = 1; k < 6; k++) lz_st2((LZ_F + 2 * k) * LZ_SLOT, f2_zero());
    const int top = ZKV_ATE_NAF_LEN - 2;
    for (int k = 0; k < nseg; k++) lz_miller_gen_seg(in, 0, top - (top + 1) * k / nseg, top - (top + 1) * (k + 1) / nseg + 1, k == 0, k == nseg - 1);
    for (int k = 0; k < 12; k++) fp_to_be32(miller_out + 32 * k, lz_ldfp((LZ_F + k) * LZ_SLOT));
    return lz_gen_subgroup_ok(in, 0, tx, ty) ? 1 : 0;
}
}
