/* zkv.h -- C ABI of the B200 batched Groth16/BN254 verifier (libzkv_b200.so).
 *
 * Drop-in boundary for the verification path of gnosisguild/stylus-zkvm-verifiers.  Every entry
 * point below cites the reference interface it replaces (paths relative to the reference root).
 * All functions launch sm_100a CUDA kernels; there is NO CPU fallback: without a usable CUDA
 * device they return ZKV_ERR_CUDA and set zkv_last_error().
 *
 * Conventions
 *   - all field elements / scalars cross the boundary as 32-byte big-endian words (the EVM ABI
 *     the reference uses, common/groth16.rs:61,112-119); G2 words are in wire order
 *     x[0],x[1],y[0],y[1] = x_im,x_re,y_im,y_re (common/types.rs:9-15 + EIP-197);
 *   - caller owns every buffer; handles are opaque and immutable after creation;
 *   - return value: 0 = ok, <0 = argument / CUDA error (message via zkv_last_error());
 *   - per-proof result: one status byte (zkv_status), `accept == (status == ZKV_OK)`.
 */
#ifndef ZKV_H
#define ZKV_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* Per-proof status = which Result the reference would return.
 * common/errors.rs:3-8, risc0/errors.rs:8-10, sp1/errors.rs:8-10. */
typedef enum {
    ZKV_OK = 0,                     /* Ok(true) / Ok(())                                  */
    ZKV_INVALID_INITIALIZATION = 1, /* InvalidInitialization()  risc0/verifier.rs:84-86   */
    ZKV_INVALID_PROOF_DATA = 2,     /* InvalidProofData()       risc0/verifier.rs:151-153,166-170; sp1/verifier.rs:64-66,79-83 */
    ZKV_SELECTOR_MISMATCH = 3,      /* SelectorMismatch / WrongVerifierSelector  risc0/verifier.rs:155-164; sp1/verifier.rs:68-77 */
    ZKV_VERIFICATION_FAILED = 4     /* VerificationFailed()     risc0/verifier.rs:191-193; sp1/verifier.rs:106-108 */
} zkv_status;

#define ZKV_ERR_ARG (-1)
#define ZKV_ERR_CUDA (-2)
#define ZKV_ERR_STATE (-3)

#define ZKV_VM_RISC0 0 /* common/types.rs:25-26 VMType::Risc0 : A is negated before pairing (groth16.rs:96-99) */
#define ZKV_VM_SP1 1   /* VMType::Sp1   : A used as is, vk stores -beta,-gamma,-delta (groth16.rs:100-103)    */

typedef struct zkv_vk zkv_vk;       /* common/types.rs:17-23 VerificationKey + per-vk device tables */
typedef struct zkv_risc0 zkv_risc0; /* risc0/verifier.rs:44-52 RiscZeroVerifier storage             */
typedef struct zkv_sp1 zkv_sp1;     /* sp1/verifier.rs:31-33 Sp1Verifier                            */

const char* zkv_last_error(void);   /* thread-local message of the last failing call */
int zkv_device_count(void);

/* ---- verification keys ------------------------------------------------------------------
 * Replaces `VerificationKey` construction (risc0/crypto.rs:81-89, sp1/crypto.rs:83-91).
 * Uploads the key to every listed device and builds, on the GPU, the fixed-base window tables
 * for the IC points, the optimal-ate line tables for beta/gamma/delta and Miller(alpha,beta).
 * n_ic = number of IC points (public inputs + 1), 2..16.  devices == NULL -> device 0 only. */
int zkv_vk_load(int vm_type, const uint8_t alpha[64], const uint8_t beta[128], const uint8_t gamma[128],
                const uint8_t delta[128], const uint8_t* ic, int n_ic, const int* devices, int n_dev, zkv_vk** out);
int zkv_vk_load_risc0(const int* devices, int n_dev, zkv_vk** out); /* the constants of risc0/crypto.rs:16-79 */
int zkv_vk_load_sp1(const int* devices, int n_dev, zkv_vk** out);   /* the constants of sp1/crypto.rs:7-81    */
void zkv_vk_free(zkv_vk* vk);

/* ---- generic Groth16 (common/groth16.rs:23-49 verify_proof_with_key) --------------------
 * proofs: n x 256 B = (a[2], b[2][2], c[2]) ; signals: n x k x 32 B, k must equal n_ic - 1
 * (a mismatch makes every status VERIFICATION_FAILED, groth16.rs:32).  status_out[i] is
 * ZKV_OK or ZKV_VERIFICATION_FAILED. */
int zkv_groth16_verify_batch(const zkv_vk* vk, const uint8_t* proofs, const uint8_t* signals, int k, size_t n, uint8_t* status_out);

/* ---- many keys in one batch: N independent verify_proof_with_key calls (common/groth16.rs:23-49) ---------
 * A set of 1..256 loaded keys (borrowed: they must outlive the set).  Every key must be loaded on every device of the set
 * (devices == NULL -> device 0); keys may differ in vm_type and n_ic.  zkv_vkset_create returns ZKV_ERR_ARG for a key missing on
 * a set device, and for a valid key with finite gamma and delta whose normalised line tables could not be built (a vanishing line
 * coefficient).  A set always runs the default schedule (shared-memory kernels, normalised lines, automatic chunking): the member
 * keys' zkv_vk_tune settings do not apply to it.
 *
 * zkv_groth16_verify_batch_keys: proof i (256 B, the layout of zkv_groth16_verify_batch) is verified under keys[key_idx[i]] with
 * the signals signals[sig_off[i] .. sig_off[i+1]) (offsets in 32-byte words, n+1 of them, non-decreasing).  status_out[i] =
 * ZKV_OK or ZKV_VERIFICATION_FAILED in caller order: exactly what zkv_groth16_verify_batch returns for that proof alone under its
 * own key, so a signal count other than that key's n_ic - 1 (groth16.rs:32) fails that proof only, the RISC Zero negation of A
 * applies to proofs of ZKV_VM_RISC0 keys only, and a key with an invalid point fails all of its proofs.  A key index >= n_keys,
 * decreasing offsets or a null pointer returns ZKV_ERR_ARG with status_out untouched; n == 0 does nothing.  A multi-device set splits
 * the batch into contiguous caller ranges.  The proofs of a device pass (up to 2^20) are grouped by key on the device before any
 * verification kernel runs; the kernel launches per pass do not depend on the number of keys (zkv_launch_count: 10 for a pass of
 * one kernel chain, 41 once the pass's slot bound n + 31 x min(n_keys, n) reaches the automatic chunking threshold of ZKV_TUNE_OVERLAP).
 * zkv_groth16_verify_batch_keys_device: the same on device-resident arrays of one set device (d_key_idx n x uint32, d_sig_off
 * n+1 x uint64 indexing d_signals directly), n <= 2^23, enqueued on `stream` (a cudaStream_t), asynchronous.  The index and offset
 * checks run on the device there: a key index >= n_keys or a decreasing offset fails that proof (ZKV_VERIFICATION_FAILED). */
typedef struct zkv_vkset zkv_vkset;
int zkv_vkset_create(const zkv_vk* const* keys, int n_keys, const int* devices, int n_dev, zkv_vkset** out);
void zkv_vkset_destroy(zkv_vkset* s);
int zkv_groth16_verify_batch_keys(const zkv_vkset* s, const uint32_t* key_idx, const uint8_t* proofs, const uint8_t* signals,
                                  const uint64_t* sig_off, size_t n, uint8_t* status_out);
int zkv_groth16_verify_batch_keys_device(const zkv_vkset* s, int device, const void* d_key_idx, const void* d_proofs,
                                         const void* d_signals, const void* d_sig_off, size_t n, void* d_status_out, void* stream);

/* ---- RISC Zero (risc0/verifier.rs) -------------------------------------------------------
 * zkv_risc0_create(vk = NULL) uses the reference's hard-coded key; a custom vk (synthetic
 * benchmarks) is borrowed, not owned.  A handle starts un-initialised, like the contract. */
int zkv_risc0_create(const zkv_vk* vk_or_null, const int* devices, int n_dev, zkv_risc0** out);
void zkv_risc0_destroy(zkv_risc0* h);
/* IRiscZeroVerifier::initialize, risc0/verifier.rs:58-76.  Returns ZKV_ERR_STATE if already initialised. */
int zkv_risc0_initialize(zkv_risc0* h, const uint8_t control_root[32], const uint8_t bn254_control_id[32]);
int zkv_risc0_is_initialized(const zkv_risc0* h);                              /* :122-124 */
int zkv_risc0_get_selector(const zkv_risc0* h, uint8_t out[4]);                /* :106-108 */
int zkv_risc0_get_control_root(const zkv_risc0* h, uint8_t out0[16], uint8_t out1[16]); /* :110-112 */
int zkv_risc0_get_bn254_control_id(const zkv_risc0* h, uint8_t out[32]);       /* :114-116 */
int zkv_risc0_get_verifier_key_digest(const zkv_risc0* h, uint8_t out[32]);    /* :118-120, crypto.rs:136-195 */
/* IRiscZeroVerifier::verify x n, risc0/verifier.rs:78-92.  seals = concatenated blobs,
 * seal_off[n+1] byte offsets; image_ids / journal_digests = n x 32 B. */
int zkv_risc0_verify_batch(const zkv_risc0* h, const uint8_t* seals, const uint64_t* seal_off, const uint8_t* image_ids,
                           const uint8_t* journal_digests, size_t n, uint8_t* status_out);
/* IRiscZeroVerifier::verify_integrity x n, risc0/verifier.rs:94-104. */
int zkv_risc0_verify_integrity_batch(const zkv_risc0* h, const uint8_t* seals, const uint64_t* seal_off,
                                     const uint8_t* claim_digests, size_t n, uint8_t* status_out);
/* single-proof forms of the two calls above; *status_out receives the zkv_status, return 0/err */
int zkv_risc0_verify(const zkv_risc0* h, const uint8_t* seal, size_t seal_len, const uint8_t image_id[32],
                     const uint8_t journal_digest[32], uint8_t* status_out);
int zkv_risc0_verify_integrity(const zkv_risc0* h, const uint8_t* seal, size_t seal_len, const uint8_t claim_digest[32], uint8_t* status_out);

/* ---- SP1 (sp1/verifier.rs) ---------------------------------------------------------------
 * vk = NULL uses sp1/crypto.rs; selector = first 4 bytes of VERIFIER_HASH (sp1/config.rs:4-9,18-20). */
int zkv_sp1_create(const zkv_vk* vk_or_null, const int* devices, int n_dev, zkv_sp1** out);
void zkv_sp1_destroy(zkv_sp1* h);
int zkv_sp1_verifier_hash(const zkv_sp1* h, uint8_t out[32]);                  /* sp1/verifier.rs:48-50 */
const char* zkv_sp1_version(const zkv_sp1* h);                                 /* sp1/verifier.rs:52-54 */
/* ISp1Verifier::verify_proof x n, sp1/verifier.rs:39-46,58-111.  vkeys n x 32 B; public values and
 * proofs are concatenated blobs with n+1 byte offsets each. */
int zkv_sp1_verify_batch(const zkv_sp1* h, const uint8_t* vkeys, const uint8_t* public_values, const uint64_t* pv_off,
                         const uint8_t* proofs, const uint64_t* proof_off, size_t n, uint8_t* status_out);
int zkv_sp1_verify_proof(const zkv_sp1* h, const uint8_t vkey[32], const uint8_t* public_values, size_t pv_len,
                         const uint8_t* proof, size_t proof_len, uint8_t* status_out);

/* ---- device-resident variants (inputs already in HBM; kernels enqueued on `stream`) ------
 * Used for kernel-only throughput.  Fixed-stride records: seals/proofs are n x 260 B (selector + 8
 * words), public values n x pv_stride B.  Single device (the one the pointers live on, which must be
 * in the handle's device list).  `stream` is a cudaStream_t passed as void*.  Asynchronous. */
int zkv_risc0_verify_batch_device(const zkv_risc0* h, int device, const void* d_seals260, const void* d_image_ids,
                                  const void* d_journal_digests, size_t n, void* d_status_out, void* stream);
int zkv_sp1_verify_batch_device(const zkv_sp1* h, int device, const void* d_vkeys, const void* d_public_values, size_t pv_stride,
                                const void* d_proofs260, size_t n, void* d_status_out, void* stream);

/* ---- pairing service (the 0x08 seam, common/groth16.rs:109-128) ---------------------------
 * n instances of a 4-pair product check e(P0,Q) e(P1,beta) e(P2,gamma) e(P3,delta) == 1 with the three
 * fixed G2 points taken from `vk`.  g1s: n x 4 x 64 B, g2s: n x 128 B.  ok_out[i] = 1 / 0, or 2 if the
 * instance would make the precompile revert (invalid point).  gt_out (optional, n x 384 B) receives the
 * final-exponentiation value, miller_out (optional) the Miller-loop value: 12 x BE-32 in tower order
 * c0.c0.c0, c0.c0.c1, c0.c1.c0, ... (convention in DESIGN.md section 3). */
int zkv_pairing4_batch(const zkv_vk* vk, const uint8_t* g1s, const uint8_t* g2s, size_t n, uint8_t* ok_out,
                       uint8_t* gt_out, uint8_t* miller_out);
int zkv_pairing4_batch_device(const zkv_vk* vk, int device, const void* d_g1s, const void* d_g2s, size_t n,
                              void* d_ok_out, void* d_gt_out, void* stream);

/* General ecPairing (precompile 0x08, the seam the reference calls at common/groth16.rs:109-128): n instances of a k-pair product check
 * with EVERY G2 point variable.  in: n x k x 192 B, each pair G1 (64 B) || G2 (128 B, wire order).  out: n x 32 B, the precompile's return
 * word (0..01 / 0..00).  reverted[i] = 1 where the call would fail (coordinate >= p, point off its curve, G2 point outside the order-r
 * subgroup); a pair with a member at infinity contributes 1; k = 0 is the empty product (true).  miller_out (optional, n x 384 B): the
 * Miller-loop value in the oracle's convention.  zkv_ec_pairing is one call on raw bytes (len % 192 != 0 -> reverted). */
int zkv_ec_pairing_batch(const uint8_t* in, int k, size_t n, uint8_t* out, uint8_t* reverted, uint8_t* miller_out, int device);
int zkv_ec_pairing(const uint8_t* in, size_t len, uint8_t out[32], uint8_t* reverted, int device);

/* ---- precompile-shaped batched services (the L1 seam, common/groth16.rs:60-73: ec_call) -----
 * zkv_ec_add_batch: n x 128 B (x1,y1,x2,y2) -> n x 64 B, EIP-196 0x06 (groth16.rs:55).
 * zkv_ec_mul_batch: n x 96 B (x,y,s)        -> n x 64 B, EIP-196 0x07 (groth16.rs:54).
 * reverted[i] = 1 where the precompile call would fail (coordinate >= p or point off the curve);
 * the corresponding output is zeroed. */
int zkv_ec_add_batch(const uint8_t* in, size_t n, uint8_t* out, uint8_t* reverted, int device);
int zkv_ec_mul_batch(const uint8_t* in, size_t n, uint8_t* out, uint8_t* reverted, int device);

/* ---- parity / debug hooks ----------------------------------------------------------------- */
/* [s_i]Q_i on the twist (on-twist check only, no subgroup requirement).  points: n x 128 B, or one
 * 128-B point used for every scalar when broadcast_point != 0.  Used to build synthetic proofs. */
int zkv_g2_mul_batch(const uint8_t* points, int broadcast_point, const uint8_t* scalars, size_t n, uint8_t* out, uint8_t* reverted, int device);
/* the key a verifier handle uses (for zkv_last_stage_ms) */
const void* zkv_risc0_vk(const zkv_risc0* h);
const void* zkv_sp1_vk(const zkv_sp1* h);
/* vk_x = IC0 + sum s_i IC_{i+1} (compute_vk_x, groth16.rs:51-58): n x k x 32 B scalars -> n x 64 B affine points */
int zkv_vk_x_batch(const zkv_vk* vk, const uint8_t* signals, int k, size_t n, uint8_t* out_points);
/* Montgomery Fp multiply self-test: out[i] = a[i]*b[i] mod p on the GPU (32-byte BE words) */
int zkv_fp_mul_batch(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out, int device);
/* Fp12 tower operations of the pairing kernels on byte operands (n x 384 B = 12 x BE-32, tower order c0.c0.c0, c0.c0.c1, ...), for
 * parity tests against the oracle: op 0 a*b, 1 a^2, 2 a * line(l0,l3,l4) with the line in b's first three Fp2 slots, 3 cyclotomic
 * squaring, 4 inverse, 5/6/7 Frobenius^1/2/3, 8 final exponentiation, 9 Miller loop of the single pair (P, Q) held in b's first six words (P.x, P.y, Q in
 * wire order; a is ignored).  b may be NULL for the unary operations.  op 16 + k (k = 0..8) runs operation k in the shared-memory-resident
 * lazily reduced form the verification kernels use (csrc/lazy.cuh); op 25 = a * (1 + (c3 + c4 v) w), the normalised-line product, with
 * c3, c4 in b's first two Fp2; op 26 = the verification kernels' Miller loop on the single pair of op 9 (fixed pairs switched off). */
int zkv_fp12_op_batch(int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out, int device);
/* G2 membership kernel alone: out[i] = 1 in G2 / 0 on twist but wrong subgroup / 2 invalid encoding or off twist */
int zkv_g2_check_batch(const uint8_t* g2s, size_t n, uint8_t* out, int device);
/* timing of the stage kernels of the last *_device / host call on `device`, milliseconds, for bench.py:
 * [0] decode+hash [1] vk_x [2] g2 check [3] miller [4] final exp ; returns number of entries */
int zkv_last_stage_ms(const void* handle_vk, int device, float* out, int cap);
/* Tuning of ONE key handle (every verifier handle built on that key sees it; there is no process-wide setting).  `handle_vk` is a
 * zkv_vk* or what zkv_risc0_vk / zkv_sp1_vk return.  Returns the previous value (value = ZKV_TUNE_QUERY only reads it), < 0 on error.
 * None of the options changes a status byte or a final-exponentiation value (tests/test_gpu_parity.py).
 *   ZKV_TUNE_OVERLAP (0..64, default 0 = automatic): a device batch is cut into that many pieces whose heavy kernels (Miller segments,
 *     final-exponentiation stages) run on side streams, so the partial last wave of one kernel is back-filled by blocks of another; the
 *     front kernels of all pieces run first.  Automatic: one chain below half a wave of the heavy kernels (SMs x 128 proofs), four pieces
 *     above (measured best at every size from 2^16 to 2^20); batches under 8192 proofs are never cut; 1 = one chain on the main stream with
 *     the per-stage events zkv_last_stage_ms reads.
 *   ZKV_TUNE_NORMALISED_LINES (0/1, default 1): verification path uses the per-key normalised gamma / delta line tables (first
 *     coefficient scaled to 1 by a subfield element: 10 instead of 13 Fp2 products per line); 0 = the unscaled lines of the pairing service.
 *   ZKV_TUNE_MILLER_SEGMENTS (1..16, default 4): chunked batches run the Miller loop as that many kernels (f, R carried in HBM).
 *   ZKV_TUNE_FINAL_EXP_STAGES (0/1, default 1): chunked batches run the final exponentiation as four stage kernels (state in HBM).
 *   ZKV_TUNE_LAYOUT (0/1, default 1): 1 = shared-memory-resident lazily reduced Miller / final-exponentiation kernels (two blocks of
 *     128 threads per SM, 28 Fp slots of shared memory per proof), 0 = the round-1 kernels (thread stack, three / two blocks per SM);
 *     kept for A/B measurements (DESIGN.md section 5). */
#define ZKV_TUNE_OVERLAP 0
#define ZKV_TUNE_NORMALISED_LINES 1
#define ZKV_TUNE_MILLER_SEGMENTS 2
#define ZKV_TUNE_FINAL_EXP_STAGES 3
#define ZKV_TUNE_LAYOUT 4
#define ZKV_TUNE_QUERY (-1)
int zkv_vk_tune(const void* handle_vk, int option, int value);
/* Kernels launched by the verification chains (decode .. final exponentiation, every chunk, segment and stage) since the library was
 * loaded; bench.py reports the difference over its timed region as gpu_launches. */
unsigned long long zkv_launch_count(void);
/* Proofs in one full wave of a heavy kernel on `device` (SM count x resident blocks per SM x 128 threads): kernel 0 = the verification
 * Miller loop, 1 = the final exponentiation (shared-memory layout); 2, 3 = the same two in the round-1 layout.  bench.py times
 * whole-wave launches for its roofline figures.  Negative = error. */
long long zkv_wave_proofs(int device, int kernel);
/* integer-pipe microbenchmark (roofline denominator): returns measured IMAD.WIDE.U32 results/s and
 * Fp-multiplications/s on `device` */
int zkv_imad_peak(int device, double* wide_per_s, double* fpmul_per_s);
/* Page-locked host memory for the batch calls.  When EVERY input array of a zkv_risc0_verify[_integrity]_batch / zkv_sp1_verify_batch /
 * zkv_groth16_verify_batch call lies in page-locked memory (these two functions, cudaHostAlloc or cudaHostRegister), the arrays are uploaded
 * from where they are, one asynchronous copy per array slice; otherwise they are first gathered into the library's own pinned staging buffer
 * by a few host threads (one extra pass over the input in host memory).  Results are identical. */
void* zkv_host_alloc(size_t bytes);
void zkv_host_free(void* p);
/* Test hook (no CUDA involved): the multi-threaded block copy the staging path uses for large input arrays. */
void zkv_test_parallel_copy(void* dst, const void* src, size_t n);
/* Known-answer self test of the production kernels on `device`: the reference's two golden proofs (the RISC Zero seal and the SP1 proof
 * of examples/{risc0,sp1}-verifier/examples/interact.rs, with the embedded keys of risc0/crypto.rs:16-79 and sp1/crypto.rs:7-81) must be
 * accepted and a one-bit tamper of each rejected with VerificationFailed, in both kernel layouts.  0 = pass, ZKV_ERR_STATE = a kernel
 * returned a wrong status (a miscompiled build: DESIGN.md section 5), other negatives as usual.  The Python mirror runs it once per
 * process on the first device before the first call (ZKV_SKIP_SELFTEST=1 skips it). */
int zkv_self_test(int device);

#ifdef __cplusplus
}
#endif
#endif
