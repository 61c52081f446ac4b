// libzkv_b200.so -- host side of the C ABI declared in include/zkv.h.
//
// Mirrors, batch-wise, the reference's verifier objects:
//   zkv_vk      <- common/types.rs:17-23 VerificationKey (+ per-vk device tables built once on the GPU)
//   zkv_risc0   <- risc0/verifier.rs:44-52 storage, :58-76 initialize, :78-104 verify / verify_integrity,
//                  :128-144 calculate_selector, risc0/crypto.rs:136-195 compute_verifier_key_digest
//   zkv_sp1     <- sp1/verifier.rs:31-54,58-111
//   groth16     <- common/groth16.rs:23-128
// Every verification entry point launches the sm_100a kernels of kernels.cuh; there is no CPU path.
// Host work is limited to what the reference does before touching curve points: length / selector
// checks (risc0/verifier.rs:151-170, sp1/verifier.rs:64-83), packing records into pinned staging,
// and the once-per-handle SHA-256 bookkeeping of initialize().
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/zkv.h"
#include "kernels.cuh"
#include "vk_constants.h"

using namespace zkv;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) return fail(ZKV_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

extern "C" const char* zkv_last_error(void) { return g_err.c_str(); }
extern "C" int zkv_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

static constexpr int TPB = 128;                    // threads per block for the heavy kernels
static constexpr size_t MAX_CHUNK = (size_t)1 << 20;   // proofs per device pass (workspace ~0.9 KB / proof)
static inline int nblk(size_t n, int tpb = TPB) { return (int)((n + tpb - 1) / tpb); }

// ------------------------------------------------------------------------------------------ host SHA helpers
static void sha_bytes(uint8_t out[32], const uint8_t* msg, size_t len) { uint32_t h[8]; sha256_msg(h, msg, len); sha256_words_to_bytes(out, h); }
static void sha_str(uint8_t out[32], const char* s) { sha_bytes(out, (const uint8_t*)s, strlen(s)); }
static void bytes_to_words(uint32_t w[8], const uint8_t b[32]) { for (int k = 0; k < 8; k++) w[k] = load_be32(b + 4 * k); }
static const uint8_t FR_R_BE[32] = {0x30, 0x64, 0x4e, 0x72, 0xe1, 0x31, 0xa0, 0x29, 0xb8, 0x50, 0x45, 0xb6, 0x81, 0x81, 0x58, 0x5d,
                                    0x28, 0x33, 0xe8, 0x48, 0x79, 0xb9, 0x70, 0x91, 0x43, 0xe1, 0xf5, 0x93, 0xf0, 0x00, 0x00, 0x01};   // R, groth16.rs:9

// ------------------------------------------------------------------------------------------ per-device context
struct DevCtx {
    int device = 0, sms = 148;
    cudaStream_t stream = nullptr;
    // per-vk tables (device memory, Montgomery form)
    VkDev* d_vk = nullptr; line_t* d_lines = nullptr; nline_t* d_nlines = nullptr; fp12* d_pre = nullptr; g1aff* d_tab = nullptr; g1aff* d_ic0 = nullptr;
    VkDev h_vk; g1aff h_ic0;
    // workspace
    size_t cap = 0;
    fp* px[4] = {nullptr, nullptr, nullptr, nullptr}; fp* py[4] = {nullptr, nullptr, nullptr, nullptr};   // four slices of ONE allocation each, `stride` entries apart (pair-major: the general Miller kernel indexes [j * stride + i])
    size_t stride = 0; uint8_t* pskip = nullptr;                                                          // pairing service: per-pair skip bytes, 4 x stride
    fp2 *qx = nullptr, *qy = nullptr, *tx = nullptr, *ty = nullptr; fp12* f = nullptr; g2j* rst = nullptr; fp* sl = nullptr; fp12* fes = nullptr; size_t fes_cap = 0; uint8_t *flags = nullptr, *status = nullptr;      /* status: scratch flag bytes of vk_x when it runs beside the G2 check */ uint32_t* scal = nullptr; size_t scal_words = 0;
    // staging
    uint8_t* d_in = nullptr; size_t d_in_cap = 0; uint8_t* d_out = nullptr; size_t d_out_cap = 0;
    uint8_t* h_pin = nullptr; size_t h_pin_cap = 0; uint8_t* h_out = nullptr; size_t h_out_cap = 0;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    float stage_ms[5] = {0, 0, 0, 0, 0};
    // overlap: a batch is cut into chunks whose kernel chains run on side streams, so the block scheduler back-fills the partial last
    // wave of one chunk's kernel with blocks of another chunk's (see run_verify)
    static constexpr int NAUX = 4;
    cudaStream_t aux[NAUX] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[NAUX] = {};
    // The workspace above is shared by every call on this key and device.  Host-buffer calls return only when their work is done; the
    // *_device calls are asynchronous, so each records `ev_busy` behind its last kernel and every later user of the workspace, on whatever
    // stream, first waits for it (ctx_acquire); a host call, or a reserve about to free a buffer, waits for it on the host (ctx_wait_idle).
    cudaEvent_t ev_busy = nullptr; bool busy = false;
    std::mutex mu;
};

// Tuning of one key handle (zkv_vk_tune): no process-wide mutable state (SURVEY.md section 8b).  Read once per batch call.
struct Tuning {
    std::atomic<int> overlap_chunks{0};     // a device batch is cut into this many kernel chains on side streams; 0 = automatic (chunk_count)
    std::atomic<int> miller_segments{4};    // chunked batches: segment kernels per Miller loop (state in HBM between them); 4 measured best (profiles/r2_chunk_sweep.txt)
    std::atomic<int> final_exp_stages{1};   // chunked batches: the final exponentiation as four stage kernels
};
static constexpr size_t PAD = 256;          // workspace slack behind a batch: surplus threads of the last block park their state there
// wait on the host for the last asynchronous user of the workspace (caller holds c->mu)
static int ctx_wait_idle(DevCtx* c) {
    if (c->busy) { CK(cudaEventSynchronize(c->ev_busy)); c->busy = false; }
    return 0;
}
// Grow the workspace to n proofs.  Growing frees buffers an earlier asynchronous call may still use, so it waits for that call first.
static int ctx_reserve(DevCtx* c, size_t n, size_t scal_words_per_proof) {
    size_t need = n * scal_words_per_proof;
    if (n > c->cap || n > c->fes_cap || need > c->scal_words) { int rc = ctx_wait_idle(c); if (rc) return rc; }
    if (n > c->cap) {
        cudaFree(c->px[0]); cudaFree(c->py[0]); cudaFree(c->pskip);
        cudaFree(c->qx); cudaFree(c->qy); cudaFree(c->tx); cudaFree(c->ty); cudaFree(c->f); cudaFree(c->flags); cudaFree(c->status); cudaFree(c->rst); cudaFree(c->sl);
        c->cap = 0;
        const size_t st = n + PAD;
        CK(cudaMalloc(&c->px[0], 4 * st * sizeof(fp))); CK(cudaMalloc(&c->py[0], 4 * st * sizeof(fp))); CK(cudaMalloc(&c->pskip, 4 * st));
        CK(cudaMemset(c->px[0], 0, 4 * st * sizeof(fp))); CK(cudaMemset(c->py[0], 0, 4 * st * sizeof(fp))); CK(cudaMemset(c->pskip, 1, 4 * st));
        for (int j = 1; j < 4; j++) { c->px[j] = c->px[0] + j * st; c->py[j] = c->py[0] + j * st; }
        c->stride = st;
        CK(cudaMalloc(&c->qx, st * sizeof(fp2))); CK(cudaMalloc(&c->qy, st * sizeof(fp2))); CK(cudaMalloc(&c->f, st * sizeof(fp12)));
        CK(cudaMemset(c->qx, 0, st * sizeof(fp2))); CK(cudaMemset(c->qy, 0, st * sizeof(fp2)));
        CK(cudaMalloc(&c->tx, st * sizeof(fp2))); CK(cudaMalloc(&c->ty, st * sizeof(fp2)));      // T = -psi^3(B) of the fused subgroup test (k_g2_target)
        CK(cudaMalloc(&c->rst, st * sizeof(g2j))); CK(cudaMalloc(&c->sl, st * 4 * sizeof(fp)));
        CK(cudaMalloc(&c->flags, n)); CK(cudaMalloc(&c->status, n));
        c->cap = n;
    }
    if (n > c->fes_cap) {      // final-exponentiation state: six Fp12 (2.3 KB) per proof
        cudaFree(c->fes); c->fes = nullptr; c->fes_cap = 0;
        CK(cudaMalloc(&c->fes, (n + PAD) * 6 * sizeof(fp12))); c->fes_cap = n;
    }
    if (need > c->scal_words) { cudaFree(c->scal); c->scal_words = 0; CK(cudaMalloc(&c->scal, need * 4)); c->scal_words = need; }
    return 0;
}
static int ctx_stage(DevCtx* c, size_t in_bytes, size_t out_bytes) {
    if (in_bytes > c->d_in_cap) { cudaFree(c->d_in); cudaFreeHost(c->h_pin); c->d_in_cap = 0; c->h_pin_cap = 0;
        size_t cap = in_bytes + in_bytes / 4 + 4096; CK(cudaMalloc(&c->d_in, cap)); CK(cudaMallocHost(&c->h_pin, cap)); c->d_in_cap = cap; c->h_pin_cap = cap; }
    if (out_bytes > c->d_out_cap) { cudaFree(c->d_out); cudaFreeHost(c->h_out); c->d_out_cap = 0; c->h_out_cap = 0;
        size_t cap = out_bytes + out_bytes / 4 + 4096; CK(cudaMalloc(&c->d_out, cap)); CK(cudaMallocHost(&c->h_out, cap)); c->d_out_cap = cap; c->h_out_cap = cap; }
    return 0;
}
// order stream `s` after the last asynchronous user of the workspace (caller holds c->mu)
static int ctx_acquire(DevCtx* c, cudaStream_t s) { if (c->busy) CK(cudaStreamWaitEvent(s, c->ev_busy, 0)); return 0; }
static int ctx_release_async(DevCtx* c, cudaStream_t s) { CK(cudaEventRecord(c->ev_busy, s)); c->busy = true; return 0; }
// A *_device call: run(s) enqueues its work on the caller's stream s (NULL is the legacy default stream, as for any CUDA call), and later
// users of the workspace are ordered behind it.
template <class F>
static int device_call(DevCtx* c, int device, void* stream, F run) {
    std::lock_guard<std::mutex> lk(c->mu);
    CK(cudaSetDevice(device));
    cudaStream_t s = (cudaStream_t)stream;
    int rc = run(s);
    if (!rc) rc = ctx_release_async(c, s);
    return rc;
}
static void ctx_free(DevCtx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaFree(c->px[0]); cudaFree(c->py[0]); cudaFree(c->pskip);
    cudaFree(c->qx); cudaFree(c->qy); cudaFree(c->tx); cudaFree(c->ty); cudaFree(c->f); cudaFree(c->flags); cudaFree(c->status); cudaFree(c->scal); cudaFree(c->rst); cudaFree(c->sl); cudaFree(c->fes);
    cudaFree(c->d_in); cudaFree(c->d_out); cudaFreeHost(c->h_pin); cudaFreeHost(c->h_out);
    cudaFree(c->d_vk); cudaFree(c->d_lines); cudaFree(c->d_nlines); cudaFree(c->d_pre); cudaFree(c->d_tab); cudaFree(c->d_ic0);
    for (auto& e : c->ev) if (e) cudaEventDestroy(e);
    for (auto& e : c->ev_join) if (e) cudaEventDestroy(e);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_busy) cudaEventDestroy(c->ev_busy);
    for (auto& a : c->aux) if (a) cudaStreamDestroy(a);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

// ------------------------------------------------------------------------------------------ verification key
struct zkv_vk {
    int vm = 0, n_ic = 0;
    uint8_t alpha[64], beta[128], gamma[128], delta[128];
    std::vector<uint8_t> ic;
    std::vector<DevCtx*> devs;
    int valid = 1;     // every key point decodes under EIP-196/197 (else each verification's precompile call reverts -> false)
    mutable Tuning tune;
};
static DevCtx* vk_ctx(const zkv_vk* vk, int device) { for (auto* c : vk->devs) if (c->device == device) return c; return nullptr; }

// streams, events and kernel attributes of a context on c->device (the workspace is allocated by the first batch)
static int ctx_init(DevCtx* c) {
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceGetAttribute(&c->sms, cudaDevAttrMultiProcessorCount, c->device));
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    for (auto& e : c->ev) CK(cudaEventCreate(&e));
    for (auto& a : c->aux) CK(cudaStreamCreateWithFlags(&a, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c->ev_busy, cudaEventDisableTiming));
    for (auto& e : c->ev_join) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CK(cudaFuncSetAttribute(k_miller_lz, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM_MILLER));
    CK(cudaFuncSetAttribute(k_final_exp_lz, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_pairing_lz, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_miller_lz_keys, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM_MILLER));
    CK(cudaFuncSetAttribute(k_final_exp_lz_keys, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM_BYTES));
    return 0;
}
static int vk_build_on(zkv_vk* vk, DevCtx* c) {
    int rc = ctx_init(c); if (rc) return rc;
    int nt = vk->n_ic - 1;
    CK(cudaMalloc(&c->d_vk, sizeof(VkDev))); CK(cudaMalloc(&c->d_lines, sizeof(line_t) * 3 * ZKV_LINES_PER_G2)); CK(cudaMalloc(&c->d_nlines, sizeof(nline_t) * 2 * ZKV_LINES_PER_G2)); CK(cudaMalloc(&c->d_pre, sizeof(fp12)));
    CK(cudaMalloc(&c->d_tab, sizeof(g1aff) * (size_t)nt * ZKV_WIN_PER_SCALAR * ZKV_WIN_ENTRIES)); CK(cudaMalloc(&c->d_ic0, sizeof(g1aff)));
    uint8_t* d_bytes; size_t nb = 64 + 384 + vk->ic.size();
    CK(cudaMalloc(&d_bytes, nb));
    std::vector<uint8_t> hb(nb);
    memcpy(hb.data(), vk->alpha, 64); memcpy(hb.data() + 64, vk->beta, 128); memcpy(hb.data() + 192, vk->gamma, 128); memcpy(hb.data() + 320, vk->delta, 128);
    memcpy(hb.data() + 448, vk->ic.data(), vk->ic.size());
    CK(cudaMemcpyAsync(d_bytes, hb.data(), nb, cudaMemcpyHostToDevice, c->stream));
    VkDev init; memset(&init, 0, sizeof init); init.valid = 1; init.norm_ok = 1;
    CK(cudaMemcpyAsync(c->d_vk, &init, sizeof init, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(c->d_lines, 0, sizeof(line_t) * 3 * ZKV_LINES_PER_G2, c->stream));
    CK(cudaMemsetAsync(c->d_nlines, 0, sizeof(nline_t) * 2 * ZKV_LINES_PER_G2, c->stream));
    k_vk_setup<<<4, 1, 0, c->stream>>>(d_bytes, d_bytes + 64, c->d_vk, c->d_lines, c->d_nlines);
    k_ic_tables<<<nt, ZKV_WIN_PER_SCALAR, 0, c->stream>>>(d_bytes + 448, c->d_tab, c->d_ic0, c->d_vk);
    k_vk_miller_ab<<<1, 1, 0, c->stream>>>(c->d_vk, c->d_lines, c->d_pre);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&c->h_vk, c->d_vk, sizeof(VkDev), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(&c->h_ic0, c->d_ic0, sizeof(g1aff), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaFree(d_bytes));
    if (!c->h_vk.valid) vk->valid = 0;
    return 0;
}

extern "C" void zkv_vk_free(zkv_vk* vk) {
    if (!vk) return;
    for (auto* c : vk->devs) ctx_free(c);
    delete vk;
}
extern "C" int zkv_vk_load(int vm_type, const uint8_t alpha[64], const uint8_t beta[128], const uint8_t gamma[128], const uint8_t delta[128],
                           const uint8_t* ic, int n_ic, const int* devices, int n_dev, zkv_vk** out) {
    if (!out || !alpha || !beta || !gamma || !delta || !ic) return fail(ZKV_ERR_ARG, "zkv_vk_load: null argument");
    if (vm_type != ZKV_VM_RISC0 && vm_type != ZKV_VM_SP1) return fail(ZKV_ERR_ARG, "zkv_vk_load: vm_type");
    if (n_ic < 2 || n_ic > 16) return fail(ZKV_ERR_ARG, "zkv_vk_load: n_ic must be 2..16");
    int ndev_sys = zkv_device_count();
    if (ndev_sys <= 0) return fail(ZKV_ERR_CUDA, "zkv_vk_load: no CUDA device (this library has no CPU path)");
    std::vector<int> devs;
    if (!devices || n_dev <= 0) devs.push_back(0); else devs.assign(devices, devices + n_dev);
    for (int d : devs) if (d < 0 || d >= ndev_sys) return fail(ZKV_ERR_ARG, "zkv_vk_load: bad device index");
    zkv_vk* vk = new zkv_vk();
    vk->vm = vm_type; vk->n_ic = n_ic;
    memcpy(vk->alpha, alpha, 64); memcpy(vk->beta, beta, 128); memcpy(vk->gamma, gamma, 128); memcpy(vk->delta, delta, 128);
    vk->ic.assign(ic, ic + 64 * (size_t)n_ic);
    for (int d : devs) {
        DevCtx* c = new DevCtx(); c->device = d; vk->devs.push_back(c);
        int rc = vk_build_on(vk, c);
        // the Miller loop needs the normalised line table of every finite gamma / delta of a valid key: a line coefficient l0 vanishes for
        // no point of G2 (DESIGN.md section 4), but key bytes come from outside
        if (!rc && c->h_vk.valid && !c->h_vk.norm_ok) rc = fail(ZKV_ERR_ARG, "zkv_vk_load: the key has no normalised gamma / delta line tables (a vanishing line coefficient)");
        if (rc) { zkv_vk_free(vk); return rc; }
    }
    *out = vk;
    return 0;
}
extern "C" int zkv_vk_load_risc0(const int* devices, int n_dev, zkv_vk** out) {
    const uint8_t* p = ZKV_RISC0_VK_AB_GD;
    return zkv_vk_load(ZKV_VM_RISC0, p, p + 64, p + 192, p + 320, ZKV_RISC0_VK_IC, 6, devices, n_dev, out);
}
extern "C" int zkv_vk_load_sp1(const int* devices, int n_dev, zkv_vk** out) {
    const uint8_t* p = ZKV_SP1_VK_AB_GD;
    return zkv_vk_load(ZKV_VM_SP1, p, p + 64, p + 192, p + 320, ZKV_SP1_VK_IC, 3, devices, n_dev, out);
}

// ------------------------------------------------------------------------------------------ the device pipeline
enum SigMode { SIG_GENERIC, SIG_RISC0_VERIFY, SIG_RISC0_INTEGRITY, SIG_SP1 };
struct Job {
    const zkv_vk* vk = nullptr; size_t n = 0;
    // proof records (device): rec i at recs + i*stride (or at recs + rec_off[i] - rec_base when rec_off is set: the caller's concatenated
    // blobs, front checks on the device), 8 x BE-32 at +off; selector (if any) in the first 4 bytes
    const uint8_t* recs = nullptr; size_t stride = 0, off = 0; int check_selector = 0; uint32_t selector_le = 0;
    const uint64_t* rec_off = nullptr; uint64_t rec_base = 0, pv_base = 0;
    SigMode mode = SIG_GENERIC;
    const uint8_t *sig_a = nullptr, *sig_b = nullptr;     // generic: signals | risc0: image_ids, journals (or claims) | sp1: vkeys, public values
    const uint64_t* pv_off = nullptr; size_t pv_stride = 0; int k = 0;
    Risc0HashConsts hc = {}; g1aff base = {}; int all_fail = 0;
    uint8_t* d_status = nullptr;
};
__global__ void k_status_all_fail(int n, const uint8_t* flags, uint8_t* status) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) status[i] = reject_status(flags[i]);
}
static std::atomic<unsigned long long> g_launches{0};   // kernels launched by the verification chains since load (bench.py's gpu_launches; a counter, not a setting)
extern "C" unsigned long long zkv_launch_count(void) { return g_launches.load(); }
// every kernel of a verification chain (enqueue_chain, keyset_pass) is launched through here, so the counter cannot miss one
template <class... P, class... A>
static void launch(void (*kernel)(P...), int grid, int block, size_t smem, cudaStream_t s, A&&... args) {
    kernel<<<grid, block, smem, s>>>(std::forward<A>(args)...);
    g_launches++;
}
extern "C" int zkv_vk_tune(const void* handle_vk, int option, int value) {
    const zkv_vk* vk = (const zkv_vk*)handle_vk;
    if (!vk) return fail(ZKV_ERR_ARG, "zkv_vk_tune: null key");
    std::atomic<int>* f; int lo, hi;
    switch (option) {
        case ZKV_TUNE_OVERLAP: f = &vk->tune.overlap_chunks; lo = 0; hi = 64; break;
        case ZKV_TUNE_MILLER_SEGMENTS: f = &vk->tune.miller_segments; lo = 1; hi = 16; break;
        case ZKV_TUNE_FINAL_EXP_STAGES: f = &vk->tune.final_exp_stages; lo = 0; hi = 1; break;
        case ZKV_TUNE_NORMALISED_LINES: case ZKV_TUNE_LAYOUT:          // fixed at 1: the shared-memory kernels with normalised lines are the only ones
            if (value == ZKV_TUNE_QUERY || value == 1) return 1;
            return fail(ZKV_ERR_ARG, "zkv_vk_tune: the round-1 kernels and the unscaled verification lines were removed; this option is fixed at 1");
        default: return fail(ZKV_ERR_ARG, "zkv_vk_tune: unknown option");
    }
    if (value == ZKV_TUNE_QUERY) return f->load();
    if (value < lo || value > hi) return fail(ZKV_ERR_ARG, "zkv_vk_tune: value out of range");
    return f->exchange(value);
}

static const bool g_debug_sync = getenv("ZKV_DEBUG_SYNC") != nullptr;      // diagnostics: synchronise after every kernel of a chain and name the one that failed
#define DBG(name) do { if (g_debug_sync) { cudaError_t e_ = cudaStreamSynchronize(s); if (e_ != cudaSuccess) return fail(ZKV_ERR_CUDA, std::string(name) + ": " + cudaGetErrorString(e_)); } } while (0)
// The end of the front phase on workspace proofs [o, o+m): vk_x (vkx(flag array) enqueues it on s) and the G2 check.  The Miller loop
// (k_miller_lz / k_miller_lz_keys) finishes the subgroup test in its last segment; the check's slot holds k_g2_target, which writes the
// point T = -psi^3(B) that test compares against, and leaves the flags alone.
// fork: the front phase of a whole chunked batch on the call's main stream.  vk_x and the G2 check are independent (the check reads what the
// decode kernel wrote, both touch disjoint flag bits of different proofs' bytes only through their own thread), and each is 1.7 waves of its
// own block shape at 2^16 proofs: side by side on two streams they fill each other's partial waves.  F_SKIPX (vk_x = infinity) and F_INVALID
// (B outside the subgroup) live in the same flag byte of a proof, so the two kernels must not write it concurrently: vk_x gets a flag array
// of its own (the front-phase scratch c->status) that is OR-ed in by the G2 check's stream afterwards.
template <class VkX>
static int enqueue_vkx_g2(DevCtx* c, size_t o, int m, uint8_t* flags, cudaStream_t s, bool fork, bool timed, VkX vkx) {
    auto g2 = [&](cudaStream_t gs) { launch(k_g2_target, nblk(m), TPB, 0, gs, m, c->qx + o, c->qy + o, c->tx + o, c->ty + o); };
    if (fork) {
        CK(cudaEventRecord(c->ev_fork, s)); CK(cudaStreamWaitEvent(c->aux[0], c->ev_fork, 0));
        g2(c->aux[0]);
        CK(cudaMemsetAsync(c->status + o, 0, m, s));
        vkx(c->status + o);
        CK(cudaEventRecord(c->ev_join[0], c->aux[0])); CK(cudaStreamWaitEvent(s, c->ev_join[0], 0));
        launch(k_or_flags, nblk(m, 256), 256, 0, s, m, flags, c->status + o);
        return 0;
    }
    vkx(flags);
    if (timed) CK(cudaEventRecord(c->ev[2], s));
    DBG("decode / signals / vk_x");
    g2(s);
    DBG("G2 check");
    if (timed) CK(cudaEventRecord(c->ev[3], s));
    return 0;
}
// NAF digits hi .. lo (of top .. 0) that segment k of an S-segment Miller loop runs
static std::pair<int, int> miller_segment(int k, int S) {
    const int top = ZKV_ATE_NAF_LEN - 2;
    return {top - (top + 1) * k / S, top - (top + 1) * (k + 1) / S + 1};
}
// MillerArgs of the verification path at workspace offset o: the pair (A, B), then (vk_x, gamma) and (C, delta) from tabled lines
static MillerArgs verify_miller_args(const DevCtx* c, size_t o) {
    MillerArgs a; memset(&a, 0, sizeof a);
    a.px[0] = c->px[0] + o; a.py[0] = c->py[0] + o; a.px[1] = c->px[2] + o; a.py[1] = c->py[2] + o; a.px[2] = c->px[3] + o; a.py[2] = c->py[3] + o;
    a.qx = c->qx + o; a.qy = c->qy + o; a.nfixed = 2;
    a.skip_bit[0] = F_SKIP0; a.skip_bit[1] = F_SKIPX; a.skip_bit[2] = F_SKIPC;
    return a;
}
// the kernel chain for proofs [o, o+m) of job j on stream s
// jo: offset of the first proof inside the job's buffers, o: offset inside the device workspace
// timed: record the per-stage events, and run the Miller loop and the final exponentiation as one launch each (no segments, no stages)
// phases: 1 = the front kernels (decode, public-input hashing, vk_x, G2 check), 2 = the heavy ones (Miller loop, final exponentiation), 3 = both
// fork_front: phase 1 of a whole chunked batch on the call's main stream (enqueue_vkx_g2)
static int enqueue_chain(DevCtx* c, const Job& j, size_t jo, size_t o, int m, cudaStream_t s, bool timed, int phases = 3, bool fork_front = false) {
    const zkv_vk* vk = j.vk;
    int ns = (j.mode == SIG_GENERIC) ? j.k : 2;
    uint32_t* scal = c->scal + o * (size_t)ns * 8;
    uint8_t* flags = c->flags + o;
    if (phases & 1) {
        if (timed) CK(cudaEventRecord(c->ev[0], s));
        launch(k_decode, nblk(m), TPB, 0, s, m, j.rec_off ? j.recs : j.recs + jo * j.stride, j.stride, j.off, j.selector_le, j.check_selector, vk->vm, j.rec_off ? j.rec_off + jo : nullptr, j.rec_base, c->px[0] + o, c->py[0] + o, c->qx + o, c->qy + o, c->px[3] + o, c->py[3] + o, flags);
        const g1aff* tab = c->d_tab; int nwin = ZKV_WIN_PER_SCALAR;
        switch (j.mode) {
            case SIG_GENERIC: launch(k_generic_signals, nblk(m), TPB, 0, s, m, j.k, j.sig_a + jo * (size_t)j.k * 32, scal, flags); break;
            case SIG_RISC0_VERIFY: launch(k_risc0_signals, nblk(m), TPB, 0, s, m, j.sig_a + jo * 32, j.sig_b + jo * 32, nullptr, 0, j.hc, scal); break;
            case SIG_RISC0_INTEGRITY: launch(k_risc0_signals, nblk(m), TPB, 0, s, m, nullptr, nullptr, j.sig_a + jo * 32, 1, j.hc, scal); break;
            case SIG_SP1: launch(k_sp1_signals, nblk(m), TPB, 0, s, m, j.sig_a + jo * 32, j.pv_off ? j.sig_b : j.sig_b + jo * j.pv_stride, j.pv_off ? j.pv_off + jo : nullptr, j.pv_base, j.pv_stride, scal, flags); break;
        }
        if (j.mode == SIG_RISC0_VERIFY || j.mode == SIG_RISC0_INTEGRITY) { tab = c->d_tab + (size_t)2 * ZKV_WIN_PER_SCALAR * ZKV_WIN_ENTRIES; nwin = 32; }   // claim_lo / claim_hi are 128-bit
        if (timed) CK(cudaEventRecord(c->ev[1], s));
        if (j.all_fail || !vk->valid) {
            launch(k_status_all_fail, nblk(m), TPB, 0, s, m, flags, j.d_status + jo);
            if (timed) for (int e = 2; e < 6; e++) CK(cudaEventRecord(c->ev[e], s));
            CK(cudaGetLastError());
            return 0;
        }
        int rc = enqueue_vkx_g2(c, o, m, flags, s, fork_front, timed, [&](uint8_t* fl) {
            launch(k_vkx, nblk(m), TPB, 0, s, m, scal, ns, nwin, tab, j.base, c->px[2] + o, c->py[2] + o, fl);
        });
        if (rc) return rc;
        if (!(phases & 2)) { CK(cudaGetLastError()); return 0; }
    }
    MillerArgs a = verify_miller_args(c, o);
    a.tabs[0] = c->d_lines + 1 * ZKV_LINES_PER_G2; a.tabs[1] = c->d_lines + 2 * ZKV_LINES_PER_G2; a.pre = c->d_pre;
    a.ntabs[0] = c->d_nlines; a.ntabs[1] = c->d_nlines + ZKV_LINES_PER_G2;
    a.vk_skip = (uint8_t)((c->h_vk.g2_inf[1] ? 2 : 0) | (c->h_vk.g2_inf[2] ? 4 : 0));
    const int segs = vk->tune.miller_segments.load(), stages = vk->tune.final_exp_stages.load();
    // shared-memory-resident kernels (lazy.cuh): segments / stages when chunked, one launch each in a timed single chain
    const int S = (segs > 1 && !timed) ? segs : 1;
    for (int k = 0; k < S; k++) {
        auto [hi, lo] = miller_segment(k, S);
        launch(k_miller_lz, nblk(m, LZ_NT), LZ_NT, LZ_SMEM_MILLER, s, m, a, flags, c->tx + o, c->ty + o, c->f + o, c->rst + o, c->sl + 4 * o, hi, lo, k == 0, k == S - 1);
        DBG("k_miller_lz");
    }
    if (timed) CK(cudaEventRecord(c->ev[4], s));
    if (stages && !timed) for (int st = 0; st < 4; st++) launch(k_final_exp_lz, nblk(m, LZ_NT), LZ_NT, LZ_SMEM_BYTES, s, m, st, st, c->f + o, c->fes + 6 * o, flags, j.d_status + jo, nullptr, 0);
    else launch(k_final_exp_lz, nblk(m, LZ_NT), LZ_NT, LZ_SMEM_BYTES, s, m, 0, 3, c->f + o, c->fes + 6 * o, flags, j.d_status + jo, nullptr, 0);
    DBG("final exponentiation");
    if (timed) CK(cudaEventRecord(c->ev[5], s));
    CK(cudaGetLastError());
    return 0;
}
// Chunks of a device batch (measured on B200: tools/sweep_chunks.sh, tools/sweep_segments.sh, profiles/r2_chunk_sweep.txt).  The heavy kernels
// hold 2 blocks of 128 threads per SM (one wave = SMs x 256 proofs), and a batch is rarely a whole number of waves: 2^16 proofs are 1.73.
// Cut into FOUR chunks whose Miller loops run as 4 segment kernels and whose final exponentiations run as 4 stage kernels on four side
// streams, the block scheduler back-fills one chunk's partial wave with another chunk's blocks; the front kernels (decode, hashing, vk_x, G2
// check) run before all of that, over the whole batch, because interleaved with heavy blocks they run at a fraction of their occupancy and
// take block slots from them.  On the final build this schedule wins at every size from half a wave up (2^16: 31.3 ms against 35.0 for one
// chain; 2^17: 60.6 against 62.7; 2^18: 121.5 against 123.8; 2^20: 488 against 499 ms); more chunks are worse at every size.  (While the front
// kernels still ran inside the chunks and the Miller loop had 8 segments, one serial chain was the faster schedule from two waves on, and for
// a while it was the automatic choice there.)  Automatic (setting 0): one chain below half a wave, four chunks above; a positive setting forces
// that many chunks (1 = one chain on the main stream with the per-stage events zkv_last_stage_ms reads).
static size_t wave_proofs_of(const DevCtx* c) { return (size_t)c->sms * 2 * ZKV_HTPB; }
static int chunk_count(const DevCtx* c, size_t n, int setting) {
    if (n < (size_t)8192) return 1;
    if (setting >= 1) return setting;
    return n < wave_proofs_of(c) / 2 ? 1 : 4;
}
// Proofs per chunk when n proofs are cut into `chunks`: a multiple of the heavy kernels' block size, so no chunk carries a second partial block.
static size_t chunk_size(size_t n, int chunks) {
    size_t per = (n + chunks - 1) / chunks;
    return (per + ZKV_HTPB - 1) / ZKV_HTPB * ZKV_HTPB;
}
// Fork `chunks` side streams off `main`, run fn(chunk_begin, chunk_len, stream) on them round-robin, join back into `main`.
template <class F>
static int fork_join(DevCtx* c, cudaStream_t main, size_t n, int chunks, F fn) {
    const size_t per = chunk_size(n, chunks);
    CK(cudaEventRecord(c->ev_fork, main));
    int used = 0, k = 0;
    for (size_t o = 0; o < n; o += per, k++) {
        cudaStream_t s = c->aux[k % DevCtx::NAUX];
        if (k < DevCtx::NAUX) { CK(cudaStreamWaitEvent(s, c->ev_fork, 0)); used = k + 1; }
        int rc = fn(o, (int)std::min(per, n - o), s); if (rc) return rc;
    }
    for (int a = 0; a < used; a++) { CK(cudaEventRecord(c->ev_join[a], c->aux[a])); CK(cudaStreamWaitEvent(main, c->ev_join[a], 0)); }
    return 0;
}
// enqueue all stages of one batch on stream s (asynchronous; completion is ordered on s); caller holds c->mu and has set the device
static int run_verify(DevCtx* c, const Job& j, cudaStream_t s) {
    if (j.n == 0) return 0;
    int ns = (j.mode == SIG_GENERIC) ? j.k : 2;
    int rc = ctx_acquire(c, s); if (rc) return rc;
    rc = ctx_reserve(c, j.n, (size_t)ns * 8); if (rc) return rc;
    int chunks = chunk_count(c, j.n, j.vk->tune.overlap_chunks.load());
    if (chunks <= 1) return enqueue_chain(c, j, 0, 0, (int)j.n, s, true);
    if (j.all_fail || !j.vk->valid) return enqueue_chain(c, j, 0, 0, (int)j.n, s, false);
    // the front kernels run once over the whole batch (at their own full occupancy), only the heavy kernels are chunked over the side streams
    rc = enqueue_chain(c, j, 0, 0, (int)j.n, s, false, 1, true); if (rc) return rc;
    return fork_join(c, s, j.n, chunks, [&](size_t o, int m, cudaStream_t hs) { return enqueue_chain(c, j, o, o, m, hs, false, 2); });
}
static void collect_stage_ms(DevCtx* c);
// memcpy of a large block by up to four threads (one thread moves 5 - 10 GB/s into pinned memory: a 45 MB piece would cost as much as a wave of kernels)
static void pcopy(void* dst, const void* src, size_t n) {
    const size_t MIN = (size_t)2 << 20;
    int parts = (int)std::min<size_t>(4, n / MIN);
    if (parts <= 1) { memcpy(dst, src, n); return; }
    std::vector<std::thread> th;
    const size_t per = ((n + parts - 1) / parts + 63) / 64 * 64;      // CEILING of n / parts: parts x per >= n, the slices cover every byte
    for (int t = 1; t < parts; t++) { size_t o = per * t; if (o >= n) break; size_t l = std::min(per, n - o); th.emplace_back([=]() { memcpy((uint8_t*)dst + o, (const uint8_t*)src + o, l); }); }
    memcpy(dst, src, std::min(per, n));
    for (auto& t : th) t.join();
}

// Host-buffer form of proofs [b, e) on one device, in passes of up to MAX_CHUNK proofs, pipelined: a pass is cut like run_verify cuts a
// batch, and every piece gets its own pack (into its slice of the pinned staging buffer) -> H2D -> kernel chain -> D2H on a side stream,
// so packing and copying piece k+1 overlap the kernels of piece k.  pack(first, count, dst) writes the input block of proofs
// [first, first + count) and returns its size in bytes; job(first, count, d_block) describes them, with pointers into their device input
// block (host_pass fills in the key, the count and the status slice).  The status bytes go to status_out[b, e).
// Where a piece's input block is assembled: in the pinned staging buffer (memcpy; large segments by several threads), or - when every source
// array of the call already lives in page-locked memory (cudaHostAlloc / cudaHostRegister) - straight in device memory, one asynchronous
// upload per segment from the caller's own arrays, with no host copy at all.
struct Sink {
    uint8_t* host; uint8_t* dev; cudaStream_t s; int bad;
    void put(size_t off, const void* src, size_t n, bool big = false) {
        if (!n) return;
        if (host) { if (big) pcopy(host + off, src, n); else memcpy(host + off, src, n); }
        else if (cudaMemcpyAsync(dev + off, src, n, cudaMemcpyHostToDevice, s) != cudaSuccess) bad = 1;
    }
};
static bool is_pinned(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}
// one pass of proofs [s0, s0 + m); on return c->h_out[0..m) holds their status bytes
template <class Pack, class MakeJob>
static int host_pass(DevCtx* c, const zkv_vk* vk, size_t s0, size_t m, int ns, Pack& pack, MakeJob& job, bool direct) {
    int rc = ctx_reserve(c, m, (size_t)ns * 8); if (rc) return rc;
    // Pieces of the pass, in upload order: `chunks` equal pieces (multiples of the heavy kernels' block size), each with its own side stream.
    // Every piece runs its front kernels first, side by side with the others', then the heavy ones (chunk_count above); with more pieces
    // than side streams (a forced setting) each piece simply runs its whole chain on stream k mod NAUX.
    struct Piece { size_t first, cnt; };
    std::vector<Piece> pcs;
    const size_t per = chunk_size(m, chunk_count(c, m, vk->tune.overlap_chunks.load()));
    for (size_t f = 0; f < m; f += per) pcs.push_back({f, std::min(per, m - f)});
    const int np = (int)pcs.size();
    // pack(first, cnt, nullptr) returns the size of a piece's block, so every piece's region of the pinned staging buffer is known up front
    // and the pieces can be packed by concurrent host threads: piece 0 on this thread, the others on up to 6 helpers (helper h packs pieces
    // h + 1, h + 1 + H, ...); ready[k] flips when piece k's block is complete.  Packing is a handful of bulk memcpy per piece.
    std::vector<size_t> bytes(np, 0), offs(np + 1, 0);
    for (int k = 0; k < np; k++) { bytes[k] = pack(s0 + pcs[k].first, pcs[k].cnt, (Sink*)nullptr); offs[k + 1] = offs[k] + (bytes[k] + 255) / 256 * 256; }
    rc = ctx_stage(c, offs[np], m); if (rc) return rc;
    const int H = direct ? 0 : std::min(np - 1, 6);
    std::vector<std::atomic<int>> ready(np);
    for (auto& r : ready) r.store(direct ? 1 : 0);
    std::vector<std::thread> helpers;
    for (int h = 0; h < H; h++) helpers.emplace_back([&, h]() {
        for (int k = h + 1; k < np; k += H) { Sink sk{c->h_pin + offs[k], nullptr, nullptr, 0}; pack(s0 + pcs[k].first, pcs[k].cnt, &sk); ready[k].store(1, std::memory_order_release); }
    });
    if (!direct) { Sink sk{c->h_pin, nullptr, nullptr, 0}; pack(s0 + pcs[0].first, pcs[0].cnt, &sk); ready[0].store(1); }
    const bool split = np > 1 && np <= DevCtx::NAUX;
    std::vector<cudaEvent_t> evs;                    // front-done event per piece
    if (split) { evs.resize((size_t)np, nullptr); for (auto& e : evs) if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) rc = fail(ZKV_ERR_CUDA, "cudaEventCreate"); }
    std::vector<Job> jobs(np);
    auto kstream = [&](int k) { return np == 1 ? c->stream : c->aux[k % DevCtx::NAUX]; };
    for (int k = 0; k < np && !rc; k++) {
        const size_t first = pcs[k].first, cnt = pcs[k].cnt, in_off = offs[k];
        cudaStream_t s = kstream(k);
        while (!ready[k].load(std::memory_order_acquire)) std::this_thread::yield();
        if (direct) { Sink sk{nullptr, c->d_in + in_off, s, 0}; pack(s0 + first, cnt, &sk); rc = sk.bad ? fail(ZKV_ERR_CUDA, "cudaMemcpyAsync (page-locked caller memory to device)") : 0; }
        else rc = cudaMemcpyAsync(c->d_in + in_off, c->h_pin + in_off, bytes[k], cudaMemcpyHostToDevice, s) == cudaSuccess ? 0 : fail(ZKV_ERR_CUDA, "cudaMemcpyAsync (host to device)");
        if (rc) break;
        jobs[k] = job(s0 + first, cnt, c->d_in + in_off);
        jobs[k].vk = vk; jobs[k].n = cnt; jobs[k].d_status = c->d_out + first;
        if (split && !(jobs[k].all_fail || !vk->valid)) {
            rc = enqueue_chain(c, jobs[k], 0, first, (int)cnt, s, false, 1);
            if (!rc && cudaEventRecord(evs[k], s) != cudaSuccess) rc = fail(ZKV_ERR_CUDA, "event (front done)");
            continue;
        }
        rc = enqueue_chain(c, jobs[k], 0, first, (int)cnt, s, np == 1);
        if (!rc && cudaMemcpyAsync(c->h_out + first, c->d_out + first, cnt, cudaMemcpyDeviceToHost, s) != cudaSuccess) rc = fail(ZKV_ERR_CUDA, "cudaMemcpyAsync (device to host)");
    }
    for (int k = 0; split && k < np && !rc; k++) {
        if (jobs[k].all_fail || !vk->valid) continue;        // (that piece ran its whole chain above)
        cudaStream_t s = kstream(k);
        for (int o = 0; o < np && !rc; o++) if (o != k && !(jobs[o].all_fail || !vk->valid) && cudaStreamWaitEvent(s, evs[o], 0) != cudaSuccess) rc = fail(ZKV_ERR_CUDA, "event wait (front done)");
        if (!rc) rc = enqueue_chain(c, jobs[k], 0, pcs[k].first, (int)pcs[k].cnt, s, false, 2);
        if (!rc && cudaMemcpyAsync(c->h_out + pcs[k].first, c->d_out + pcs[k].first, pcs[k].cnt, cudaMemcpyDeviceToHost, s) != cudaSuccess) rc = fail(ZKV_ERR_CUDA, "cudaMemcpyAsync (device to host)");
    }
    for (auto& t : helpers) t.join();
    if (rc) { cudaDeviceSynchronize(); for (auto e : evs) if (e) cudaEventDestroy(e); return rc; }
    if (np == 1) { CK(cudaStreamSynchronize(c->stream)); collect_stage_ms(c); }
    else for (int a = 0; a < DevCtx::NAUX; a++) CK(cudaStreamSynchronize(c->aux[a]));
    for (auto e : evs) if (e) cudaEventDestroy(e);
    return 0;
}
template <class Pack, class MakeJob>
static int host_pipeline(DevCtx* c, const zkv_vk* vk, size_t b, size_t e, int ns, uint8_t* status_out, Pack pack, MakeJob job, bool direct) {
    int rc = ctx_wait_idle(c);      // a host call blocks anyway: wait out an earlier asynchronous device call here
    for (size_t s0 = b; s0 < e && !rc; s0 += MAX_CHUNK) {
        const size_t m = std::min(MAX_CHUNK, e - s0);
        rc = host_pass(c, vk, s0, m, ns, pack, job, direct);
        if (!rc) memcpy(status_out + s0, c->h_out, m);
    }
    return rc;
}
static void collect_stage_ms(DevCtx* c) {
    for (int e = 0; e < 5; e++) { float ms = 0; if (cudaEventElapsedTime(&ms, c->ev[e], c->ev[e + 1]) != cudaSuccess) { cudaGetLastError(); ms = 0; } c->stage_ms[e] = ms; }
}

// Split `n` items over the contexts (one per device) in contiguous ranges and run fn(ctx, begin, end) on one host thread per device.
template <class F>
static int for_each_device(const std::vector<DevCtx*>& devs, size_t n, F fn) {
    size_t nd = devs.size();
    if (nd == 1 || n < 4096) {
        DevCtx* c = devs[0];
        std::lock_guard<std::mutex> lk(c->mu);
        CK(cudaSetDevice(c->device));
        return fn(c, (size_t)0, n);
    }
    std::vector<int> rcs(nd, 0); std::vector<std::string> errs(nd);
    std::vector<std::thread> th;
    for (size_t d = 0; d < nd; d++) {
        size_t b = n * d / nd, e = n * (d + 1) / nd;
        th.emplace_back([&, d, b, e]() {
            DevCtx* c = devs[d];
            std::lock_guard<std::mutex> lk(c->mu);
            if (cudaSetDevice(c->device) != cudaSuccess) { rcs[d] = ZKV_ERR_CUDA; errs[d] = "cudaSetDevice"; return; }
            rcs[d] = fn(c, b, e);
            if (rcs[d]) errs[d] = g_err;
        });
    }
    for (auto& t : th) t.join();
    for (size_t d = 0; d < nd; d++) if (rcs[d]) return fail(rcs[d], errs[d]);
    return 0;
}

// ------------------------------------------------------------------------------------------ generic Groth16
static bool offsets_ok(const uint64_t* off, size_t n) { for (size_t i = 0; i < n; i++) if (off[i + 1] < off[i]) return false; return true; }
extern "C" int zkv_groth16_verify_batch(const zkv_vk* vk, const uint8_t* proofs, const uint8_t* signals, int k, size_t n, uint8_t* status_out) {
    if (!vk || (n && (!proofs || !status_out)) || k < 0 || (n && k && !signals)) return fail(ZKV_ERR_ARG, "zkv_groth16_verify_batch: bad argument");
    if (n == 0) return 0;
    if (k + 1 != vk->n_ic) { memset(status_out, ZKV_VERIFICATION_FAILED, n); return 0; }        // groth16.rs:32
    const bool direct = n >= 4096 && is_pinned(proofs) && (k == 0 || is_pinned(signals));      // page-locked caller arrays are uploaded in place
    return for_each_device(vk->devs, n, [&](DevCtx* c, size_t b, size_t e) -> int {
        return host_pipeline(c, vk, b, e, k, status_out,
            [&](size_t first, size_t cnt, Sink* dst) -> size_t {
                if (dst) { dst->put(0, proofs + first * 256, cnt * 256, true); dst->put(cnt * 256, signals + first * (size_t)k * 32, cnt * (size_t)k * 32, true); }
                return cnt * (256 + (size_t)k * 32);
            },
            [&](size_t, size_t cnt, uint8_t* d) -> Job {
                Job j;
                j.recs = d; j.stride = 256; j.off = 0; j.mode = SIG_GENERIC; j.sig_a = d + cnt * 256; j.k = k; j.base = c->h_ic0;
                return j;
            }, direct);
    });
}

// ------------------------------------------------------------------------------------------ key sets: N verify_proof_with_key calls (groth16.rs:23-49)
// A set borrows its keys' device tables and owns, per device, a workspace context without key tables plus the grouping arrays.  A call groups
// each device pass by key on the device (kernels.cuh, "key sets"), runs the front kernels over the pass in slot order and the heavy kernels
// chunked like run_verify, then scatters the slot statuses back to caller order.
struct SetDev {
    DevCtx* c = nullptr;
    KeyDesc* d_keys = nullptr;
    uint32_t* perm = nullptr; uint8_t* slot_key = nullptr; uint8_t* slot_status = nullptr; size_t slot_cap = 0;
    uint32_t* tile = nullptr; size_t tile_cap = 0; uint32_t* total = nullptr;
};
struct zkv_vkset {
    std::vector<const zkv_vk*> keys;
    std::vector<SetDev> devs;
    std::vector<DevCtx*> ctxs;            // devs[d].c (for_each_device)
    int ns_max = 1;                       // signals per proof of the widest key: the scalar stride of a slot
};
static SetDev* set_dev(const zkv_vkset* s, int device) {
    for (auto& d : s->devs) if (d.c->device == device) return const_cast<SetDev*>(&d);
    return nullptr;
}
extern "C" void zkv_vkset_destroy(zkv_vkset* s) {
    if (!s) return;
    for (auto& d : s->devs) {
        if (!d.c) continue;
        cudaSetDevice(d.c->device);
        cudaFree(d.d_keys); cudaFree(d.perm); cudaFree(d.slot_key); cudaFree(d.slot_status); cudaFree(d.tile); cudaFree(d.total);
        ctx_free(d.c);
    }
    delete s;
}
static int vkset_build_on(zkv_vkset* s, SetDev& sd) {
    int rc = ctx_init(sd.c); if (rc) return rc;
    std::vector<KeyDesc> h(s->keys.size());
    for (size_t k = 0; k < h.size(); k++) {
        const zkv_vk* vk = s->keys[k];
        const DevCtx* kc = vk_ctx(vk, sd.c->device);
        KeyDesc& q = h[k]; memset(&q, 0, sizeof q);
        q.base = kc->h_ic0; q.tab = kc->d_tab; q.nt[0] = kc->d_nlines; q.nt[1] = kc->d_nlines + ZKV_LINES_PER_G2; q.pre = kc->d_pre;
        q.ns = vk->n_ic - 1; q.vm = vk->vm; q.reject = !vk->valid;
        q.vk_skip = (uint8_t)((kc->h_vk.g2_inf[1] ? 2 : 0) | (kc->h_vk.g2_inf[2] ? 4 : 0));
    }
    CK(cudaMalloc(&sd.d_keys, sizeof(KeyDesc) * h.size())); CK(cudaMalloc(&sd.total, sizeof(uint32_t)));
    CK(cudaMemcpy(sd.d_keys, h.data(), sizeof(KeyDesc) * h.size(), cudaMemcpyHostToDevice));
    return 0;
}
extern "C" int zkv_vkset_create(const zkv_vk* const* keys, int n_keys, const int* devices, int n_dev, zkv_vkset** out) {
    if (!out || !keys) return fail(ZKV_ERR_ARG, "zkv_vkset_create: null argument");
    if (n_keys < 1 || n_keys > ZKV_MAX_KEYS) return fail(ZKV_ERR_ARG, "zkv_vkset_create: n_keys must be 1..256");
    for (int k = 0; k < n_keys; k++) if (!keys[k]) return fail(ZKV_ERR_ARG, "zkv_vkset_create: null key");
    int ndev_sys = zkv_device_count();
    if (ndev_sys <= 0) return fail(ZKV_ERR_CUDA, "zkv_vkset_create: no CUDA device (this library has no CPU path)");
    std::vector<int> devs;
    if (!devices || n_dev <= 0) devs.push_back(0); else devs.assign(devices, devices + n_dev);
    for (int d : devs) if (d < 0 || d >= ndev_sys) return fail(ZKV_ERR_ARG, "zkv_vkset_create: bad device index");
    for (int k = 0; k < n_keys; k++)
        for (int d : devs) {
            const DevCtx* kc = vk_ctx(keys[k], d);
            if (!kc) return fail(ZKV_ERR_ARG, "zkv_vkset_create: key " + std::to_string(k) + " is not loaded on device " + std::to_string(d));
        }
    zkv_vkset* s = new zkv_vkset();
    s->keys.assign(keys, keys + n_keys);
    for (auto* vk : s->keys) s->ns_max = std::max(s->ns_max, vk->n_ic - 1);
    s->devs.resize(devs.size());
    for (size_t j = 0; j < devs.size(); j++) {
        SetDev& sd = s->devs[j];
        sd.c = new DevCtx(); sd.c->device = devs[j]; s->ctxs.push_back(sd.c);
        int rc = vkset_build_on(s, sd);
        if (rc) { zkv_vkset_destroy(s); return rc; }
    }
    *out = s;
    return 0;
}
// Slots of a pass of m records: each key present pads its group by at most 31 slots (a multiple of 32, so chunks keep whole warps)
static size_t slot_bound(size_t m, size_t n_keys) { return (m + 31 * std::min(n_keys, m) + 31) / 32 * 32; }
// Grow the set's grouping arrays to S slots and ntk per-tile counters; like ctx_reserve, it waits for an asynchronous user before freeing.
static int set_reserve(SetDev* sd, size_t S, size_t ntk) {
    if (S > sd->slot_cap || ntk > sd->tile_cap) { int rc = ctx_wait_idle(sd->c); if (rc) return rc; }
    if (S > sd->slot_cap) {
        cudaFree(sd->perm); cudaFree(sd->slot_key); cudaFree(sd->slot_status); sd->slot_cap = 0;
        CK(cudaMalloc(&sd->perm, S * sizeof(uint32_t))); CK(cudaMalloc(&sd->slot_key, S)); CK(cudaMalloc(&sd->slot_status, S)); sd->slot_cap = S;
    }
    if (ntk > sd->tile_cap) { cudaFree(sd->tile); sd->tile_cap = 0; CK(cudaMalloc(&sd->tile, ntk * sizeof(uint32_t))); sd->tile_cap = ntk; }
    return 0;
}
// One device pass of m records already in device memory (key_idx, 256-byte proofs, signal words with offsets relative to sig_base), enqueued
// on stream st; statuses in caller order to d_status.  Caller holds c->mu and has set the device.  Launches: 3 grouping kernels, decode,
// signals, vk_x, G2 check, Miller loop, final exponentiation, status scatter = 10 for a pass of one chain; from chunk_count's threshold on,
// + 1 (flag merge of the forked front) and 4 chunks x (4 Miller segments + 4 final-exponentiation stages) instead of 2: 41.
static int keyset_pass(const zkv_vkset* s, SetDev* sd, size_t m, const uint32_t* d_key_idx, const uint8_t* d_proofs, const uint8_t* d_sig,
                       const uint64_t* d_sig_off, uint64_t sig_base, uint8_t* d_status, cudaStream_t st) {
    DevCtx* c = sd->c;
    const int nk = (int)s->keys.size(), ns = s->ns_max;
    const size_t S = slot_bound(m, (size_t)nk), ntiles = (m + ZKV_GROUP_TILE - 1) / ZKV_GROUP_TILE;
    int rc = ctx_acquire(c, st); if (rc) return rc;
    rc = ctx_reserve(c, S, (size_t)ns * 8); if (rc) return rc;
    rc = set_reserve(sd, S, ntiles * nk); if (rc) return rc;
    CK(cudaMemsetAsync(sd->perm, 0xff, S * sizeof(uint32_t), st)); CK(cudaMemsetAsync(sd->slot_key, 0, S, st));
    launch(k_group_count, (int)ntiles, 256, 0, st, (int)m, nk, d_key_idx, sd->tile);
    launch(k_group_scan, 1, ZKV_MAX_KEYS, 0, st, (int)ntiles, nk, sd->tile, sd->slot_key, sd->total);
    launch(k_group_scatter, (int)ntiles, 256, 0, st, (int)m, nk, d_key_idx, sd->tile, sd->perm, sd->slot_key);
    const int n = (int)S;
    uint8_t* flags = c->flags;
    launch(k_decode_keys, nblk(n), TPB, 0, st, n, sd->perm, sd->slot_key, sd->d_keys, nk, d_key_idx, d_proofs, c->px[0], c->py[0], c->qx, c->qy, c->px[3], c->py[3], flags);
    launch(k_signals_keys, nblk(n), TPB, 0, st, n, sd->perm, sd->slot_key, sd->d_keys, d_sig, d_sig_off, sig_base, ns, c->scal, flags);
    const int chunks = chunk_count(c, S, 0);
    rc = enqueue_vkx_g2(c, 0, n, flags, st, chunks > 1, false, [&](uint8_t* fl) {   // forked when chunked: the front phase of run_verify's schedule
        launch(k_vkx_keys, nblk(n), TPB, 0, st, n, sd->perm, sd->slot_key, sd->d_keys, c->scal, ns, c->px[2], c->py[2], fl);
    });
    if (rc) return rc;
    auto heavy = [&](size_t o, int mm, cudaStream_t hs, int segs, bool staged) -> int {
        const MillerArgs a = verify_miller_args(c, o);
        for (int k = 0; k < segs; k++) {
            auto [hi, lo] = miller_segment(k, segs);
            launch(k_miller_lz_keys, nblk(mm, LZ_NT), LZ_NT, LZ_SMEM_MILLER, hs, sd->total, o, mm, a, sd->slot_key + o, sd->d_keys, flags + o, c->tx + o, c->ty + o, c->f + o, c->rst + o, c->sl + 4 * o, hi, lo, k == 0, k == segs - 1);
        }
        if (staged) for (int q = 0; q < 4; q++) launch(k_final_exp_lz_keys, nblk(mm, LZ_NT), LZ_NT, LZ_SMEM_BYTES, hs, sd->total, o, mm, q, q, c->f + o, c->fes + 6 * o, flags + o, sd->slot_status + o);
        else launch(k_final_exp_lz_keys, nblk(mm, LZ_NT), LZ_NT, LZ_SMEM_BYTES, hs, sd->total, o, mm, 0, 3, c->f + o, c->fes + 6 * o, flags + o, sd->slot_status + o);
        return 0;
    };
    if (chunks <= 1) rc = heavy(0, n, st, 1, false);
    else rc = fork_join(c, st, S, chunks, [&](size_t o, int mm, cudaStream_t hs) { return heavy(o, mm, hs, 4, true); });
    if (rc) return rc;
    launch(k_status_to_caller, nblk(n), TPB, 0, st, n, sd->total, sd->perm, sd->slot_status, d_status);
    CK(cudaGetLastError());
    return 0;
}
extern "C" int zkv_groth16_verify_batch_keys(const zkv_vkset* s, const uint32_t* key_idx, const uint8_t* proofs, const uint8_t* signals,
                                             const uint64_t* sig_off, size_t n, uint8_t* status_out) {
    if (!s || (n && (!key_idx || !proofs || !sig_off || !status_out))) return fail(ZKV_ERR_ARG, "zkv_groth16_verify_batch_keys: null argument");
    if (n == 0) return 0;
    if (n > 0xffffffffull) return fail(ZKV_ERR_ARG, "batch too large");
    for (size_t i = 0; i < n; i++) if (key_idx[i] >= s->keys.size()) return fail(ZKV_ERR_ARG, "zkv_groth16_verify_batch_keys: key index " + std::to_string(key_idx[i]) + " out of range");
    if (!offsets_ok(sig_off, n)) return fail(ZKV_ERR_ARG, "zkv_groth16_verify_batch_keys: signal offsets must be non-decreasing");
    const bool any_sig = sig_off[n] != sig_off[0];
    if (any_sig && !signals) return fail(ZKV_ERR_ARG, "zkv_groth16_verify_batch_keys: null signals");
    const bool direct = n >= 4096 && is_pinned(key_idx) && is_pinned(proofs) && is_pinned(sig_off) && (!any_sig || is_pinned(signals));   // page-locked caller arrays are uploaded in place
    return for_each_device(s->ctxs, n, [&](DevCtx* c, size_t b, size_t e) -> int {
        SetDev* sd = set_dev(s, c->device);
        if (int rc = ctx_wait_idle(c)) return rc;      // a host call blocks anyway: wait out an earlier asynchronous device call here
        // A pass is grouped as a whole, so it is uploaded as a whole before its kernels run: [key_idx][signal offsets][proofs][signal words]
        for (size_t s0 = b; s0 < e; s0 += MAX_CHUNK) {
            const size_t m = std::min(MAX_CHUNK, e - s0), words = (size_t)(sig_off[s0 + m] - sig_off[s0]);
            const size_t o_off = (m * 4 + 255) / 256 * 256, o_pr = o_off + ((m + 1) * 8 + 255) / 256 * 256, o_sig = o_pr + m * 256, bytes = o_sig + words * 32;
            int rc = ctx_stage(c, bytes, m); if (rc) return rc;
            Sink sk{direct ? nullptr : c->h_pin, c->d_in, c->stream, 0};
            sk.put(0, key_idx + s0, m * 4, true); sk.put(o_off, sig_off + s0, (m + 1) * 8, true); sk.put(o_pr, proofs + s0 * 256, m * 256, true);
            if (words) sk.put(o_sig, signals + sig_off[s0] * 32, words * 32, true);
            if (sk.bad) return fail(ZKV_ERR_CUDA, "cudaMemcpyAsync (page-locked caller memory to device)");
            if (!direct) CK(cudaMemcpyAsync(c->d_in, c->h_pin, bytes, cudaMemcpyHostToDevice, c->stream));
            rc = keyset_pass(s, sd, m, (const uint32_t*)c->d_in, c->d_in + o_pr, c->d_in + o_sig, (const uint64_t*)(c->d_in + o_off), sig_off[s0], c->d_out, c->stream);
            if (rc) return rc;
            CK(cudaMemcpyAsync(c->h_out, c->d_out, m, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            memcpy(status_out + s0, c->h_out, m);
        }
        return 0;
    });
}
extern "C" int zkv_groth16_verify_batch_keys_device(const zkv_vkset* s, int device, const void* d_key_idx, const void* d_proofs, const void* d_signals,
                                                    const void* d_sig_off, size_t n, void* d_status_out, void* stream) {
    if (!s || !d_key_idx || !d_proofs || !d_signals || !d_sig_off || !d_status_out) return fail(ZKV_ERR_ARG, "zkv_groth16_verify_batch_keys_device: null argument");
    SetDev* sd = set_dev(s, device);
    if (!sd) return fail(ZKV_ERR_ARG, "device not in the set's device list");
    if (n > MAX_CHUNK * 8) return fail(ZKV_ERR_ARG, "device batch too large");
    if (n == 0) return 0;
    return device_call(sd->c, device, stream, [&](cudaStream_t st) {
        return keyset_pass(s, sd, n, (const uint32_t*)d_key_idx, (const uint8_t*)d_proofs, (const uint8_t*)d_signals, (const uint64_t*)d_sig_off, 0, (uint8_t*)d_status_out, st);
    });
}

// ------------------------------------------------------------------------------------------ RISC Zero
struct zkv_risc0 {
    const zkv_vk* vk = nullptr; zkv_vk* owned = nullptr;
    int initialized = 0;
    uint8_t control_root_0[16], control_root_1[16], bn254_control_id[32], selector[4], vk_digest[32];
    Risc0HashConsts hc; g1aff base; int all_fail = 0;
};
// risc0/crypto.rs:136-195 compute_verifier_key_digest (over this handle's key)
static void risc0_vk_digest(uint8_t out[32], const zkv_vk* vk) {
    uint8_t ic_tag[32], vk_tag[32], cur[32], buf[32 * 7 + 2];
    sha_str(ic_tag, "risc0_groth16.VerifyingKey.IC"); sha_str(vk_tag, "risc0_groth16.VerifyingKey");
    memset(cur, 0, 32);
    for (int i = vk->n_ic - 1; i >= 0; i--) {        // tagged_list -> tagged_list_cons, :124-134
        memcpy(buf, ic_tag, 32); sha_bytes(buf + 32, vk->ic.data() + 64 * i, 64); memcpy(buf + 64, cur, 32); buf[96] = 0x02; buf[97] = 0x00;
        sha_bytes(cur, buf, 98);
    }
    memcpy(buf, vk_tag, 32); sha_bytes(buf + 32, vk->alpha, 64); sha_bytes(buf + 64, vk->beta, 128); sha_bytes(buf + 96, vk->gamma, 128); sha_bytes(buf + 128, vk->delta, 128);
    memcpy(buf + 160, cur, 32); buf[192] = 0x05; buf[193] = 0x00;    // tagged_struct: 5 down-digests, :112-122
    sha_bytes(out, buf, 194);
}
extern "C" int zkv_risc0_create(const zkv_vk* vk_or_null, const int* devices, int n_dev, zkv_risc0** out) {
    if (!out) return fail(ZKV_ERR_ARG, "zkv_risc0_create: null out");
    zkv_risc0* h = new zkv_risc0();
    if (vk_or_null) { if (vk_or_null->n_ic != 6 || vk_or_null->vm != ZKV_VM_RISC0) { delete h; return fail(ZKV_ERR_ARG, "zkv_risc0_create: need a ZKV_VM_RISC0 key with 6 IC points"); } h->vk = vk_or_null; }
    else { int rc = zkv_vk_load_risc0(devices, n_dev, &h->owned); if (rc) { delete h; return rc; } h->vk = h->owned; }
    *out = h; return 0;
}
extern "C" void zkv_risc0_destroy(zkv_risc0* h) { if (!h) return; if (h->owned) zkv_vk_free(h->owned); delete h; }

extern "C" int zkv_risc0_initialize(zkv_risc0* h, const uint8_t control_root[32], const uint8_t bn254_control_id[32]) {
    if (!h || !control_root || !bn254_control_id) return fail(ZKV_ERR_ARG, "zkv_risc0_initialize: null argument");
    if (h->initialized) return fail(ZKV_ERR_STATE, "AlreadyInitialized");                     // risc0/verifier.rs:59-61
    // split_digest(control_root), risc0/crypto.rs:103-110: reverse the 32 bytes, low = rev[16..], high = rev[..16]
    uint8_t rev[32]; for (int i = 0; i < 32; i++) rev[i] = control_root[31 - i];
    memcpy(h->control_root_0, rev + 16, 16); memcpy(h->control_root_1, rev, 16);
    memcpy(h->bn254_control_id, bn254_control_id, 32);
    // calculate_selector, risc0/verifier.rs:128-144
    uint8_t buf[130], d[32];
    sha_str(buf, "risc0.Groth16ReceiptVerifierParameters"); memcpy(buf + 32, control_root, 32);
    for (int i = 0; i < 32; i++) buf[64 + i] = bn254_control_id[31 - i];
    risc0_vk_digest(h->vk_digest, h->vk); memcpy(buf + 96, h->vk_digest, 32); buf[128] = 0x03; buf[129] = 0x00;
    sha_bytes(d, buf, 130); memcpy(h->selector, d, 4);
    // per-proof hashing constants (risc0/types.rs:62-95, config.rs:5-32)
    uint8_t tag[32]; sha_str(tag, "risc0.Output"); bytes_to_words(h->hc.tag_out, tag);
    sha_str(tag, "risc0.ReceiptClaim");
    { uint32_t st[8], w[16]; sha256_init(st); bytes_to_words(w, tag); for (int k = 8; k < 16; k++) w[k] = 0; sha256_compress(st, w); memcpy(h->hc.claim_mid, st, 32); }
    bytes_to_words(h->hc.sys0, ZKV_RISC0_SYSTEM_STATE_ZERO_DIGEST);
    // signals 0,1,4 are instance constants (verifier.rs:172-179): fold them into the vk_x base point K = IC0 + s0 IC1 + s1 IC2 + s4 IC5
    h->all_fail = memcmp(bn254_control_id, FR_R_BE, 32) >= 0;                                  // groth16.rs:32-34: signal >= R
    DevCtx* c = h->vk->devs[0];
    {
        std::lock_guard<std::mutex> lk(c->mu);
        CK(cudaSetDevice(c->device));
        int rc = ctx_wait_idle(c); if (rc) return rc;
        rc = ctx_reserve(c, 1, 24); if (rc) return rc;
        uint32_t sc[24]; memset(sc, 0, sizeof sc);
        uint8_t w32[32];
        memset(w32, 0, 32); memcpy(w32 + 16, h->control_root_0, 16); for (int k = 0; k < 8; k++) sc[k] = load_be32(w32 + 4 * (7 - k));
        memset(w32, 0, 32); memcpy(w32 + 16, h->control_root_1, 16); for (int k = 0; k < 8; k++) sc[8 + k] = load_be32(w32 + 4 * (7 - k));
        for (int k = 0; k < 8; k++) sc[16 + k] = load_be32(bn254_control_id + 4 * (7 - k));
        CK(cudaMemcpyAsync(c->scal, sc, sizeof sc, cudaMemcpyHostToDevice, c->stream));
        CK(cudaMemsetAsync(c->flags, 0, 1, c->stream));
        if (!h->all_fail && h->vk->valid) {
            k_vkx<<<1, 1, 0, c->stream>>>(1, c->scal, 2, ZKV_WIN_PER_SCALAR, c->d_tab, c->h_ic0, c->px[2], c->py[2], c->flags);
            g1aff mid;
            CK(cudaMemcpyAsync(&mid.x, c->px[2], sizeof(fp), cudaMemcpyDeviceToHost, c->stream)); CK(cudaMemcpyAsync(&mid.y, c->py[2], sizeof(fp), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            k_vkx<<<1, 1, 0, c->stream>>>(1, c->scal + 16, 1, ZKV_WIN_PER_SCALAR, c->d_tab + (size_t)4 * ZKV_WIN_PER_SCALAR * ZKV_WIN_ENTRIES, mid, c->px[2], c->py[2], c->flags);
            CK(cudaMemcpyAsync(&h->base.x, c->px[2], sizeof(fp), cudaMemcpyDeviceToHost, c->stream)); CK(cudaMemcpyAsync(&h->base.y, c->py[2], sizeof(fp), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            CK(cudaGetLastError());
        } else memset(&h->base, 0, sizeof h->base);
    }
    h->initialized = 1;
    return 0;
}
extern "C" int zkv_risc0_is_initialized(const zkv_risc0* h) { return h ? h->initialized : 0; }
extern "C" int zkv_risc0_get_selector(const zkv_risc0* h, uint8_t out[4]) { if (!h || !out) return fail(ZKV_ERR_ARG, "null"); if (h->initialized) memcpy(out, h->selector, 4); else memset(out, 0, 4); return 0; }
extern "C" int zkv_risc0_get_control_root(const zkv_risc0* h, uint8_t out0[16], uint8_t out1[16]) {
    if (!h || !out0 || !out1) return fail(ZKV_ERR_ARG, "null");
    if (h->initialized) { memcpy(out0, h->control_root_0, 16); memcpy(out1, h->control_root_1, 16); } else { memset(out0, 0, 16); memset(out1, 0, 16); }
    return 0;
}
extern "C" int zkv_risc0_get_bn254_control_id(const zkv_risc0* h, uint8_t out[32]) { if (!h || !out) return fail(ZKV_ERR_ARG, "null"); if (h->initialized) memcpy(out, h->bn254_control_id, 32); else memset(out, 0, 32); return 0; }
extern "C" int zkv_risc0_get_verifier_key_digest(const zkv_risc0* h, uint8_t out[32]) { if (!h || !out) return fail(ZKV_ERR_ARG, "null"); risc0_vk_digest(out, h->vk); return 0; }

static uint32_t sel_le(const uint8_t s[4]) { return (uint32_t)s[0] | (uint32_t)s[1] << 8 | (uint32_t)s[2] << 16 | (uint32_t)s[3] << 24; }
// Host-buffer batches upload the caller's arrays AS THEY ARE (four bulk copies per chunk into pinned staging: offsets, the two 32-byte
// arrays, the seal bytes) and leave the front checks of verify_integrity_internal (risc0/verifier.rs:151-170) to k_decode; round 1
// filtered and repacked proof by proof on the host, which cost 7 % of the end-to-end rate.
static int risc0_batch(const zkv_risc0* h, const uint8_t* seals, const uint64_t* seal_off, const uint8_t* a32, const uint8_t* b32, int integrity, size_t n, uint8_t* status_out) {
    if (!h || (n && (!seals || !seal_off || !a32 || (!integrity && !b32) || !status_out))) return fail(ZKV_ERR_ARG, "zkv_risc0_verify_batch: null argument");
    if (n == 0) return 0;
    if (n > 0xffffffffull) return fail(ZKV_ERR_ARG, "batch too large");
    if (!offsets_ok(seal_off, n)) return fail(ZKV_ERR_ARG, "seal offsets must be non-decreasing");
    if (!h->initialized) { memset(status_out, ZKV_INVALID_INITIALIZATION, n); return 0; }     // risc0/verifier.rs:84-86, 99-101
    const zkv_vk* vk = h->vk;
    const bool direct = n >= 4096 && is_pinned(seals) && is_pinned(seal_off) && is_pinned(a32) && (integrity || is_pinned(b32));      // page-locked caller arrays are uploaded in place
    const size_t per = integrity ? 32 : 64;
    return for_each_device(vk->devs, n, [&](DevCtx* c, size_t b, size_t e) -> int {
        // piece block layout: [offsets (cnt + 1) x 8][a32 cnt x 32][b32 cnt x 32][seal bytes][slack: k_decode never reads past a record's own length]
        return host_pipeline(c, vk, b, e, 2, status_out,
            [&](size_t i0, size_t cnt, Sink* dst) -> size_t {
                const size_t bytes = (size_t)(seal_off[i0 + cnt] - seal_off[i0]);
                if (!dst) return (cnt + 1) * 8 + cnt * per + bytes + 320;
                size_t p = 0;
                dst->put(p, seal_off + i0, (cnt + 1) * 8); p += (cnt + 1) * 8;
                dst->put(p, a32 + i0 * 32, cnt * 32); p += cnt * 32;
                if (!integrity) { dst->put(p, b32 + i0 * 32, cnt * 32); p += cnt * 32; }
                dst->put(p, seals + seal_off[i0], bytes, true); p += bytes;
                return p + 320;
            },
            [&](size_t i0, size_t cnt, uint8_t* d) -> Job {
                Job j;
                j.rec_off = (const uint64_t*)d; j.rec_base = seal_off[i0]; j.off = 4; j.stride = 260; j.check_selector = 1; j.selector_le = sel_le(h->selector);
                j.mode = integrity ? SIG_RISC0_INTEGRITY : SIG_RISC0_VERIFY;
                j.sig_a = d + (cnt + 1) * 8; j.sig_b = j.sig_a + cnt * 32; j.recs = j.sig_a + cnt * per;
                j.hc = h->hc; j.base = h->base; j.all_fail = h->all_fail;
                return j;
            }, direct);
    });
}
extern "C" int zkv_risc0_verify_batch(const zkv_risc0* h, const uint8_t* seals, const uint64_t* seal_off, const uint8_t* image_ids, const uint8_t* journal_digests, size_t n, uint8_t* status_out) {
    return risc0_batch(h, seals, seal_off, image_ids, journal_digests, 0, n, status_out);
}
extern "C" int zkv_risc0_verify_integrity_batch(const zkv_risc0* h, const uint8_t* seals, const uint64_t* seal_off, const uint8_t* claim_digests, size_t n, uint8_t* status_out) {
    return risc0_batch(h, seals, seal_off, claim_digests, nullptr, 1, n, status_out);
}
extern "C" int zkv_risc0_verify(const zkv_risc0* h, const uint8_t* seal, size_t seal_len, const uint8_t image_id[32], const uint8_t journal_digest[32], uint8_t* status_out) {
    uint64_t off[2] = {0, seal_len}; uint8_t dummy = 0;
    return risc0_batch(h, seal ? seal : &dummy, off, image_id, journal_digest, 0, 1, status_out);
}
extern "C" int zkv_risc0_verify_integrity(const zkv_risc0* h, const uint8_t* seal, size_t seal_len, const uint8_t claim_digest[32], uint8_t* status_out) {
    uint64_t off[2] = {0, seal_len}; uint8_t dummy = 0;
    return risc0_batch(h, seal ? seal : &dummy, off, claim_digest, nullptr, 1, 1, status_out);
}
extern "C" int zkv_risc0_verify_batch_device(const zkv_risc0* h, int device, const void* d_seals260, const void* d_image_ids, const void* d_journal_digests, size_t n, void* d_status_out, void* stream) {
    if (!h || !d_seals260 || !d_image_ids || !d_journal_digests || !d_status_out) return fail(ZKV_ERR_ARG, "zkv_risc0_verify_batch_device: null argument");
    DevCtx* c = vk_ctx(h->vk, device);
    if (!c) return fail(ZKV_ERR_ARG, "device not in the handle's device list");
    if (n > MAX_CHUNK * 8) return fail(ZKV_ERR_ARG, "device batch too large");
    if (!h->initialized) {      // no kernel, no use of the workspace
        CK(cudaSetDevice(device));
        CK(cudaMemsetAsync(d_status_out, ZKV_INVALID_INITIALIZATION, n, (cudaStream_t)stream));
        return 0;
    }
    Job j;
    j.vk = h->vk; j.n = n; j.recs = (const uint8_t*)d_seals260; j.stride = 260; j.off = 4; j.check_selector = 1; j.selector_le = sel_le(h->selector);
    j.mode = SIG_RISC0_VERIFY; j.sig_a = (const uint8_t*)d_image_ids; j.sig_b = (const uint8_t*)d_journal_digests; j.hc = h->hc; j.base = h->base; j.all_fail = h->all_fail;
    j.d_status = (uint8_t*)d_status_out;
    return device_call(c, device, stream, [&](cudaStream_t s) { return run_verify(c, j, s); });
}

// ------------------------------------------------------------------------------------------ SP1
struct zkv_sp1 { const zkv_vk* vk = nullptr; zkv_vk* owned = nullptr; uint8_t verifier_hash[32]; };
extern "C" int zkv_sp1_create(const zkv_vk* vk_or_null, const int* devices, int n_dev, zkv_sp1** out) {
    if (!out) return fail(ZKV_ERR_ARG, "zkv_sp1_create: null out");
    zkv_sp1* h = new zkv_sp1();
    memcpy(h->verifier_hash, ZKV_SP1_VERIFIER_HASH, 32);
    if (vk_or_null) { if (vk_or_null->n_ic != 3 || vk_or_null->vm != ZKV_VM_SP1) { delete h; return fail(ZKV_ERR_ARG, "zkv_sp1_create: need a ZKV_VM_SP1 key with 3 IC points"); } h->vk = vk_or_null; }
    else { int rc = zkv_vk_load_sp1(devices, n_dev, &h->owned); if (rc) { delete h; return rc; } h->vk = h->owned; }
    *out = h; return 0;
}
extern "C" void zkv_sp1_destroy(zkv_sp1* h) { if (!h) return; if (h->owned) zkv_vk_free(h->owned); delete h; }
extern "C" int zkv_sp1_verifier_hash(const zkv_sp1* h, uint8_t out[32]) { if (!h || !out) return fail(ZKV_ERR_ARG, "null"); memcpy(out, h->verifier_hash, 32); return 0; }
extern "C" const char* zkv_sp1_version(const zkv_sp1*) { return ZKV_SP1_VERSION; }

extern "C" int zkv_sp1_verify_batch(const zkv_sp1* h, const uint8_t* vkeys, const uint8_t* public_values, const uint64_t* pv_off, const uint8_t* proofs, const uint64_t* proof_off, size_t n, uint8_t* status_out) {
    if (!h || (n && (!vkeys || !public_values || !pv_off || !proofs || !proof_off || !status_out))) return fail(ZKV_ERR_ARG, "zkv_sp1_verify_batch: null argument");
    if (n == 0) return 0;
    if (n > 0xffffffffull) return fail(ZKV_ERR_ARG, "batch too large");
    if (!offsets_ok(proof_off, n) || !offsets_ok(pv_off, n)) return fail(ZKV_ERR_ARG, "proof / public-value offsets must be non-decreasing");
    const zkv_vk* vk = h->vk;
    const bool direct = n >= 4096 && is_pinned(proofs) && is_pinned(proof_off) && is_pinned(pv_off) && is_pinned(vkeys) && is_pinned(public_values);      // page-locked caller arrays are uploaded in place
    return for_each_device(vk->devs, n, [&](DevCtx* c, size_t b, size_t e) -> int {
        // piece block layout: [proof offsets (cnt + 1) x 8][public-value offsets (cnt + 1) x 8][vkeys cnt x 32][proof bytes][public values][slack]
        return host_pipeline(c, vk, b, e, 2, status_out,
            [&](size_t i0, size_t cnt, Sink* dst) -> size_t {
                const size_t pr = (size_t)(proof_off[i0 + cnt] - proof_off[i0]), pv = (size_t)(pv_off[i0 + cnt] - pv_off[i0]);
                if (!dst) return (cnt + 1) * 16 + cnt * 32 + pr + pv + 320;
                size_t p = 0;
                dst->put(p, proof_off + i0, (cnt + 1) * 8); p += (cnt + 1) * 8;
                dst->put(p, pv_off + i0, (cnt + 1) * 8); p += (cnt + 1) * 8;
                dst->put(p, vkeys + i0 * 32, cnt * 32); p += cnt * 32;
                dst->put(p, proofs + proof_off[i0], pr, true); p += pr;
                dst->put(p, public_values + pv_off[i0], pv, true); p += pv;
                return p + 320;
            },
            [&](size_t i0, size_t cnt, uint8_t* d) -> Job {
                Job j;
                j.rec_off = (const uint64_t*)d; j.rec_base = proof_off[i0]; j.off = 4; j.stride = 260; j.check_selector = 1; j.selector_le = sel_le(h->verifier_hash);
                j.mode = SIG_SP1; j.pv_off = (const uint64_t*)(d + (cnt + 1) * 8); j.pv_base = pv_off[i0];
                j.sig_a = d + (cnt + 1) * 16; j.recs = j.sig_a + cnt * 32; j.sig_b = j.recs + (size_t)(proof_off[i0 + cnt] - proof_off[i0]);
                j.base = c->h_ic0;
                return j;
            }, direct);
    });
}
extern "C" int zkv_sp1_verify_proof(const zkv_sp1* h, const uint8_t vkey[32], const uint8_t* public_values, size_t pv_len, const uint8_t* proof, size_t proof_len, uint8_t* status_out) {
    uint64_t po[2] = {0, proof_len}, vo[2] = {0, pv_len}; uint8_t dummy = 0;
    return zkv_sp1_verify_batch(h, vkey, public_values ? public_values : &dummy, vo, proof ? proof : &dummy, po, 1, status_out);
}
extern "C" int zkv_sp1_verify_batch_device(const zkv_sp1* h, int device, const void* d_vkeys, const void* d_public_values, size_t pv_stride, const void* d_proofs260, size_t n, void* d_status_out, void* stream) {
    if (!h || !d_vkeys || !d_public_values || !d_proofs260 || !d_status_out) return fail(ZKV_ERR_ARG, "zkv_sp1_verify_batch_device: null argument");
    DevCtx* c = vk_ctx(h->vk, device);
    if (!c) return fail(ZKV_ERR_ARG, "device not in the handle's device list");
    if (n > MAX_CHUNK * 8) return fail(ZKV_ERR_ARG, "device batch too large");
    Job j;
    j.vk = h->vk; j.n = n; j.recs = (const uint8_t*)d_proofs260; j.stride = 260; j.off = 4; j.check_selector = 1; j.selector_le = sel_le(h->verifier_hash);
    j.mode = SIG_SP1; j.sig_a = (const uint8_t*)d_vkeys; j.sig_b = (const uint8_t*)d_public_values; j.pv_off = nullptr; j.pv_stride = pv_stride; j.base = c->h_ic0;
    j.d_status = (uint8_t*)d_status_out;
    return device_call(c, device, stream, [&](cudaStream_t s) { return run_verify(c, j, s); });
}


extern "C" void zkv_test_parallel_copy(void* dst, const void* src, size_t n) { pcopy(dst, src, n); }
extern "C" void* zkv_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (zkv_device_count() <= 0 || cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); fail(ZKV_ERR_CUDA, "zkv_host_alloc: cudaHostAlloc failed"); return nullptr; }
    return p;
}
extern "C" void zkv_host_free(void* p) { if (p) cudaFreeHost(p); }

// ------------------------------------------------------------------------------------------ known-answer self test (include/zkv.h)
extern "C" int zkv_self_test(int device) {
    if (zkv_device_count() <= device || device < 0) return fail(ZKV_ERR_CUDA, "no such CUDA device (this library has no CPU path)");
    zkv_risc0* r0 = nullptr; zkv_sp1* s1 = nullptr;
    int rc = zkv_risc0_create(nullptr, &device, 1, &r0);
    if (!rc) rc = zkv_risc0_initialize(r0, ZKV_RISC0_FIXTURE_CONTROL_ROOT, ZKV_RISC0_FIXTURE_BN254_CONTROL_ID);
    if (!rc) rc = zkv_sp1_create(nullptr, &device, 1, &s1);
    if (!rc) {
        uint8_t st[4] = {255, 255, 255, 255};
        uint8_t seal[sizeof ZKV_RISC0_FIXTURE_SEAL], proof[sizeof ZKV_SP1_FIXTURE_PROOF];
        memcpy(seal, ZKV_RISC0_FIXTURE_SEAL, sizeof seal); memcpy(proof, ZKV_SP1_FIXTURE_PROOF, sizeof proof);
        rc = zkv_risc0_verify(r0, seal, sizeof seal, ZKV_RISC0_FIXTURE_IMAGE_ID, ZKV_RISC0_FIXTURE_JOURNAL_DIGEST, &st[0]);
        seal[4 + 100] ^= 0x04;                               // one bit of B: still a field element, no longer a valid proof
        if (!rc) rc = zkv_risc0_verify(r0, seal, sizeof seal, ZKV_RISC0_FIXTURE_IMAGE_ID, ZKV_RISC0_FIXTURE_JOURNAL_DIGEST, &st[1]);
        if (!rc) rc = zkv_sp1_verify_proof(s1, ZKV_SP1_FIXTURE_VKEY, ZKV_SP1_FIXTURE_PUBLIC_VALUES, sizeof ZKV_SP1_FIXTURE_PUBLIC_VALUES, proof, sizeof proof, &st[2]);
        uint8_t vkey[32]; memcpy(vkey, ZKV_SP1_FIXTURE_VKEY, 32); vkey[31] ^= 1;      // another program key: a different public input
        if (!rc) rc = zkv_sp1_verify_proof(s1, vkey, ZKV_SP1_FIXTURE_PUBLIC_VALUES, sizeof ZKV_SP1_FIXTURE_PUBLIC_VALUES, proof, sizeof proof, &st[3]);
        if (!rc && !(st[0] == ZKV_OK && st[2] == ZKV_OK && st[1] != ZKV_OK && st[1] != 255 && st[3] == ZKV_VERIFICATION_FAILED)) {
            char msg[160]; snprintf(msg, sizeof msg, "zkv_self_test: kernels returned statuses %d %d %d %d for the reference's golden proofs and their tampers; expected 0, reject, 0, 1", st[0], st[1], st[2], st[3]);
            rc = fail(ZKV_ERR_STATE, msg);
        }
    }
    if (r0) zkv_risc0_destroy(r0);
    if (s1) zkv_sp1_destroy(s1);
    return rc;
}
// ------------------------------------------------------------------------------------------ pairing service (0x08 seam)
static int pairing4_chain(DevCtx* c, size_t o, int n, const uint8_t* d_g1s, const uint8_t* d_g2s, uint8_t* d_ok, uint8_t* d_gt, uint8_t* d_miller, cudaStream_t s, bool timed) {
    uint8_t* flags = c->flags + o;
    if (timed) CK(cudaEventRecord(c->ev[0], s));
    k_g1_decode4<<<nblk(n), TPB, 0, s>>>(n, d_g1s + o * 256, d_g2s + o * 128, c->px[0] + o, c->py[0] + o, c->px[1] + o, c->py[1] + o, c->px[2] + o, c->py[2] + o, c->px[3] + o, c->py[3] + o, c->qx + o, c->qy + o, flags);
    if (timed) { CK(cudaEventRecord(c->ev[1], s)); CK(cudaEventRecord(c->ev[2], s)); }
    k_g2_check<<<nblk(n), TPB, 0, s>>>(n, c->qx + o, c->qy + o, flags);
    if (timed) CK(cudaEventRecord(c->ev[3], s));
    // shared-memory-resident general Miller loop: one variable pair + the three tabled key points, unscaled lines (the oracle's Miller value)
    const uint8_t vk_skip = (uint8_t)((c->h_vk.g2_inf[0] ? 2 : 0) | (c->h_vk.g2_inf[1] ? 4 : 0) | (c->h_vk.g2_inf[2] ? 8 : 0));
    k_pairing4_skip<<<nblk(n), TPB, 0, s>>>(n, c->stride, flags, vk_skip, c->pskip + o);
    LzGenIn gi; memset(&gi, 0, sizeof gi);
    gi.px = c->px[0] + o; gi.py = c->py[0] + o; gi.qx = c->qx + o; gi.qy = c->qy + o; gi.rst = c->rst + o; gi.pskip = c->pskip + o; gi.stride = c->stride; gi.nvar = 1; gi.nfix = 3;
    for (int j = 0; j < 3; j++) gi.tabs[j] = c->d_lines + (size_t)j * ZKV_LINES_PER_G2;
    k_pairing_lz<<<nblk(n, LZ_NT), LZ_NT, LZ_SMEM_BYTES, s>>>(n, gi, c->f + o, ZKV_ATE_NAF_LEN - 2, 0, 1, 1);
    if (timed) CK(cudaEventRecord(c->ev[4], s));
    if (d_miller) k_f12_to_bytes<<<nblk(n), TPB, 0, s>>>(n, c->f + o, d_miller + o * 384);
    k_final_exp_lz<<<nblk(n, LZ_NT), LZ_NT, LZ_SMEM_BYTES, s>>>(n, 0, 3, c->f + o, c->fes + 6 * o, flags, d_ok + o, d_gt ? d_gt + o * 384 : nullptr, 1);
    if (timed) CK(cudaEventRecord(c->ev[5], s));
    CK(cudaGetLastError());
    return 0;
}
static int run_pairing4(DevCtx* c, const zkv_vk* vk, size_t n_, const uint8_t* d_g1s, const uint8_t* d_g2s, uint8_t* d_ok, uint8_t* d_gt, uint8_t* d_miller, cudaStream_t s) {
    if (n_ == 0) return 0;
    int rc = ctx_acquire(c, s); if (rc) return rc;
    rc = ctx_reserve(c, n_, 8); if (rc) return rc;
    if (!vk->valid) {   // a fixed G2 point is invalid: every call reverts
        CK(cudaMemsetAsync(d_ok, 2, n_, s)); if (d_gt) CK(cudaMemsetAsync(d_gt, 0, n_ * 384, s)); if (d_miller) CK(cudaMemsetAsync(d_miller, 0, n_ * 384, s));
        for (int e = 0; e < 6; e++) CK(cudaEventRecord(c->ev[e], s));
        return 0;
    }
    int chunks = chunk_count(c, n_, vk->tune.overlap_chunks.load());
    // the pairing service's chunks carry their own decode / G2-check kernels: from two waves on one serial chain is the faster schedule here
    // (2^22 instances: 1.70 M against 1.63 M instances/s with four chunks)
    if (vk->tune.overlap_chunks.load() == 0 && n_ >= 2 * wave_proofs_of(c)) chunks = 1;
    if (chunks <= 1) return pairing4_chain(c, 0, (int)n_, d_g1s, d_g2s, d_ok, d_gt, d_miller, s, true);
    return fork_join(c, s, n_, chunks, [&](size_t o, int m, cudaStream_t st) { return pairing4_chain(c, o, m, d_g1s, d_g2s, d_ok, d_gt, d_miller, st, false); });
}
extern "C" int zkv_pairing4_batch(const zkv_vk* vk, const uint8_t* g1s, const uint8_t* g2s, size_t n, uint8_t* ok_out, uint8_t* gt_out, uint8_t* miller_out) {
    if (!vk || (n && (!g1s || !g2s || !ok_out))) return fail(ZKV_ERR_ARG, "zkv_pairing4_batch: null argument");
    if (n == 0) return 0;
    const size_t CH = (size_t)1 << 18;
    return for_each_device(vk->devs, n, [&](DevCtx* c, size_t b, size_t e) -> int {
        if (int rc = ctx_wait_idle(c)) return rc;      // a host call blocks anyway: wait out an earlier asynchronous device call here
        for (size_t s0 = b; s0 < e; s0 += CH) {
            size_t m = std::min(CH, e - s0);
            size_t ob = m + (gt_out ? m * 384 : 0) + (miller_out ? m * 384 : 0);
            int rc = ctx_stage(c, m * 384, ob); if (rc) return rc;
            memcpy(c->h_pin, g1s + s0 * 256, m * 256); memcpy(c->h_pin + m * 256, g2s + s0 * 128, m * 128);
            CK(cudaMemcpyAsync(c->d_in, c->h_pin, m * 384, cudaMemcpyHostToDevice, c->stream));
            uint8_t* d_gt = gt_out ? c->d_out + m : nullptr; uint8_t* d_ml = miller_out ? c->d_out + m + (gt_out ? m * 384 : 0) : nullptr;
            rc = run_pairing4(c, vk, m, c->d_in, c->d_in + m * 256, c->d_out, d_gt, d_ml, c->stream); if (rc) return rc;
            CK(cudaMemcpyAsync(c->h_out, c->d_out, ob, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            collect_stage_ms(c);
            memcpy(ok_out + s0, c->h_out, m);
            if (gt_out) memcpy(gt_out + s0 * 384, c->h_out + m, m * 384);
            if (miller_out) memcpy(miller_out + s0 * 384, c->h_out + m + (gt_out ? m * 384 : 0), m * 384);
        }
        return 0;
    });
}
extern "C" int zkv_pairing4_batch_device(const zkv_vk* vk, int device, const void* d_g1s, const void* d_g2s, size_t n, void* d_ok_out, void* d_gt_out, void* stream) {
    if (!vk || !d_g1s || !d_g2s || !d_ok_out) return fail(ZKV_ERR_ARG, "zkv_pairing4_batch_device: null argument");
    DevCtx* c = vk_ctx(vk, device);
    if (!c) return fail(ZKV_ERR_ARG, "device not in the key's device list");
    if (n > MAX_CHUNK * 8) return fail(ZKV_ERR_ARG, "device batch too large");
    return device_call(c, device, stream, [&](cudaStream_t s) {
        return run_pairing4(c, vk, n, (const uint8_t*)d_g1s, (const uint8_t*)d_g2s, (uint8_t*)d_ok_out, (uint8_t*)d_gt_out, nullptr, s);
    });
}

// ------------------------------------------------------------------------------------------ hooks and small services
extern "C" int zkv_vk_x_batch(const zkv_vk* vk, const uint8_t* signals, int k, size_t n, uint8_t* out_points) {
    if (!vk || !signals || !out_points || k + 1 != vk->n_ic) return fail(ZKV_ERR_ARG, "zkv_vk_x_batch: bad argument");
    if (n == 0) return 0;
    if (n > MAX_CHUNK * 8) return fail(ZKV_ERR_ARG, "zkv_vk_x_batch: batch too large");
    DevCtx* c = vk->devs[0];
    std::lock_guard<std::mutex> lk(c->mu);
    CK(cudaSetDevice(c->device));
    int rc = ctx_wait_idle(c); if (rc) return rc;
    rc = ctx_reserve(c, n, (size_t)k * 8); if (rc) return rc;
    rc = ctx_stage(c, n * (size_t)k * 32, n * 64); if (rc) return rc;
    CK(cudaMemcpyAsync(c->d_in, signals, n * (size_t)k * 32, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(c->flags, 0, n, c->stream));
    k_generic_signals<<<nblk(n), TPB, 0, c->stream>>>((int)n, k, c->d_in, c->scal, c->flags);
    k_vkx<<<nblk(n), TPB, 0, c->stream>>>((int)n, c->scal, k, ZKV_WIN_PER_SCALAR, c->d_tab, c->h_ic0, c->px[2], c->py[2], c->flags);
    k_points_to_bytes<<<nblk(n), TPB, 0, c->stream>>>((int)n, c->px[2], c->py[2], c->d_out);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out_points, c->d_out, n * 64, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

// stand-alone scratch launcher for the stateless services below
template <class L>
static int with_scratch(int device, const void* in0, size_t b0, const void* in1, size_t b1, void* out0, size_t ob0, void* out1, size_t ob1, L launch) {
    if (zkv_device_count() <= device || device < 0) return fail(ZKV_ERR_CUDA, "no such CUDA device (this library has no CPU path)");
    CK(cudaSetDevice(device));
    uint8_t *d0 = nullptr, *d1 = nullptr, *o0 = nullptr, *o1 = nullptr;
    CK(cudaMalloc(&d0, b0 + 16)); CK(cudaMalloc(&d1, b1 + 16)); CK(cudaMalloc(&o0, ob0 + 16)); CK(cudaMalloc(&o1, ob1 + 16));
    CK(cudaMemcpy(d0, in0, b0, cudaMemcpyHostToDevice)); if (b1) CK(cudaMemcpy(d1, in1, b1, cudaMemcpyHostToDevice));
    launch(d0, d1, o0, o1);
    cudaError_t e = cudaGetLastError(); if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) { e = cudaMemcpy(out0, o0, ob0, cudaMemcpyDeviceToHost); if (e == cudaSuccess && ob1) e = cudaMemcpy(out1, o1, ob1, cudaMemcpyDeviceToHost); }
    cudaFree(d0); cudaFree(d1); cudaFree(o0); cudaFree(o1);
    if (e != cudaSuccess) return fail(ZKV_ERR_CUDA, cudaGetErrorString(e));
    return 0;
}
extern "C" int zkv_fp_mul_batch(const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out, int device) {
    if (!a || !b || !out) return fail(ZKV_ERR_ARG, "null");
    if (n == 0) return 0;
    uint8_t dummy;
    return with_scratch(device, a, n * 32, b, n * 32, out, n * 32, &dummy, 0, [&](uint8_t* d0, uint8_t* d1, uint8_t* o0, uint8_t*) { k_fp_mul_bytes<<<nblk(n), TPB>>>((int)n, d0, d1, o0); });
}
extern "C" int zkv_fp12_op_batch(int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out, int device) {
    const bool slots = op >= 16;                    // 16 + k: the shared-memory-resident form (lazy.cuh) of operation k
    const int k = slots ? op - 16 : op;
    if (!a || !out || k < 0 || k > (slots ? 10 : 9) || ((k == 0 || k == 2 || k == 9 || k == 10) && !b)) return fail(ZKV_ERR_ARG, "zkv_fp12_op_batch: bad argument");
    if (n == 0) return 0;
    uint8_t dummy;
    if (!slots)
        return with_scratch(device, a, n * 384, b ? b : &dummy, b ? n * 384 : 0, out, n * 384, &dummy, 0,
                            [&](uint8_t* d0, uint8_t* d1, uint8_t* o0, uint8_t*) { k_fp12_op<<<nblk(n, ZKV_HTPB), ZKV_HTPB>>>((int)n, k, d0, b ? d1 : nullptr, o0); });
    const size_t launched = (size_t)nblk(n, LZ_NT) * LZ_NT;
    std::vector<uint8_t> sink(1);
    // second output buffer of with_scratch doubles as the kernel's per-thread scratch (7 Fp12 per launched thread); nothing is copied back from it
    if (zkv_device_count() <= device || device < 0) return fail(ZKV_ERR_CUDA, "no such CUDA device (this library has no CPU path)");
    CK(cudaSetDevice(device));
    CK(cudaFuncSetAttribute(k_lz_fp12_op, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM_MILLER));
    fp12* scratch = nullptr; CK(cudaMalloc(&scratch, launched * 7 * sizeof(fp12)));
    nline_t* ztab = nullptr; CK(cudaMalloc(&ztab, ZKV_LINES_PER_G2 * sizeof(nline_t))); CK(cudaMemset(ztab, 0, ZKV_LINES_PER_G2 * sizeof(nline_t)));
    int rc = with_scratch(device, a, n * 384, b ? b : &dummy, b ? n * 384 : 0, out, n * 384, &dummy, 0,
                          [&](uint8_t* d0, uint8_t* d1, uint8_t* o0, uint8_t*) { k_lz_fp12_op<<<nblk(n, LZ_NT), LZ_NT, LZ_SMEM_MILLER>>>((int)n, k, d0, b ? d1 : nullptr, o0, scratch, ztab); });
    cudaFree(scratch); cudaFree(ztab);
    return rc;
}
extern "C" int zkv_g2_check_batch(const uint8_t* g2s, size_t n, uint8_t* out, int device) {
    if (!g2s || !out) return fail(ZKV_ERR_ARG, "null");
    if (n == 0) return 0;
    uint8_t dummy;
    return with_scratch(device, g2s, n * 128, &dummy, 0, out, n, &dummy, 0, [&](uint8_t* d0, uint8_t*, uint8_t* o0, uint8_t*) { k_g2_check_bytes<<<nblk(n), TPB>>>((int)n, d0, o0); });
}
extern "C" int zkv_ec_add_batch(const uint8_t* in, size_t n, uint8_t* out, uint8_t* reverted, int device) {
    if (!in || !out || !reverted) return fail(ZKV_ERR_ARG, "null");
    if (n == 0) return 0;
    uint8_t dummy;
    return with_scratch(device, in, n * 128, &dummy, 0, out, n * 64, reverted, n, [&](uint8_t* d0, uint8_t*, uint8_t* o0, uint8_t* o1) { k_ec_add<<<nblk(n), TPB>>>((int)n, d0, o0, o1); });
}
extern "C" int zkv_ec_mul_batch(const uint8_t* in, size_t n, uint8_t* out, uint8_t* reverted, int device) {
    if (!in || !out || !reverted) return fail(ZKV_ERR_ARG, "null");
    if (n == 0) return 0;
    uint8_t dummy;
    return with_scratch(device, in, n * 96, &dummy, 0, out, n * 64, reverted, n, [&](uint8_t* d0, uint8_t*, uint8_t* o0, uint8_t* o1) { k_ec_mul<<<nblk(n), TPB>>>((int)n, d0, o0, o1); });
}
extern "C" int zkv_g2_mul_batch(const uint8_t* points, int broadcast_point, const uint8_t* scalars, size_t n, uint8_t* out, uint8_t* reverted, int device) {
    if (!points || !scalars || !out || !reverted) return fail(ZKV_ERR_ARG, "null");
    if (n == 0) return 0;
    return with_scratch(device, points, broadcast_point ? 128 : n * 128, scalars, n * 32, out, n * 128, reverted, n,
                        [&](uint8_t* d0, uint8_t* d1, uint8_t* o0, uint8_t* o1) { k_g2_mul<<<nblk(n), TPB>>>((int)n, d0, broadcast_point, d1, o0, o1); });
}
// ------------------------------------------------------------------------------------------ general ecPairing service (0x08, groth16.rs:109-128)
// n instances of a k-pair product check with EVERY G2 point variable: the byte semantics of the precompile (EIP-197): each pair is
// G1 (64 B) || G2 (128 B); a coordinate >= p, a point off its curve or a G2 point outside the order-r subgroup makes the call fail
// (reverted[i] = 1, out word zero); a pair with a member at infinity contributes 1; k = 0 is the empty product (true).
// out: n x 32 B, the precompile's return word (0...01 or 0...00); miller_out (optional, n x 384 B): the Miller-loop value.
static int ec_pairing_on(int device, const uint8_t* in, int k, size_t n, uint8_t* out, uint8_t* reverted, uint8_t* miller_out) {
    CK(cudaSetDevice(device));
    CK(cudaFuncSetAttribute(k_pairing_lz, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM_BYTES));
    CK(cudaFuncSetAttribute(k_final_exp_lz, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM_BYTES));
    const size_t CH = (size_t)1 << 16;
    const size_t cap = std::min(CH, (n + LZ_NT - 1) / LZ_NT * LZ_NT), K = (size_t)k;
    uint8_t *d_in = nullptr, *d_pst = nullptr, *d_pskip = nullptr, *d_ifl = nullptr, *d_st = nullptr, *d_ml = nullptr;
    fp *d_px = nullptr, *d_py = nullptr; fp2 *d_qx = nullptr, *d_qy = nullptr; g2j* d_r = nullptr; fp12 *d_f = nullptr, *d_fes = nullptr;
    auto release = [&]() { cudaFree(d_in); cudaFree(d_pst); cudaFree(d_pskip); cudaFree(d_ifl); cudaFree(d_st); cudaFree(d_ml); cudaFree(d_px); cudaFree(d_py); cudaFree(d_qx); cudaFree(d_qy); cudaFree(d_r); cudaFree(d_f); cudaFree(d_fes); };
#define CKR(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { release(); return fail(ZKV_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } } while (0)
    CKR(cudaMalloc(&d_in, cap * K * 192)); CKR(cudaMalloc(&d_pst, cap * K)); CKR(cudaMalloc(&d_pskip, cap * K)); CKR(cudaMalloc(&d_ifl, cap)); CKR(cudaMalloc(&d_st, cap));
    CKR(cudaMalloc(&d_px, cap * K * sizeof(fp))); CKR(cudaMalloc(&d_py, cap * K * sizeof(fp))); CKR(cudaMalloc(&d_qx, cap * K * sizeof(fp2))); CKR(cudaMalloc(&d_qy, cap * K * sizeof(fp2)));
    CKR(cudaMalloc(&d_r, cap * K * sizeof(g2j))); CKR(cudaMalloc(&d_f, cap * sizeof(fp12))); CKR(cudaMalloc(&d_fes, cap * 6 * sizeof(fp12)));
    if (miller_out) CKR(cudaMalloc(&d_ml, cap * 384));
    std::vector<uint8_t> h_st(cap), h_ifl(cap);
    for (size_t s0 = 0; s0 < n; s0 += CH) {
        const size_t m = std::min(CH, n - s0);
        const int blocks = nblk(m, LZ_NT);
        CKR(cudaMemcpy(d_in, in + s0 * K * 192, m * K * 192, cudaMemcpyHostToDevice));
        CKR(cudaMemset(d_px, 0, cap * K * sizeof(fp))); CKR(cudaMemset(d_py, 0, cap * K * sizeof(fp))); CKR(cudaMemset(d_qx, 0, cap * K * sizeof(fp2))); CKR(cudaMemset(d_qy, 0, cap * K * sizeof(fp2)));
        CKR(cudaMemset(d_pst, F_SKIP0, cap * K)); CKR(cudaMemset(d_pskip, 1, cap * K));          // padding entries: skipped pairs
        k_pairing_decode<<<nblk(m * K), TPB>>>((int)m, k, cap, d_in, d_px, d_py, d_qx, d_qy, d_pst);
        k_g2_check<<<nblk(cap * K), TPB>>>((int)(cap * K), d_qx, d_qy, d_pst);
        k_pairing_flags<<<nblk(m), TPB>>>((int)m, k, cap, d_pst, d_pskip, d_ifl);
        LzGenIn gi; memset(&gi, 0, sizeof gi);
        gi.px = d_px; gi.py = d_py; gi.qx = d_qx; gi.qy = d_qy; gi.rst = d_r; gi.pskip = d_pskip; gi.stride = cap; gi.nvar = k; gi.nfix = 0;
        k_pairing_lz<<<blocks, LZ_NT, LZ_SMEM_BYTES>>>((int)m, gi, d_f, ZKV_ATE_NAF_LEN - 2, 0, 1, 1);
        if (miller_out) k_f12_to_bytes<<<nblk(m), TPB>>>((int)m, d_f, d_ml);
        k_final_exp_lz<<<blocks, LZ_NT, LZ_SMEM_BYTES>>>((int)m, 0, 3, d_f, d_fes, d_ifl, d_st, nullptr, 1);
        CKR(cudaGetLastError());
        CKR(cudaMemcpy(h_st.data(), d_st, m, cudaMemcpyDeviceToHost)); CKR(cudaMemcpy(h_ifl.data(), d_ifl, m, cudaMemcpyDeviceToHost));
        if (miller_out) CKR(cudaMemcpy(miller_out + s0 * 384, d_ml, m * 384, cudaMemcpyDeviceToHost));
        for (size_t t = 0; t < m; t++) {
            uint8_t* o = out + (s0 + t) * 32; memset(o, 0, 32);
            if (h_ifl[t]) { reverted[s0 + t] = 1; if (miller_out) memset(miller_out + (s0 + t) * 384, 0, 384); }
            else { reverted[s0 + t] = 0; o[31] = h_st[t] == 1 ? 1 : 0; }
        }
    }
#undef CKR
    release();
    return 0;
}
extern "C" int zkv_ec_pairing_batch(const uint8_t* in, int k, size_t n, uint8_t* out, uint8_t* reverted, uint8_t* miller_out, int device) {
    if (!out || !reverted || k < 0 || k > 64 || (k && n && !in)) return fail(ZKV_ERR_ARG, "zkv_ec_pairing_batch: bad argument");
    if (n == 0) return 0;
    if (zkv_device_count() <= device || device < 0) return fail(ZKV_ERR_CUDA, "no such CUDA device (this library has no CPU path)");
    if (k == 0) {                                           // empty product: true, no curve work at all (EIP-197)
        for (size_t i = 0; i < n; i++) { memset(out + 32 * i, 0, 32); out[32 * i + 31] = 1; reverted[i] = 0; }
        if (miller_out) for (size_t i = 0; i < n; i++) { memset(miller_out + 384 * i, 0, 384); miller_out[384 * i + 31] = 1; }
        return 0;
    }
    return ec_pairing_on(device, in, k, n, out, reverted, miller_out);
}
// one precompile call on raw bytes: len must be a multiple of 192 (else the call fails: *reverted = 1)
extern "C" int zkv_ec_pairing(const uint8_t* in, size_t len, uint8_t out[32], uint8_t* reverted, int device) {
    if (!out || !reverted || (len && !in)) return fail(ZKV_ERR_ARG, "zkv_ec_pairing: null argument");
    if (len % 192) { memset(out, 0, 32); *reverted = 1; return 0; }
    return zkv_ec_pairing_batch(in, (int)(len / 192), 1, out, reverted, nullptr, device);
}

extern "C" int zkv_last_stage_ms(const void* handle_vk, int device, float* out, int cap) {
    const zkv_vk* vk = (const zkv_vk*)handle_vk;
    if (!vk || !out) return fail(ZKV_ERR_ARG, "null");
    DevCtx* c = vk_ctx(vk, device);
    if (!c) return fail(ZKV_ERR_ARG, "device not in the key's device list");
    std::lock_guard<std::mutex> lk(c->mu);
    if (cudaSetDevice(device) == cudaSuccess) { cudaEventSynchronize(c->ev[5]); collect_stage_ms(c); }
    int m = std::min(cap, 5);
    for (int i = 0; i < m; i++) out[i] = c->stage_ms[i];
    return m;
}
extern "C" const void* zkv_risc0_vk(const zkv_risc0* h) { return h ? h->vk : nullptr; }
extern "C" const void* zkv_sp1_vk(const zkv_sp1* h) { return h ? h->vk : nullptr; }

// proofs in one full wave of a heavy kernel on `device` (SMs x resident blocks per SM x threads per block): 0 = k_miller_lz, 1 = k_final_exp_lz
extern "C" long long zkv_wave_proofs(int device, int kernel) {
    if (zkv_device_count() <= device || device < 0) return fail(ZKV_ERR_CUDA, "no such CUDA device");
    if (cudaSetDevice(device) != cudaSuccess) return fail(ZKV_ERR_CUDA, "cudaSetDevice failed");
    cudaDeviceProp prop; if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(ZKV_ERR_CUDA, "cudaGetDeviceProperties failed");
    int per_sm = 0;
    cudaError_t e; int tpb;
    switch (kernel) {
        case 0: tpb = LZ_NT; cudaFuncSetAttribute(k_miller_lz, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM_MILLER); e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_miller_lz, LZ_NT, LZ_SMEM_MILLER); break;
        case 1: tpb = LZ_NT; cudaFuncSetAttribute(k_final_exp_lz, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SMEM_BYTES); e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_final_exp_lz, LZ_NT, LZ_SMEM_BYTES); break;
        default: return fail(ZKV_ERR_ARG, "zkv_wave_proofs: kernel must be 0 or 1 (2 and 3, the round-1 kernels, were removed)");
    }
    if (e != cudaSuccess) return fail(ZKV_ERR_CUDA, cudaGetErrorString(e));
    return (long long)prop.multiProcessorCount * per_sm * tpb;
}
extern "C" int zkv_imad_peak(int device, double* wide_per_s, double* fpmul_per_s) {
    if (zkv_device_count() <= device || device < 0) return fail(ZKV_ERR_CUDA, "no such CUDA device");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, device));
    int blocks = prop.multiProcessorCount * 8, threads = 256;
    uint64_t* d_out; fp* d_fp;
    CK(cudaMalloc(&d_out, (size_t)blocks * threads * 8)); CK(cudaMalloc(&d_fp, (size_t)blocks * threads * sizeof(fp)));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    float best_w = 1e30f, best_f = 1e30f;
    const int it_w = 4096, it_f = 2048;
    for (int rep = 0; rep < 5; rep++) {
        CK(cudaEventRecord(e0)); k_imad_wide<<<blocks, threads>>>((uint32_t*)d_out, 0x9e3779b9u, 0x7f4a7c15u, it_w); CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1));
        float ms; CK(cudaEventElapsedTime(&ms, e0, e1)); if (rep) best_w = std::min(best_w, ms);
        CK(cudaEventRecord(e0)); k_fpmul_chain<<<blocks, threads>>>(d_fp, it_f); CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1));
        CK(cudaEventElapsedTime(&ms, e0, e1)); if (rep) best_f = std::min(best_f, ms);
    }
    CK(cudaGetLastError());
    if (wide_per_s) *wide_per_s = (double)blocks * threads * it_w * 64.0 / (best_w * 1e-3);
    if (fpmul_per_s) *fpmul_per_s = (double)blocks * threads * it_f * 2.0 / (best_f * 1e-3);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d_out); cudaFree(d_fp);
    return 0;
}
