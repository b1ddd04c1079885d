// capi.cu — device context, key upload, the batched circuit-bootstrap pipeline and the fused AES paths behind the C ABI
// of include/tfhe_aes_cuda.h.  No CPU fallback: every entry point that computes fails with TAC_ERR_CUDA when there is
// no usable CUDA device.
#include "../../include/tfhe_aes_cuda.h"
#include "kernels_common.cuh"
#include "aes_plan.h"
#include "aes_ccm.h"
#include "aes_gcm.h"
#include "kernels_gemm_umma.cuh"
#include "ep_step.cuh"
#include "shape_launch.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

using namespace tac;

namespace {

// last error of the calling thread (entry points may be used from many threads; a per-context string would race)
thread_local std::string g_error;

// device memory owned by the context: freed when the buffer is, or when ensure() replaces it by a larger one
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
    ~DevBuf() { if (p) cudaFree(p); }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// AES-GCM: the GHASH key table H^1..H^depth [K][depth][128][kN+1] of a key set, valid while its schedules are resident
struct GcmTable { DevBuf buf; int depth = 0; bool valid = false; };

// A set of resident AES-128 key schedules: the single schedule (n = 1) or the key table (n entries), each with its inverse
// schedules and its GHASH key table.  w [n][44 words][4][8][kN+1]; dk, the equivalent inverse cipher's schedules, same
// layout, valid while made from (or uploaded for) the resident w.  n = 0: absent.  Writing w sets n = 0 and marks dk and
// the GHASH table stale first; n is set once w is complete.  The state errors name the calls that fix them.
struct KeySet {
    DevBuf w, dk;
    int n = 0;
    bool dk_valid = false;
    GcmTable gcm;
    const char *absent, *no_dk, *no_gcm;
    KeySet(const char* absent, const char* no_dk, const char* no_gcm) : absent(absent), no_dk(no_dk), no_gcm(no_gcm) {}
};

struct Lut {
    int n_in, n_out;
    size_t len;          // words per output
    uint64_t* dev;
};

enum Stage { ST_KS = 0, ST_PBS, ST_PFKS, ST_FFT, ST_VP, ST_COUNT };
constexpr uint32_t kFixCap = 1u << 16;

}  // namespace

// a circuit_bootstrap call waiting in the coalescing queue (tac_wopbs_coalesced)
struct PendingWopbs {
    int lut_id, batch;
    const uint64_t* in;
    uint64_t* out;
    int rc = 0;
    bool done = false;
    std::string err;
};

struct tac_ctx {
    // Every entry point takes `mu` (recursive: entry points call each other), so a context may be shared by any number of
    // host threads — the reference calls circuit_bootstrap from rayon workers (fhe_sbox_gal_mul_pbs.rs:33-41, main.rs:148-152).
    std::recursive_mutex mu;
    // coalescing queue: concurrent single-SBOX callers are merged into one batched pass
    std::mutex q_mu;
    std::condition_variable q_cv;
    std::vector<PendingWopbs*> q_pending;
    bool q_leader = false;
    int q_window_us = 200, q_max_batch = 4096;
    uint64_t q_passes = 0, q_requests = 0;
    TacParams p;
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    // keys
    DevBuf bsk_f;                        // cplx
    DevBuf ksk, pfpksk, ks_corr, pfks_corr;
    DevBuf ks_planes;                    // byte planes of the KSK
    DevBuf pfks_planes;                  // byte-plane tiles of the PFPKSK for the tcgen05 GEMM (kernels_gemm_umma.cuh)
    DevBuf pfks_fix;                     // uint32: [0] = count, then uint2 (ct, k) entries
    bool keys_allocated = false, keys_valid = false;
    // tables
    DevBuf wT;                     // cplx: combined twist/twiddle table (ep_core.cuh)
    const ShapeOps* ops = nullptr; // kernels of this (N, k)
    // LUTs
    std::vector<Lut> luts;
    int aes_lut24 = -1, aes_lut8 = -1, aes_lut1 = -1;
    int aes_lut_inv32 = -1, aes_lut_inv8 = -1, aes_lut_key32 = -1;   // decryption: InvS·{14,11,13,9}, InvS, b·{14,11,13,9}
    int ccm_lut_zero8 = -1, ccm_lut_ones8 = -1, ccm_lut_ones2 = -1;   // AES-CCM tag check: byte == 0, 8 bits all 1, 2 bits all 1
    int gf_lut_mul = -1;                 // GF(2^128) product: 8 → 7 carry-less product of two 4-bit polynomials
    // AES keys: the single schedule and, for AES under many keys, a table of schedules; neither replaces the other
    KeySet single{"no key schedule on the device (tac_aes_set_key_schedule)",
                  "no inverse key schedule for the resident key schedule (tac_aes_inv_key_schedule or tac_aes_set_inv_key_schedule)",
                  "no GHASH key table for the resident key schedule (tac_aes_gcm_hash_key)"};
    KeySet table{"no key table on the device (tac_aes_key_table or tac_aes_set_key_table)",
                 "no inverse key table for the resident key table (tac_aes_inv_key_table or tac_aes_set_inv_key_table)",
                 "no GHASH key table for the resident key table (tac_aes_gcm_hash_key_table)"};
    DevBuf rc_rows;                  // trivial(RC[1..10]) as byte ciphertexts [10][8][kN+1], uploaded once
    // workspace
    DevBuf ws_in, ws_out, ws_small, ws_ksdig, ws_pbs, ws_pfdig, ws_ggsw, ws_ggswf, ws_tree_a, ws_tree_b, ws_state, ws_muls, ws_misc;
    DevBuf ws_plan, ws_rep;          // public-block AES: uploaded plan tables / public bytes, compact S-box inputs
    // AES-CCM, apart from the buffers aes_blocks_dev reuses on every call: the public call's output (rows 0..n−1 are the
    // CBC-MAC chain state), the chain input / tag check, and the descriptors of all steps
    DevBuf ccm_pub, ccm_work, ccm_desc;
    // AES-GCM: the linear layer's descriptors, group sums and level outputs; the product's GGSW index table, box outputs
    // and operands; a transciphering call's buffers
    DevBuf lin_desc, lin_sum, lin_lvl, gf_idx, gf_box, gf_ops, gf_prod, gcm_pub, gcm_dy;
    int gf_idx_np = 0;                   // products per pass gf_idx was built for
    size_t max_cts = 16384;
    uint32_t fix_cap = kFixCap;      // capacity of the PFKS tie list in use (TAC_FIX_CAP lowers it: exercises the overflow path)
    // profiling: one event tuple per pipeline pass, recorded without synchronising; read back by tac_ctx_stage_times
    bool profiling = false;
    struct ProfRec { cudaEvent_t ev[ST_COUNT + 1]; };
    std::vector<ProfRec> prof_pool;
    size_t prof_used = 0;
    uint64_t launches = 0;

    int big() const { return p.k * p.N; }
    int G() const { return p.k + 1; }
    size_t bsk_cplx() const { return (size_t)p.n * p.pbs_l * G() * G() * (p.N / 2); }
    size_t ksk_words() const { return (size_t)big() * p.ks_l * (p.n + 1); }
    size_t pfpksk_words() const { return (size_t)G() * (big() + 1) * p.pfks_l * G() * p.N; }
};

namespace {

int fail(tac_ctx*, int code, const std::string& msg) {
    g_error = msg;
    return code;
}
#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess) return fail(ctx, TAC_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
    } while (0)
#define LOCK(ctx) std::lock_guard<std::recursive_mutex> lock__((ctx)->mu)
#define TRY(call)              \
    do {                       \
        int rc__ = (call);     \
        if (rc__) return rc__; \
    } while (0)

// room for `bytes` in b (contents not kept when it grows); `what` names the buffer in the error text
int ensure(tac_ctx* ctx, DevBuf& b, size_t bytes, const char* what = "a device buffer") {
    if (b.cap >= bytes) return TAC_OK;
    b = DevBuf();
    if (cudaMalloc(&b.p, bytes) != cudaSuccess) {
        cudaGetLastError();          // clear the allocation error so that the next launch check does not report it
        b.p = nullptr;
        return fail(ctx, TAC_ERR_CUDA, std::string(what) + " (" + std::to_string(bytes >> 20) + " MiB) does not fit in device memory");
    }
    b.cap = bytes;
    return TAC_OK;
}
inline int grid1d(size_t total, int block, int sms) {
    const size_t need = (total + block - 1) / block;
    const size_t cap = (size_t)sms * 16;
    return (int)std::max<size_t>(1, std::min(need, cap));
}
int post_launch(tac_ctx* ctx, const char* what) {
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, TAC_ERR_CUDA, std::string(what) + " launch: " + cudaGetErrorString(e));
    return TAC_OK;
}
bool supported_shape(const TacParams& p) {
    return (p.N == 512 && p.k == 4) || (p.N == 1024 && p.k == 2);
}

// Constraints of the kernels beyond (N, k); violating any of them used to give silently wrong ciphertexts.
std::string unsupported_params(const TacParams& p) {
    const long big = (long)p.k * p.N;
    if (p.n < 1 || p.n > 2048) return "lwe_dimension out of range";
    if ((p.n & 1) == 0) return "lwe_dimension must be odd (the integer GEMM works on column pairs of the (n+1)-wide keyswitch key)";
    if (p.pbs_l < 1 || p.pbs_l > 4 || p.pbs_b < 1 || p.pbs_b > 15 || p.pbs_b * p.pbs_l > 63)
        return "pbs decomposition: need level <= 4, base_log <= 15 (digits are cached as 16-bit fields)";
    if (p.cbs_l < 1 || p.cbs_l > 2) return "cbs_level must be 1 or 2 (the vertical-packing kernels are instantiated for these)";
    if (p.cbs_b < 1 || p.cbs_b > 15 || p.cbs_b * p.cbs_l > 62) return "cbs_base_log must be in [1, 15]";
    if (p.ks_l < 1 || p.ks_b < 1 || p.ks_b > 7 || p.ks_b * p.ks_l > 63) return "keyswitch decomposition: base_log must be <= 7 (one byte limb on the tensor cores)";
    if (p.pfks_l < 1 || p.pfks_b < 1 || p.pfks_b > 31 || p.pfks_b * p.pfks_l > 63) return "pfks decomposition: base_log must be <= 31";
    // s32 tensor-memory accumulators hold 2 byte-limb products per k: exact while K·2·255² < 2^31
    if (big * p.ks_l >= 16000 || (big + 1) * p.pfks_l >= 16000) return "decomposed length K = dim·level must stay below 16000 (s32 accumulators of the byte-limb GEMM)";
    if (p.max_noise_sq < 1) return "max_noise_level_squared must be positive";
    return "";
}

// ---------------------------------------------------------------------------------------------- launch wrappers
KLaunch klaunch(tac_ctx* ctx) { return KLaunch{ctx->stream, ctx->wT.as<cplx>(), ctx->sm_count}; }
int check_launch(tac_ctx* ctx, cudaError_t e, const char* what) {
    ctx->launches++;
    if (e == cudaErrorInvalidValue) return fail(ctx, TAC_ERR_ARG, std::string(what) + ": unsupported level count / shape for this parameter set");
    if (e != cudaSuccess) return fail(ctx, TAC_ERR_CUDA, std::string(what) + " launch: " + cudaGetErrorString(e));
    return TAC_OK;
}
int poly_fft(tac_ctx* ctx, const uint64_t* polys, size_t npoly, cplx* out) {
    if (npoly == 0) return TAC_OK;
    return check_launch(ctx, ctx->ops->poly_fft(klaunch(ctx), polys, npoly, 1.0 / (ctx->p.N / 2), out), "poly_fft_kernel");
}

int gemm(tac_ctx* ctx, const uint32_t* dig, int nct, int Kd, const uint64_t* key, int W, int nkeys, const uint64_t* corr,
         const uint64_t* last_col_add, size_t add_stride, uint64_t* out) {
    if (nct == 0) return TAC_OK;
    const int tiles = (W + 127) / 128;
    if (nct >= 256) {
        dim3 grid(tiles * nkeys, (nct + 63) / 64);
        lwe_gemm_kernel<16><<<grid, 256, 0, ctx->stream>>>(dig, nct, Kd, key, W, nkeys, corr, last_col_add, add_stride, out);
    } else {
        dim3 grid(tiles * nkeys, (nct + 15) / 16);
        lwe_gemm_kernel<4><<<grid, 256, 0, ctx->stream>>>(dig, nct, Kd, key, W, nkeys, corr, last_col_add, add_stride, out);
    }
    return post_launch(ctx, "lwe_gemm_kernel");
}

// alpha: the bootstrap returns (sign bit of the input)·2·alpha; circuit bootstrapping uses 2^(63 − cbs_b·level), bit extraction 2^(delta_log + i − 1)
int pbs(tac_ctx* ctx, const uint64_t* small, int nct, uint64_t* out, uint64_t alpha = 0) {
    if (nct == 0) return TAC_OK;
    const TacParams& p = ctx->p;
    if (alpha == 0) alpha = 1ull << (63 - p.cbs_b * p.cbs_l);
    return check_launch(ctx, ctx->ops->pbs(klaunch(ctx), p.pbs_l, small, nct, p.n, ctx->bsk_f.as<cplx>(), p.pbs_b, alpha, out), "pbs kernel");
}

// vertical packing of `nbox` boxes from Fourier GGSWs ([nbox][n_in][cbs_l][G][G][M]) → out [nbox][n_out][big+1]
int vertical_packing(tac_ctx* ctx, const Lut& lut, const cplx* ggsw_f, int nbox, uint64_t* out) {
    const TacParams& p = ctx->p;
    const int logN = ilog2(p.N);
    const int tree_bits = lut.n_in > logN ? lut.n_in - logN : 0;
    const uint64_t* init = nullptr;
    if (tree_bits > 0) {
        // CMux tree, level order: layer j uses GGSW (tree_bits-1-j)  ([U] wop_pbs.rs::cmux_tree_memory_optimized)
        const size_t glwe = (size_t)ctx->G() * p.N;
        int nodes = 1 << tree_bits;
        TRY(ensure(ctx, ctx->ws_tree_a, (size_t)nbox * lut.n_out * (nodes / 2) * glwe * 8));
        TRY(ensure(ctx, ctx->ws_tree_b, (size_t)nbox * lut.n_out * std::max(1, nodes / 4) * glwe * 8));
        const uint64_t* cur = nullptr;
        uint64_t* bufs[2] = {ctx->ws_tree_a.as<uint64_t>(), ctx->ws_tree_b.as<uint64_t>()};
        int which = 0;
        for (int j = 0; j < tree_bits; j++) {
            uint64_t* dst = bufs[which];
            TRY(check_launch(ctx, ctx->ops->tree(klaunch(ctx), p.cbs_l, ggsw_f, nbox, lut.n_in, tree_bits - 1 - j, lut.dev, lut.len, cur, nodes, lut.n_out, p.cbs_b, dst),
                             "cmux_tree_kernel"));
            cur = dst; which ^= 1; nodes /= 2;
        }
        init = cur;
    }
    return check_launch(ctx, ctx->ops->vp(klaunch(ctx), p.cbs_l, ggsw_f, nbox, lut.n_in, tree_bits, lut.dev, lut.len, init, lut.n_out, p.cbs_b, out), "vp_kernel");
}

int stage_event(tac_ctx* ctx, int idx) {
    if (!ctx->profiling) return TAC_OK;
    if (idx == 0) {
        if (ctx->prof_used == ctx->prof_pool.size()) {
            tac_ctx::ProfRec r;
            for (auto& e : r.ev) CU(cudaEventCreate(&e));
            ctx->prof_pool.push_back(r);
        }
        ctx->prof_used++;
    }
    CU(cudaEventRecord(ctx->prof_pool[ctx->prof_used - 1].ev[idx], ctx->stream));
    return TAC_OK;
}

// exact integer GEMM on the 5th-generation tensor cores (kernels_gemm_umma.cuh); DA / KP are operand tiles
template <int NLIMB>
int gemm_umma(tac_ctx* ctx, const uint8_t* DA, int nct, const uint8_t* KP, int W, int nkeys, int nkb, const uint64_t* corr,
              const uint64_t* last_col_add, size_t add_stride, uint64_t* out) {
    CU(cudaFuncSetAttribute(lwe_gemm_umma_kernel<NLIMB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UgCfg<NLIMB>::SMEM));
    const int mtiles = (nct + UG_MT - 1) / UG_MT, ntiles = (W + UG_NT - 1) / UG_NT;
    lwe_gemm_umma_kernel<NLIMB><<<mtiles * ntiles * nkeys, UG_THREADS, UgCfg<NLIMB>::SMEM, ctx->stream>>>(DA, nct, mtiles, KP, W, nkeys, nkb, corr, last_col_add,
                                                                                                      add_stride, out);
    return post_launch(ctx, NLIMB == 2 ? "lwe_gemm_umma_kernel<2>" : "lwe_gemm_umma_kernel<1>");
}
// keyswitch on the tensor cores (single digit limb): in [nct][big+1] → small [nct][n+1]
int stage_ks(tac_ctx* ctx, const uint64_t* in, int nct, uint64_t* small) {
    const TacParams& p = ctx->p;
    const int big = ctx->big(), Kd = big * p.ks_l, nkb = (Kd + UG_KB - 1) / UG_KB;
    const int W = p.n + 1, mpad = ((nct + UG_MT - 1) / UG_MT) * UG_MT;
    TRY(ensure(ctx, ctx->ws_ksdig, (size_t)nkb * 2 * mpad * 16));
    uint8_t* DA = ctx->ws_ksdig.as<uint8_t>();
    uint32_t* fix = ctx->pfks_fix.as<uint32_t>();
    umma_digit_tiles_kernel<<<grid1d((size_t)mpad * nkb * 2, 256, ctx->sm_count), 256, 0, ctx->stream>>>(
        in, nct, mpad, big + 1, p.ks_b, p.ks_l, Kd, nkb, 1, DA, fix, reinterpret_cast<uint2*>(fix + 2), 0);
    TRY(post_launch(ctx, "umma_digit_tiles_kernel(ks)"));
    return gemm_umma<1>(ctx, DA, nct, ctx->ks_planes.as<uint8_t>(), W, 1, nkb, ctx->ks_corr.as<uint64_t>(), in + big, (size_t)big + 1, small);
}
// PFKS with all k+1 keys on the tensor cores: in [nct][big+1] → ggsw_std [nct][G][G·N]
int stage_pfks(tac_ctx* ctx, const uint64_t* in, int nct, uint64_t* ggsw) {
    const TacParams& p = ctx->p;
    const int big1 = ctx->big() + 1, Kd = big1 * p.pfks_l, nkb = (Kd + UG_KB - 1) / UG_KB;
    const int W = ctx->G() * p.N, mpad = ((nct + UG_MT - 1) / UG_MT) * UG_MT;
    const uint64_t* pfpksk = ctx->pfpksk.as<uint64_t>();
    uint32_t* fix = ctx->pfks_fix.as<uint32_t>();
    if (p.pfks_b > 16) {       // digits wider than 16 bits (params_sqrd_lvl_1: base 2^24): 64-bit integer-pipe GEMM
        TRY(ensure(ctx, ctx->ws_pfdig, (size_t)nct * Kd * 4));
        pfks_digits_kernel<<<grid1d((size_t)nct * big1, 256, ctx->sm_count), 256, 0, ctx->stream>>>(in, nct, big1, p.pfks_b, p.pfks_l, ctx->ws_pfdig.as<uint32_t>());
        TRY(post_launch(ctx, "pfks_digits_kernel"));
        return gemm(ctx, ctx->ws_pfdig.as<uint32_t>(), nct, Kd, pfpksk, W, ctx->G(), ctx->pfks_corr.as<uint64_t>(), nullptr, 0, ggsw);
    }
    TRY(ensure(ctx, ctx->ws_pfdig, (size_t)2 * nkb * 2 * mpad * 16));
    CU(cudaMemsetAsync(fix, 0, 4, ctx->stream));
    uint8_t* DA = ctx->ws_pfdig.as<uint8_t>();
    umma_digit_tiles_kernel<<<grid1d((size_t)mpad * nkb * 2, 256, ctx->sm_count), 256, 0, ctx->stream>>>(
        in, nct, mpad, big1, p.pfks_b, p.pfks_l, Kd, nkb, 0, DA, fix, reinterpret_cast<uint2*>(fix + 2), ctx->fix_cap);
    TRY(post_launch(ctx, "umma_digit_tiles_kernel(pfks)"));
    TRY(gemm_umma<2>(ctx, DA, nct, ctx->pfks_planes.as<uint8_t>(), W, ctx->G(), nkb, ctx->pfks_corr.as<uint64_t>(), nullptr, 0, ggsw));
    pfks_fixup_kernel<<<64, 256, 0, ctx->stream>>>(fix, reinterpret_cast<const uint2*>(fix + 2), ctx->fix_cap, pfpksk, Kd, W, ctx->G(), ggsw);
    TRY(post_launch(ctx, "pfks_fixup_kernel"));
    // more ties than the list holds (crafted / trivial inputs): this kernel re-derives them all; otherwise it returns at once
    pfks_fixup_scan_kernel<<<dim3((ctx->G() * W + 255) / 256, std::min(nct, 2 * ctx->sm_count)), 256, 0, ctx->stream>>>(
        fix, ctx->fix_cap, in, nct, big1, p.pfks_b, p.pfks_l, pfpksk, Kd, W, ctx->G(), ggsw);
    return post_launch(ctx, "pfks_fixup_scan_kernel");
}

// The GGSW stage of a circuit bootstrap: keyswitch → PBS (one per level) → PFKS → FFT of nct input bits [nct][big+1] into
// Fourier GGSWs ggsw_f [nct][cbs_l][G][G][M] (room provided by the caller)
int ggsw_stage(tac_ctx* ctx, const uint64_t* cin, int nct, cplx* ggsw_f) {
    const TacParams& p = ctx->p;
    const int big1 = ctx->big() + 1, G = ctx->G(), lc = p.cbs_l;
    const size_t ggsw_words = (size_t)G * G * p.N;
    TRY(ensure(ctx, ctx->ws_small, (size_t)nct * (p.n + 1) * 8));
    TRY(ensure(ctx, ctx->ws_pbs, (size_t)nct * lc * big1 * 8));
    TRY(ensure(ctx, ctx->ws_ggsw, (size_t)nct * lc * ggsw_words * 8));
    TRY(stage_event(ctx, 0));
    TRY(stage_ks(ctx, cin, nct, ctx->ws_small.as<uint64_t>()));                       // extract_dual_bit_from_bit
    TRY(stage_event(ctx, 1));
    // circuit_bootstrap_boolean: one homomorphic_shift_boolean per level (all four shipped parameter sets have one level)
    if (lc == 1) {
        TRY(pbs(ctx, ctx->ws_small.as<uint64_t>(), nct, ctx->ws_pbs.as<uint64_t>()));
    } else {
        TRY(ensure(ctx, ctx->ws_tree_a, (size_t)nct * big1 * 8));
        for (int lv = 1; lv <= lc; lv++) {          // level lv lands at [ct][lv-1] so that the PFKS rows come out as [ct][level][row]
            TRY(pbs(ctx, ctx->ws_small.as<uint64_t>(), nct, ctx->ws_tree_a.as<uint64_t>(), 1ull << (63 - p.cbs_b * lv)));
            CU(cudaMemcpy2DAsync(ctx->ws_pbs.as<uint64_t>() + (size_t)(lv - 1) * big1, (size_t)lc * big1 * 8, ctx->ws_tree_a.p, (size_t)big1 * 8,
                                 (size_t)big1 * 8, (size_t)nct, cudaMemcpyDeviceToDevice, ctx->stream));
        }
    }
    TRY(stage_event(ctx, 2));
    TRY(stage_pfks(ctx, ctx->ws_pbs.as<uint64_t>(), nct * lc, ctx->ws_ggsw.as<uint64_t>()));
    TRY(stage_event(ctx, 3));
    TRY(poly_fft(ctx, ctx->ws_ggsw.as<uint64_t>(), (size_t)nct * lc * G * G, ggsw_f));   // fill_with_forward_fourier
    return stage_event(ctx, 4);
}

// the whole circuit bootstrap for `nbox` boxes resident on the device: the GGSW stage, then vertical packing
int wopbs_dev(tac_ctx* ctx, const Lut& lut, int nbox, const uint64_t* in, uint64_t* out) {
    const TacParams& p = ctx->p;
    if (!ctx->keys_valid) return fail(ctx, TAC_ERR_STATE, "evaluation keys not uploaded");
    const int big1 = ctx->big() + 1, G = ctx->G(), M = p.N / 2, lc = p.cbs_l;
    const int max_boxes = (int)std::max<size_t>(1, ctx->max_cts / ((size_t)lut.n_in * lc));
    for (int b0 = 0; b0 < nbox; b0 += max_boxes) {
        const int nb = std::min(max_boxes, nbox - b0);
        const int nct = nb * lut.n_in;
        const uint64_t* cin = in + (size_t)b0 * lut.n_in * big1;
        uint64_t* cout = out + (size_t)b0 * lut.n_out * big1;
        TRY(ensure(ctx, ctx->ws_ggswf, (size_t)nct * lc * G * G * M * sizeof(cplx)));
        TRY(ggsw_stage(ctx, cin, nct, ctx->ws_ggswf.as<cplx>()));
        TRY(vertical_packing(ctx, lut, ctx->ws_ggswf.as<cplx>(), nb, cout));
        TRY(stage_event(ctx, 5));
    }
    return TAC_OK;
}

int get_lut(tac_ctx* ctx, int id, const Lut** out) {
    if (id < 0 || id >= (int)ctx->luts.size()) return fail(ctx, TAC_ERR_STATE, "unknown LUT id");
    *out = &ctx->luts[id];
    return TAC_OK;
}

// LUT closures of the AES binding (reference fhe_impls/shortint_woppbs_1bit.rs:18-44, :94-129)
uint8_t gf_mul(uint8_t a, uint8_t b) {           // src/aes_128.rs:42-56
    uint8_t r = 0;
    for (int i = 0; i < 8; i++) {
        if (b & 1) r ^= a;
        const bool hi = a & 0x80;
        a = (uint8_t)(a << 1);
        if (hi) a ^= 0x1b;
        b >>= 1;
    }
    return r;
}
void sbox_table(uint8_t s[256]) {
    // S-box generated from its definition (multiplicative inverse in GF(2^8) followed by the affine map); equals the
    // table at src/aes_128.rs:18-35
    uint8_t p = 1, q = 1;
    do {
        p = (uint8_t)(p ^ (p << 1) ^ ((p & 0x80) ? 0x1b : 0));
        q ^= (uint8_t)(q << 1); q ^= (uint8_t)(q << 2); q ^= (uint8_t)(q << 4);
        if (q & 0x80) q ^= 0x09;
        const uint8_t x = (uint8_t)(q ^ (uint8_t)((q << 1) | (q >> 7)) ^ (uint8_t)((q << 2) | (q >> 6)) ^ (uint8_t)((q << 3) | (q >> 5)) ^ (uint8_t)((q << 4) | (q >> 4)));
        s[p] = (uint8_t)(x ^ 0x63);
    } while (p != 1);
    s[0] = 0x63;
}
// the n_in → n_out LUT of f (tac_generate_lut), registered on the context; its id into *id
int register_aes_lut(tac_ctx* ctx, int n_in, int n_out, const uint64_t* f, int* id) {
    std::vector<uint64_t> t(tac_lut_len(n_in, ctx->p.N) * n_out);
    tac_generate_lut(n_in, n_out, ctx->p.N, f, t.data());
    const int r = tac_lut_register(ctx, n_in, n_out, t.data(), t.size());
    if (r < 0) return r;
    *id = r;
    return TAC_OK;
}
int ensure_aes_luts(tac_ctx* ctx) {
    if (ctx->aes_lut24 >= 0) return TAC_OK;
    uint8_t S[256]; sbox_table(S);
    std::vector<uint64_t> f(256);
    for (int b = 0; b < 256; b++) f[b] = ((uint64_t)gf_mul(S[b], 1) << 16) | ((uint64_t)gf_mul(S[b], 2) << 8) | (uint64_t)gf_mul(S[b], 3);
    TRY(register_aes_lut(ctx, 8, 24, f.data(), &ctx->aes_lut24));
    for (int b = 0; b < 256; b++) f[b] = S[b];
    TRY(register_aes_lut(ctx, 8, 8, f.data(), &ctx->aes_lut8));
    const uint64_t ident[2] = {0, 1};
    return register_aes_lut(ctx, 1, 1, ident, &ctx->aes_lut1);
}
// LUTs of the equivalent inverse cipher (FIPS-197 §5.3.5), registered on the first decryption call only.  Outputs in the
// order of aes_mix_columns_kernel<false>: the byte times {14, 11, 13, 9}, 8 bits each, MSB first.
int ensure_aes_inv_luts(tac_ctx* ctx) {
    if (ctx->aes_lut_inv32 >= 0) return TAC_OK;
    uint8_t S[256], IS[256]; sbox_table(S);
    for (int b = 0; b < 256; b++) IS[S[b]] = (uint8_t)b;
    auto inv_mix = [](uint8_t b) {
        return ((uint64_t)gf_mul(b, 14) << 24) | ((uint64_t)gf_mul(b, 11) << 16) | ((uint64_t)gf_mul(b, 13) << 8) | (uint64_t)gf_mul(b, 9);
    };
    std::vector<uint64_t> f(256);
    for (int b = 0; b < 256; b++) f[b] = inv_mix(IS[b]);
    TRY(register_aes_lut(ctx, 8, 32, f.data(), &ctx->aes_lut_inv32));
    for (int b = 0; b < 256; b++) f[b] = IS[b];
    TRY(register_aes_lut(ctx, 8, 8, f.data(), &ctx->aes_lut_inv8));
    for (int b = 0; b < 256; b++) f[b] = inv_mix((uint8_t)b);
    return register_aes_lut(ctx, 8, 32, f.data(), &ctx->aes_lut_key32);
}

// static squared-noise bookkeeping of the AES circuit (NoiseLevelWithComponents::add_assign, shortint_woppbs_1bit.rs:63-77):
// round keys are fresh or bootstrapped (level 1); SBOX outputs carry 8·NOMINAL (:325)
int aes_noise_check(tac_ctx* ctx, int in_noise_sq, int rounds) {
    const int maxn = ctx->p.max_noise_sq;
    if (in_noise_sq + 1 > maxn || (rounds > 1 && 4 * 8 + 1 > maxn) || 8 + 1 > maxn)
        return fail(ctx, TAC_ERR_NOISE, "NoiseTooBig: the AES circuit needs max_noise_level_squared >= 33");
    return TAC_OK;
}

// The AES rounds of tac_aes_{en,de}crypt{,_public}_blocks_dev, forward cipher or equivalent inverse cipher (FIPS-197 §5.3.5):
//   Forward  s = in + w[0];        s = MixColumns(ShiftRows(S(s))) + w[rd]                for rd = 1 … rounds−1;  out = ShiftRows(S(s)) + w[40..43]
//   Inverse  s = in + dk[40..43];  s = InvMixColumns(InvShiftRows(InvS(s))) + dk[rounds−rd];                      out = InvShiftRows(InvS(s)) + dk[0..3]
// The final round adds w[40..43] (dk[0..3]) for every `rounds`, so decryption inverts encryption for the same `rounds`.
// Input: ciphertexts in device memory (in_dev), or, with in_dev NULL, PUBLIC blocks on the host (blocks_host, aes_plan.h):
// state0 = k_first + trivial(block), each round bootstraps only the plan's representatives, in one compact batch, and the
// mix-columns / final-round kernels read every position's S-box row through the plan's index table.  Rounds whose plan is
// the identity (every round of ciphertext input; from round 3 on when all blocks differ) run on the full state in place.
// xor_host (public input only; NULL: none) is XORed into the output.
// keys: the schedule (w or dk) of the direction.  key_idx_host: NULL, or (AES under many keys) the index of every block's
// schedule in the table at `keys`; it travels to the device with the plan, every round kernel offsets block b's round
// keys by key_idx[b] schedules, and the plan shares a bootstrap only among blocks of the same key.  Callers validate it.
int aes_blocks_dev(tac_ctx* ctx, AesDir dir, const uint64_t* keys, const int32_t* key_idx_host, int n_blocks, int rounds, int in_noise_sq,
                   const uint64_t* in_dev, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_dev) {
    const bool fwd = dir == AesDir::Forward, pub = in_dev == nullptr;
    std::vector<AesRoundPlan> plan;
    if (pub) {
        if (aes_public_plan_build(n_blocks, rounds, blocks_host, dir, plan, key_idx_host)) return fail(ctx, TAC_ERR_ARG, "n_blocks / rounds out of range, or NULL blocks");
    } else {
        if (n_blocks < 0 || rounds < 1 || rounds > 10) return fail(ctx, TAC_ERR_ARG, "n_blocks / rounds out of range");
        plan.assign(rounds, AesRoundPlan{16 * (int64_t)n_blocks, true});
    }
    if (n_blocks == 0) return TAC_OK;
    TRY(aes_noise_check(ctx, in_noise_sq, rounds));
    TRY(fwd ? ensure_aes_luts(ctx) : ensure_aes_inv_luts(ctx));
    const size_t L = (size_t)ctx->big() + 1, byte_words = 8 * L, blk = 16 * byte_words;
    const size_t npos = (size_t)n_blocks * 16, total = (size_t)n_blocks * blk;
    const size_t key_words = key_idx_host ? 11 * blk : 0;        // one schedule: 44 words = 11 round keys of a block's size
    // per direction: S-box LUTs S·{1,2,3} / S or InvS·{14,11,13,9} / InvS, round keys, (Inv)ShiftRows kernels
    const Lut& lut_mid = ctx->luts[fwd ? ctx->aes_lut24 : ctx->aes_lut_inv32];
    const Lut& lut_last = ctx->luts[fwd ? ctx->aes_lut8 : ctx->aes_lut_inv8];
    const uint64_t* k_first = fwd ? keys : keys + (size_t)10 * blk;
    const uint64_t* k_last = fwd ? keys + (size_t)10 * blk : keys;
    const auto mix_columns = fwd ? aes_mix_columns_kernel<true> : aes_mix_columns_kernel<false>;
    const auto final_round = fwd ? aes_final_round_kernel<true> : aes_final_round_kernel<false>;
    // one upload: public input's blocks and XOR bytes, the key index, then rep_pos / idx of every round that shares
    std::vector<size_t> off_rep(rounds, 0), off_idx(rounds, 0);
    std::vector<uint8_t> host;
    size_t max_rep = 0, bytes = pub ? 2 * npos : 0;
    const size_t off_kidx = bytes;
    if (key_idx_host) bytes += (size_t)n_blocks * 4;
    if (pub) {
        for (int r = 0; r < rounds; r++) {
            if (plan[r].identity) continue;
            off_rep[r] = bytes; bytes += (size_t)plan[r].boxes * 4;
            off_idx[r] = bytes; bytes += npos * 4;
            max_rep = std::max(max_rep, (size_t)plan[r].boxes);
        }
    }
    if (bytes) {
        host.assign(bytes, 0);
        if (pub) {
            std::memcpy(host.data(), blocks_host, npos);
            if (xor_host) std::memcpy(host.data() + npos, xor_host, npos);
            for (int r = 0; r < rounds; r++) {
                if (plan[r].identity) continue;
                std::memcpy(host.data() + off_rep[r], plan[r].rep_pos.data(), (size_t)plan[r].boxes * 4);
                std::memcpy(host.data() + off_idx[r], plan[r].idx.data(), npos * 4);
            }
        }
        if (key_idx_host) std::memcpy(host.data() + off_kidx, key_idx_host, (size_t)n_blocks * 4);
        TRY(ensure(ctx, ctx->ws_plan, bytes));
    }
    TRY(ensure(ctx, ctx->ws_state, total * 8));
    TRY(ensure(ctx, ctx->ws_muls, total * (fwd ? 3 : 4) * 8));
    if (pub) TRY(ensure(ctx, ctx->ws_rep, std::max<size_t>(1, max_rep) * byte_words * 8));
    // pageable source: the call returns once the bytes are staged, so `host` may go out of scope before the copy lands
    if (bytes) CU(cudaMemcpyAsync(ctx->ws_plan.p, host.data(), host.size(), cudaMemcpyHostToDevice, ctx->stream));
    const uint8_t* d_plan = ctx->ws_plan.as<uint8_t>();
    const int32_t* kidx = key_idx_host ? reinterpret_cast<const int32_t*>(d_plan + off_kidx) : nullptr;
    auto rep_pos = [&](int r) { return plan[r].identity ? nullptr : reinterpret_cast<const int32_t*>(d_plan + off_rep[r]); };
    auto idx = [&](int r) { return plan[r].identity ? nullptr : reinterpret_cast<const int32_t*>(d_plan + off_idx[r]); };
    uint64_t* state = ctx->ws_state.as<uint64_t>();
    uint64_t* muls = ctx->ws_muls.as<uint64_t>();
    uint64_t* rep = ctx->ws_rep.as<uint64_t>();
    const int g = grid1d(total, 256, ctx->sm_count);
    // S-box inputs of round rd (1-based) for its representatives → `in`
    auto sbox_inputs = [&](int rd, const uint64_t** in) -> int {
        const int r = rd - 1;
        const size_t n_words = (size_t)plan[r].boxes * byte_words;
        if (rd == 1 && !pub) {
            aes_add_round_key_kernel<<<g, 256, 0, ctx->stream>>>(in_dev, k_first, blk, total, state, kidx, key_words);          // :96-99
            TRY(post_launch(ctx, "aes_add_round_key_kernel"));
            *in = state;
        } else if (rd == 1) {
            uint64_t* dst = plan[r].identity ? state : rep;
            aes_public_round1_kernel<<<grid1d(n_words, 256, ctx->sm_count), 256, 0, ctx->stream>>>(k_first, d_plan, rep_pos(r), (int)L, n_words, dst, kidx, key_words);
            TRY(post_launch(ctx, "aes_public_round1_kernel"));
            *in = dst;
        } else if (plan[r].identity) {
            *in = state;
        } else {
            aes_gather_bytes_kernel<<<grid1d(n_words, 256, ctx->sm_count), 256, 0, ctx->stream>>>(state, rep_pos(r), (int)L, n_words, rep);
            TRY(post_launch(ctx, "aes_gather_bytes_kernel"));
            *in = rep;
        }
        return TAC_OK;
    };
    const uint64_t* in = nullptr;
    for (int rd = 1; rd < rounds; rd++) {
        TRY(sbox_inputs(rd, &in));
        TRY(wopbs_dev(ctx, lut_mid, (int)plan[rd - 1].boxes, in, muls));                                      // sub_bytes_with_gal_mul :27-48
        mix_columns<<<g, 256, 0, ctx->stream>>>(muls, keys + (size_t)(fwd ? rd : rounds - rd) * blk, (int)L, total, state, idx(rd - 1), kidx, key_words);
        TRY(post_launch(ctx, "aes_mix_columns_kernel"));
    }
    TRY(sbox_inputs(rounds, &in));
    TRY(wopbs_dev(ctx, lut_last, (int)plan[rounds - 1].boxes, in, muls));                                     // sub_bytes :51-58
    final_round<<<g, 256, 0, ctx->stream>>>(muls, k_last, (int)L, total, out_dev, idx(rounds - 1), xor_host ? d_plan + npos : nullptr, kidx, key_words);
    return post_launch(ctx, "aes_final_round_kernel");
}

size_t key_sched_bytes(const tac_ctx* ctx) { return (size_t)44 * 32 * (ctx->big() + 1) * 8; }

// The key set of a call, checked on the host before anything is enqueued: the single schedule, or (keyed) the key table
// with an index in [0, n) for each of the n_items blocks or records.  Decrypting needs a valid dk, which the single set may
// hold without its w (tac_aes_set_inv_key_schedule).
int keys_for(tac_ctx* ctx, AesDir dir, bool keyed, const int32_t* key_idx, int n_items, KeySet** out) {
    KeySet& ks = keyed ? ctx->table : ctx->single;
    const bool inv = dir == AesDir::Inverse;
    if (ks.n < 1 && (keyed || !inv)) return fail(ctx, TAC_ERR_STATE, ks.absent);
    if (inv && !ks.dk_valid) return fail(ctx, TAC_ERR_STATE, ks.no_dk);
    if (keyed && n_items > 0 && !key_idx) return fail(ctx, TAC_ERR_ARG, "NULL key index");
    for (int b = 0; keyed && b < n_items; b++)
        if (key_idx[b] < 0 || key_idx[b] >= ks.n)
            return fail(ctx, TAC_ERR_ARG, "key index " + std::to_string(key_idx[b]) + " of block " + std::to_string(b) + " outside [0, " +
                                              std::to_string(ks.n) + ")");
    *out = &ks;
    return TAC_OK;
}

// Every AES block entry point: the keys of `dir` (keys_for), then aes_blocks_dev over ciphertexts `in`, or, with `in`
// NULL, over public blocks_host.  host: `in` and `out` are host buffers, staged through ws_in and ws_out.
int aes_call(tac_ctx* ctx, AesDir dir, bool keyed, const int32_t* key_idx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in,
             const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out, bool host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    KeySet* ks;
    TRY(keys_for(ctx, dir, keyed, key_idx, n_blocks, &ks));
    const uint64_t* keys = (dir == AesDir::Forward ? ks->w : ks->dk).as<uint64_t>();
    if (!host) return aes_blocks_dev(ctx, dir, keys, key_idx, n_blocks, rounds, in_noise_sq, in, blocks_host, xor_host, out);
    if (n_blocks <= 0) return n_blocks == 0 ? TAC_OK : fail(ctx, TAC_ERR_ARG, "negative n_blocks");
    const size_t bytes = (size_t)n_blocks * 128 * (ctx->big() + 1) * 8;
    if (in) TRY(ensure(ctx, ctx->ws_in, bytes));
    TRY(ensure(ctx, ctx->ws_out, bytes));
    if (in) CU(cudaMemcpyAsync(ctx->ws_in.p, in, bytes, cudaMemcpyHostToDevice, ctx->stream));
    TRY(aes_blocks_dev(ctx, dir, keys, key_idx, n_blocks, rounds, in_noise_sq, in ? ctx->ws_in.as<uint64_t>() : nullptr, blocks_host, xor_host,
                       ctx->ws_out.as<uint64_t>()));
    CU(cudaMemcpyAsync(out, ctx->ws_out.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}

int key_schedule_noise_check(tac_ctx* ctx) {
    if (8 + 1 > ctx->p.max_noise_sq) return fail(ctx, TAC_ERR_NOISE, "NoiseTooBig: key schedule needs max_noise_level_squared >= 9");
    return TAC_OK;
}
int inv_key_schedule_noise_check(tac_ctx* ctx) {
    if (4 * 8 > ctx->p.max_noise_sq) return fail(ctx, TAC_ERR_NOISE, "NoiseTooBig: the inverse key schedule needs max_noise_level_squared >= 32");
    return TAC_OK;
}

// fhe_sbox_gal_mul_pbs::key_schedule (:134-164) with boot_word (:166-180) and sub_word (:182-191) on the device, for K keys
// at once: key_bits_host [K][128][kN+1] → ek [K][44 words][4][8][kN+1].  Each of the 40 steps bootstraps all K keys
// together: sub_word is one pass over 4K bytes, boot_word one over 32K bits, and aes_key_step_kernel forms the sums of all
// keys.  sub_word bootstraps w[i−1] as it is (the bootstrap of a byte does not depend on its neighbours in the batch) and
// the step kernel reads it rotated, so w[i−1] of every key is used where the previous boot_word left it, contiguous.
int key_expand(tac_ctx* ctx, int K, const uint64_t* key_bits_host, uint64_t* ek) {
    TRY(ensure_aes_luts(ctx));
    const size_t L = (size_t)ctx->big() + 1, byte = 8 * L, word = 4 * byte, sched = 44 * word;
    TRY(ensure(ctx, ctx->ws_state, (size_t)K * 3 * word * 8));
    uint64_t* prev = ctx->ws_state.as<uint64_t>();      // [K][word]: w[i−1] of every key
    uint64_t* sub = prev + (size_t)K * word;             // [K][word]: SubWord(w[i−1])
    uint64_t* acc = sub + (size_t)K * word;              // [K][word]: the sums boot_word bootstraps
    CU(cudaMemcpy2DAsync(ek, sched * 8, key_bits_host, 4 * word * 8, 4 * word * 8, (size_t)K, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpy2DAsync(prev, word * 8, key_bits_host + 3 * word, 4 * word * 8, word * 8, (size_t)K, cudaMemcpyHostToDevice, ctx->stream));
    // trivial(RC) constants: body += encode_bit(1) on the set bits of RC[i/4], byte 0 (:154; Byte::trivial data_model.rs:35-43).
    // All ten rows are uploaded once per context, so the 40 steps below enqueue without a host synchronisation.
    if (!ctx->rc_rows.p) {
        static const uint8_t RC[11] = {0x00, 0x01, 0x02, 0x04, 0x08, 0x10, 0x20, 0x40, 0x80, 0x1B, 0x36};
        std::vector<uint64_t> rows((size_t)10 * byte, 0ull);
        for (int r = 1; r <= 10; r++)
            for (int bit = 0; bit < 8; bit++)
                if (RC[r] & (0x80 >> bit)) rows[(size_t)(r - 1) * byte + (size_t)bit * L + (L - 1)] = tac_encode_bit(1);
        TRY(ensure(ctx, ctx->rc_rows, rows.size() * 8));
        CU(cudaMemcpy(ctx->rc_rows.p, rows.data(), rows.size() * 8, cudaMemcpyHostToDevice));
    }
    const size_t total = (size_t)K * word;
    for (int i = 4; i < 44; i++) {
        const bool rot = i % 4 == 0;
        if (rot) TRY(wopbs_dev(ctx, ctx->luts[ctx->aes_lut8], 4 * K, prev, sub));                                  // sub_word
        aes_key_step_kernel<<<grid1d(total, 256, ctx->sm_count), 256, 0, ctx->stream>>>(ek, sched, i, rot ? sub : nullptr,
                                                                                        ctx->rc_rows.as<uint64_t>() + (size_t)(i / 4 - 1) * byte, (int)L, total, acc);
        TRY(post_launch(ctx, "aes_key_step_kernel"));
        TRY(wopbs_dev(ctx, ctx->luts[ctx->aes_lut1], 32 * K, acc, prev));                                          // boot_word → bootstrap_assign
        CU(cudaMemcpy2DAsync(ek + (size_t)i * word, sched * 8, prev, word * 8, word * 8, (size_t)K, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    return TAC_OK;
}

// inverse key schedules of K schedules w [K][44 words] → dk, same layout: dk[0..3] = w[0..3], dk[40..43] = w[40..43],
// dk[4rd..4rd+3] = InvMixColumns(w[4rd..4rd+3]) for rd = 1..9.  One 8 → 32 circuit bootstrap (b·{14, 11, 13, 9}) of the
// 144K key bytes, the InvMixColumns sums (squared noise 32), then one 1-bit bootstrap per sum bit back to level 1 (as
// boot_word does in the forward key schedule).  Keys go in groups that fill one pipeline pass, which bounds the workspace.
int inv_key_expand(tac_ctx* ctx, int K, const uint64_t* w, uint64_t* dk) {
    TRY(ensure_aes_luts(ctx));
    TRY(ensure_aes_inv_luts(ctx));
    const size_t L = (size_t)ctx->big() + 1, byte = 8 * L, word = 4 * byte, sched = 44 * word, mid = 36 * word;
    const int n_key_bytes = 9 * 16;                          // round keys 1..9
    CU(cudaMemcpy2DAsync(dk, sched * 8, w, sched * 8, 4 * word * 8, (size_t)K, cudaMemcpyDeviceToDevice, ctx->stream));
    CU(cudaMemcpy2DAsync(dk + 40 * word, sched * 8, w + 40 * word, sched * 8, 4 * word * 8, (size_t)K, cudaMemcpyDeviceToDevice, ctx->stream));
    const int group = (int)std::max<size_t>(1, ctx->max_cts / (8 * (size_t)n_key_bytes));
    for (int k0 = 0; k0 < K; k0 += group) {
        const int nk = std::min(group, K - k0);
        TRY(ensure(ctx, ctx->ws_in, (size_t)nk * mid * 8));
        TRY(ensure(ctx, ctx->ws_muls, (size_t)nk * n_key_bytes * 32 * L * 8));
        TRY(ensure(ctx, ctx->ws_state, (size_t)nk * n_key_bytes * byte * 8));
        TRY(ensure(ctx, ctx->ws_out, (size_t)nk * mid * 8));
        uint64_t* keys = ctx->ws_in.as<uint64_t>();          // [nk][36 words]: w[4..39] of the group
        uint64_t* muls = ctx->ws_muls.as<uint64_t>();
        uint64_t* sums = ctx->ws_state.as<uint64_t>();
        uint64_t* bits = ctx->ws_out.as<uint64_t>();         // [nk][36 words]: dk[4..39] of the group
        CU(cudaMemcpy2DAsync(keys, mid * 8, w + (size_t)k0 * sched + 4 * word, sched * 8, mid * 8, (size_t)nk, cudaMemcpyDeviceToDevice, ctx->stream));
        TRY(wopbs_dev(ctx, ctx->luts[ctx->aes_lut_key32], nk * n_key_bytes, keys, muls));
        const size_t total = (size_t)nk * n_key_bytes * byte;
        aes_inv_mix_key_kernel<<<grid1d(total, 256, ctx->sm_count), 256, 0, ctx->stream>>>(muls, (int)L, total, sums);
        TRY(post_launch(ctx, "aes_inv_mix_key_kernel"));
        TRY(wopbs_dev(ctx, ctx->luts[ctx->aes_lut1], nk * n_key_bytes * 8, sums, bits));
        CU(cudaMemcpy2DAsync(dk + (size_t)k0 * sched + 4 * word, sched * 8, bits, mid * 8, mid * 8, (size_t)nk, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    return TAC_OK;
}

// ------------------------------------------------------------------------------------------------ key sets
// w about to change: the set is absent, its dk and GHASH table stale, until the new w is complete
void ks_reset(KeySet& ks) { ks.n = 0; ks.dk_valid = false; ks.gcm.valid = false; }

// room for K schedules in w or dk (contents not kept when it grows; the single set's never grows, as K is 1)
int ks_alloc(tac_ctx* ctx, DevBuf& b, int K) {
    return ensure(ctx, b, (size_t)K * key_sched_bytes(ctx), ("a key set of " + std::to_string(K) + " schedules").c_str());
}

// K schedules [K][44 words][4][8][kN+1] from the host into w; w_host NULL: the caller fills w (tac_aes_key_schedule_buffer)
int ks_set(tac_ctx* ctx, KeySet& ks, int K, const uint64_t* w_host) {
    ks_reset(ks);
    TRY(ks_alloc(ctx, ks.w, K));
    if (w_host) {
        CU(cudaMemcpyAsync(ks.w.p, w_host, (size_t)K * key_sched_bytes(ctx), cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    ks.n = K;
    return TAC_OK;
}

// w of K keys expanded on the device from their bits [K][128][kN+1] (key_expand); w_host: NULL or room for the schedules
int ks_expand(tac_ctx* ctx, KeySet& ks, int K, const uint64_t* key_bits_host, uint64_t* w_host) {
    TRY(key_schedule_noise_check(ctx));
    ks_reset(ks);
    TRY(ks_alloc(ctx, ks.w, K));
    TRY(key_expand(ctx, K, key_bits_host, ks.w.as<uint64_t>()));
    if (w_host) CU(cudaMemcpyAsync(w_host, ks.w.p, (size_t)K * key_sched_bytes(ctx), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ks.n = K;
    return TAC_OK;
}

// dk of every schedule of the set, derived on the device (inv_key_expand); dk_host: NULL or room for them
int ks_invert(tac_ctx* ctx, KeySet& ks, uint64_t* dk_host) {
    if (ks.n < 1) return fail(ctx, TAC_ERR_STATE, ks.absent);
    TRY(inv_key_schedule_noise_check(ctx));
    ks.dk_valid = false;
    TRY(ks_alloc(ctx, ks.dk, ks.n));
    TRY(inv_key_expand(ctx, ks.n, ks.w.as<uint64_t>(), ks.dk.as<uint64_t>()));
    if (dk_host) CU(cudaMemcpyAsync(dk_host, ks.dk.p, (size_t)ks.n * key_sched_bytes(ctx), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ks.dk_valid = true;
    return TAC_OK;
}

// K inverse schedules from the host into dk
int ks_set_inv(tac_ctx* ctx, KeySet& ks, int K, const uint64_t* dk_host) {
    ks.dk_valid = false;
    TRY(ks_alloc(ctx, ks.dk, K));
    CU(cudaMemcpyAsync(ks.dk.p, dk_host, (size_t)K * key_sched_bytes(ctx), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ks.dk_valid = true;
    return TAC_OK;
}

// ------------------------------------------------------------------------------------------------ AES-CCM
// LUTs of the tag check, registered on the first AES-CCM call: 8 → 1 "byte is zero", 8 → 1 "all 8 bits set", 2 → 1 "both set"
int ensure_ccm_luts(tac_ctx* ctx) {
    if (ctx->ccm_lut_ones2 >= 0) return TAC_OK;
    std::vector<uint64_t> f(256);
    for (int v = 0; v < 256; v++) f[v] = v == 0;
    TRY(register_aes_lut(ctx, 8, 1, f.data(), &ctx->ccm_lut_zero8));
    for (int v = 0; v < 256; v++) f[v] = v == 255;
    TRY(register_aes_lut(ctx, 8, 1, f.data(), &ctx->ccm_lut_ones8));
    const uint64_t both[4] = {0, 0, 0, 1};
    return register_aes_lut(ctx, 2, 1, both, &ctx->ccm_lut_ones2);
}

// The checks AES-CCM and AES-GCM make on the host before they enqueue anything: the records (shape: ccm_shape or
// gcm_shape, bad_record the error text after "<what> <index>: "), Σ p into *pt_bytes, a middle round over chain inputs of
// squared noise in_noise_sq, the keys (key_idx NULL: the single schedule) into *ks and the evaluation keys
template <class Shape>
int records_check(tac_ctx* ctx, int n_msgs, const int32_t* key_idx, const tac_ccm_msg* msgs, int (*shape)(const tac_ccm_msg&, Shape&),
                  const char* what, const char* bad_record, int in_noise_sq, KeySet** ks, uint64_t* pt_bytes) {
    if (n_msgs < 0) return fail(ctx, TAC_ERR_ARG, "negative n_msgs");
    if (n_msgs > 0 && !msgs) return fail(ctx, TAC_ERR_ARG, "NULL messages");
    *pt_bytes = 0;
    for (int c = 0; c < n_msgs; c++) {
        Shape s;
        if (shape(msgs[c], s)) return fail(ctx, TAC_ERR_ARG, std::string(what) + " " + std::to_string(c) + ": " + bad_record);
        *pt_bytes += s.p;
    }
    TRY(aes_noise_check(ctx, in_noise_sq, 10));
    TRY(keys_for(ctx, AesDir::Forward, key_idx != nullptr, key_idx, n_msgs, ks));
    if (!ctx->keys_valid) return fail(ctx, TAC_ERR_STATE, "evaluation keys not uploaded");
    return TAC_OK;
}
int outputs_check(tac_ctx* ctx, int n_msgs, uint64_t pt_bytes, const uint64_t* pt_out, const uint64_t* valid_out) {
    if ((n_msgs > 0 && !valid_out) || (pt_bytes > 0 && !pt_out)) return fail(ctx, TAC_ERR_ARG, "NULL output");
    return TAC_OK;
}

// every check of an AES-CCM call
int ccm_check(tac_ctx* ctx, int n_msgs, const int32_t* key_idx, const tac_ccm_msg* msgs, const uint64_t* pt_out, const uint64_t* valid_out,
              KeySet** ks, uint64_t* pt_bytes) {
    TRY(records_check(ctx, n_msgs, key_idx, msgs, ccm_shape, "AES-CCM message",
                      "need a nonce of 7..13 bytes, a tag length in {4, 6, …, 16}, data_len >= tag_len, a payload below 2^(8q) bytes and no "
                      "NULL pointer with a non-zero length",
                      18, ks, pt_bytes));           // a chain input X ⊕ P carries 18; a middle round 33
    return outputs_check(ctx, n_msgs, *pt_bytes, pt_out, valid_out);
}

// The validity bits of n tags from their differences D [n][16][8][L] (1 exactly when D is all zero): byte == 0 over 16·n
// bytes, all-8-set over 2·n groups, both-set over n pairs.  scratch: room for [n][16][L] + [n][2][L].
int tag_validity(tac_ctx* ctx, int n, const uint64_t* diff, uint64_t* scratch, uint64_t* valid_out) {
    const size_t L = (size_t)ctx->big() + 1;
    uint64_t* zero = scratch;                                // [n][16][L]: byte b of D is zero
    uint64_t* ones = zero + (size_t)n * 16 * L;              // [n][2][L]: bytes 0..7 / 8..15 all zero
    TRY(wopbs_dev(ctx, ctx->luts[ctx->ccm_lut_zero8], 16 * n, diff, zero));
    TRY(wopbs_dev(ctx, ctx->luts[ctx->ccm_lut_ones8], 2 * n, zero, ones));
    return wopbs_dev(ctx, ctx->luts[ctx->ccm_lut_ones2], n, ones, valid_out);
}

// AES-CCM transciphering of n messages (aes_ccm.h): one public-block AES call for B_0, A_0 and A_1..A_m of every message,
// the CBC-MAC chain in place on the B_0 rows (step s: aes_ccm_chain_input_kernel over the first a_s sorted messages, then
// one encrypted-block AES call of a_s blocks), then the tag check: aes_ccm_tag_diff_kernel forms D = MSB_t(X) ⊕ E(A_0) ⊕ U
// per message (caller order, 16 bytes, those >= t trivial zero) and three circuit bootstraps reduce it to one bit:
// byte == 0 over 16·n bytes, all-8-set over 2·n groups, both-set over n pairs.  Squared noise: chain inputs 18 (9 in a step
// of AAD blocks only), D 18, the zero tests 8, the 8-bit ANDs 8, the validity bit 2; the plaintext bits 9.  The
// descriptors of all steps, the ranks and the tag lengths travel to the device in one upload into ccm_desc, since
// aes_blocks_dev reuses ws_plan on every call.
int aes_ccm_dev(tac_ctx* ctx, int n_msgs, const int32_t* key_idx, const tac_ccm_msg* msgs, uint64_t* pt_out, uint64_t* valid_out) {
    KeySet* ks;
    uint64_t pt_bytes;
    TRY(ccm_check(ctx, n_msgs, key_idx, msgs, pt_out, valid_out, &ks, &pt_bytes));
    if (n_msgs == 0) return TAC_OK;
    TRY(ensure_ccm_luts(ctx));
    CcmPlan plan;
    ccm_plan_build(n_msgs, msgs, key_idx, plan);
    const int n = n_msgs;
    const uint64_t* keys = ks->w.as<uint64_t>();
    const size_t L = (size_t)ctx->big() + 1, byte_words = 8 * L, blk = 16 * byte_words;
    const int64_t rows = (int64_t)(plan.pub_blocks.size() / 16);
    TRY(ensure(ctx, ctx->ccm_pub, (size_t)rows * blk * 8));
    TRY(ensure(ctx, ctx->ccm_work, ((size_t)n * blk + (size_t)n * 18 * L) * 8));
    const size_t desc_bytes = plan.desc.size() * sizeof(CcmChainDesc);
    std::vector<uint8_t> host(desc_bytes + (size_t)n * 8);
    if (desc_bytes) std::memcpy(host.data(), plan.desc.data(), desc_bytes);
    std::memcpy(host.data() + desc_bytes, plan.rank.data(), (size_t)n * 4);
    std::memcpy(host.data() + desc_bytes + (size_t)n * 4, plan.tag_len.data(), (size_t)n * 4);
    TRY(ensure(ctx, ctx->ccm_desc, host.size()));
    // pageable source: the call returns once the bytes are staged
    CU(cudaMemcpyAsync(ctx->ccm_desc.p, host.data(), host.size(), cudaMemcpyHostToDevice, ctx->stream));
    const CcmChainDesc* d_desc = ctx->ccm_desc.as<CcmChainDesc>();
    const int32_t* d_rank = reinterpret_cast<const int32_t*>(ctx->ccm_desc.as<uint8_t>() + desc_bytes);
    const int32_t* d_tag_len = d_rank + n;
    uint64_t* pub = ctx->ccm_pub.as<uint64_t>();
    uint64_t* work = ctx->ccm_work.as<uint64_t>();

    TRY(aes_blocks_dev(ctx, AesDir::Forward, keys, key_idx ? plan.pub_kidx.data() : nullptr, (int)rows, 10, 0, nullptr, plan.pub_blocks.data(),
                       plan.pub_xor.data(), pub));
    size_t d0 = 0;
    for (size_t s = 0; s < plan.active.size(); s++) {
        const int a = plan.active[s];
        const size_t total = (size_t)a * blk;
        aes_ccm_chain_input_kernel<<<grid1d(total, 256, ctx->sm_count), 256, 0, ctx->stream>>>(pub, d_desc + d0, (int)L, total, work);
        TRY(post_launch(ctx, "aes_ccm_chain_input_kernel"));
        TRY(aes_blocks_dev(ctx, AesDir::Forward, keys, key_idx ? plan.kidx_sorted.data() : nullptr, a, 10, plan.adds_plaintext[s] ? 18 : 9, work,
                           nullptr, nullptr, pub));
        d0 += (size_t)a;
    }

    uint64_t* diff = work;                                   // [n][16][8][L], then tag_validity's scratch
    aes_ccm_tag_diff_kernel<<<grid1d((size_t)n * blk, 256, ctx->sm_count), 256, 0, ctx->stream>>>(pub, d_rank, d_tag_len, n, (int)L, (size_t)n * blk, diff);
    TRY(post_launch(ctx, "aes_ccm_tag_diff_kernel"));
    TRY(tag_validity(ctx, n, diff, diff + (size_t)n * blk, valid_out));
    // plaintext: the first p bytes of a message's A_1..A_m rows, contiguous, into its place in the caller's order
    for (int c = 0; c < n; c++)
        if (plan.shape[c].p)
            CU(cudaMemcpyAsync(pt_out + (size_t)plan.pt_off[c] * byte_words, pub + (size_t)plan.pt_row[c] * blk, plan.shape[c].p * byte_words * 8,
                               cudaMemcpyDeviceToDevice, ctx->stream));
    return TAC_OK;
}

// ------------------------------------------------------------------------------------------------ AES-GCM (aes_gcm.h)
// Runs a linear-layer plan: srcs are the plan's input sources 0..first_src−1; level k's group sums go through one 1-bit
// circuit bootstrap each into source first_src + k; the final gather-add writes row r to out row out_row[r] (or r).  All
// descriptors travel in one upload into lin_desc.
int lin_run(tac_ctx* ctx, const LinPlan& plan, const std::vector<const uint64_t*>& srcs, const std::vector<uint32_t>* out_row, uint64_t* out) {
    if ((int)(srcs.size() + plan.levels.size()) > kLinMaxSrc) return fail(ctx, TAC_ERR_ARG, "linear layer: too many sources");
    TRY(ensure_aes_luts(ctx));
    const size_t L = (size_t)ctx->big() + 1;
    std::vector<uint32_t> host;
    std::vector<size_t> off;
    auto put = [&](const std::vector<uint32_t>& v) { off.push_back(host.size()); host.insert(host.end(), v.begin(), v.end()); };
    size_t lvl_rows = 0, max_rows = 0;
    for (const LinSums& l : plan.levels) {
        put(l.row_ptr); put(l.terms);
        lvl_rows += l.rows(); max_rows = std::max(max_rows, l.rows());
    }
    put(plan.final.row_ptr); put(plan.final.terms);
    if (out_row) put(*out_row);
    const size_t cbit_off = host.size() * 4;
    const size_t nrows = plan.final.rows();
    if (nrows == 0) return TAC_OK;
    std::vector<uint8_t> bytes(cbit_off + nrows);
    std::memcpy(bytes.data(), host.data(), cbit_off);
    std::memcpy(bytes.data() + cbit_off, plan.final.cbit.data(), nrows);
    TRY(ensure(ctx, ctx->lin_desc, bytes.size()));
    TRY(ensure(ctx, ctx->lin_sum, std::max<size_t>(1, max_rows) * L * 8));
    TRY(ensure(ctx, ctx->lin_lvl, std::max<size_t>(1, lvl_rows) * L * 8));
    // pageable source: the call returns once the bytes are staged
    CU(cudaMemcpyAsync(ctx->lin_desc.p, bytes.data(), bytes.size(), cudaMemcpyHostToDevice, ctx->stream));
    const uint32_t* d = ctx->lin_desc.as<uint32_t>();
    LinSrcs s{};
    for (size_t i = 0; i < srcs.size(); i++) s.p[i] = srcs[i];
    uint64_t* lvl = ctx->lin_lvl.as<uint64_t>();
    size_t k = 0;
    for (size_t i = 0; i < plan.levels.size(); i++, k += 2) {
        const size_t rows = plan.levels[i].rows();
        lwe_gather_add_kernel<<<grid1d(rows * L, 256, ctx->sm_count), 256, 0, ctx->stream>>>(s, d + off[k], d + off[k + 1], nullptr, nullptr, (int)L,
                                                                                            rows * L, ctx->lin_sum.as<uint64_t>());
        TRY(post_launch(ctx, "lwe_gather_add_kernel"));
        TRY(wopbs_dev(ctx, ctx->luts[ctx->aes_lut1], (int)rows, ctx->lin_sum.as<uint64_t>(), lvl));            // refresh to squared noise 1
        s.p[srcs.size() + i] = lvl;
        lvl += rows * L;
    }
    lwe_gather_add_kernel<<<grid1d(nrows * L, 256, ctx->sm_count), 256, 0, ctx->stream>>>(
        s, d + off[k], d + off[k + 1], ctx->lin_desc.as<uint8_t>() + cbit_off, out_row ? d + off[k + 2] : nullptr, (int)L, nrows * L, out);
    return post_launch(ctx, "lwe_gather_add_kernel");
}

// copies rows: out row r (or out_row[r]) = row rows[r] of src
int gather_rows(tac_ctx* ctx, const uint64_t* src, const std::vector<uint32_t>& rows, const std::vector<uint32_t>* out_row, uint64_t* out) {
    LinPlan plan;
    for (uint32_t r : rows) {
        plan.final.terms.push_back(lin_id(0, r));
        plan.final.row_ptr.push_back((uint32_t)plan.final.terms.size());
    }
    plan.final.cbit.assign(rows.size(), 0);
    return lin_run(ctx, plan, {src}, out_row, out);
}

int ensure_gf_lut(tac_ctx* ctx) {
    if (ctx->gf_lut_mul >= 0) return TAC_OK;
    std::vector<uint64_t> f(256);
    for (int v = 0; v < 256; v++) f[v] = gf128_box_fn(v);
    return register_aes_lut(ctx, 8, 7, f.data(), &ctx->gf_lut_mul);
}

// n encrypted GF(2^128) products out = a · b, operands [n][128][kN+1] at squared noise <= max_noise_level_squared, output
// bits at squared noise 1 (out row p·128 + j, or out_row[p·128 + j]).  Per pass of np products: the GGSW stage over the
// 128·np bits of a and of b, 1024·np boxes of vertical packing over GGSWs picked by index (box (i, j) of product p: nibble i
// of a, nibble j of b), then the linear layer (sums, reduction mod x^128 + x^7 + x^2 + x + 1, refreshes).
int gf128_mul_dev(tac_ctx* ctx, int n, const uint64_t* a, const uint64_t* b, uint64_t* out, const std::vector<uint32_t>* out_row = nullptr) {
    if (n <= 0) return TAC_OK;
    if (!ctx->keys_valid) return fail(ctx, TAC_ERR_STATE, "evaluation keys not uploaded");
    TRY(ensure_gf_lut(ctx));
    const TacParams& p = ctx->p;
    const size_t L = (size_t)ctx->big() + 1, ggsw_cplx = (size_t)p.cbs_l * ctx->G() * ctx->G() * (p.N / 2);
    // products per pass: their GGSWs fill one pipeline pass, and their boxes one launch (grid.y <= 65535)
    const int np_max = (int)std::max<size_t>(1, std::min<size_t>(ctx->max_cts / 256, 65535 / 1024));
    if (ctx->gf_idx_np != np_max) {
        // GGSWs of a pass: [a bits of its products][b bits], np_max·128 each
        std::vector<int32_t> idx((size_t)np_max * 1024 * 8);
        for (int q = 0; q < np_max; q++)
            for (int i = 0; i < 32; i++)
                for (int j = 0; j < 32; j++)
                    for (int k = 0; k < 4; k++) {
                        int32_t* e = &idx[(((size_t)q * 1024) + i * 32 + j) * 8];
                        e[k] = q * 128 + 4 * i + k;
                        e[4 + k] = np_max * 128 + q * 128 + 4 * j + k;
                    }
        TRY(ensure(ctx, ctx->gf_idx, idx.size() * 4));
        CU(cudaMemcpy(ctx->gf_idx.p, idx.data(), idx.size() * 4, cudaMemcpyHostToDevice));
        ctx->gf_idx_np = np_max;
    }
    const Lut& lut = ctx->luts[ctx->gf_lut_mul];
    for (int p0 = 0; p0 < n; p0 += np_max) {
        const int np = std::min(np_max, n - p0);
        TRY(ensure(ctx, ctx->ws_ggswf, (size_t)2 * np_max * 128 * ggsw_cplx * sizeof(cplx)));
        TRY(ensure(ctx, ctx->gf_box, (size_t)np * 1024 * 7 * L * 8));
        cplx* gf = ctx->ws_ggswf.as<cplx>();
        TRY(ggsw_stage(ctx, a + (size_t)p0 * 128 * L, 128 * np, gf));
        TRY(stage_event(ctx, 5));
        TRY(ggsw_stage(ctx, b + (size_t)p0 * 128 * L, 128 * np, gf + (size_t)np_max * 128 * ggsw_cplx));
        TRY(check_launch(ctx, ctx->ops->vp_gather(klaunch(ctx), p.cbs_l, gf, ctx->gf_idx.as<int32_t>(), 1024 * np, 8, lut.dev, lut.len, 7, p.cbs_b,
                                                  ctx->gf_box.as<uint64_t>()), "vp_gather_kernel"));
        TRY(stage_event(ctx, 5));
        std::vector<LinRow> rows;
        gf128_rows(np, rows);
        LinPlan plan;
        if (lin_plan_build(rows, p.max_noise_sq, 1, 1, plan)) return fail(ctx, TAC_ERR_NOISE, "GF(2^128) product: the sums do not fit max_noise_level_squared");
        std::vector<uint32_t> orow;
        if (out_row) orow.assign(out_row->begin() + (size_t)p0 * 128, out_row->begin() + (size_t)(p0 + np) * 128);
        TRY(lin_run(ctx, plan, {ctx->gf_box.as<uint64_t>()}, out_row ? &orow : nullptr, out_row ? out : out + (size_t)p0 * 128 * L));
    }
    return TAC_OK;
}

int gf_noise_check(tac_ctx* ctx) {
    // the box outputs of one unreduced coefficient are summed 8 at a time (squared noise 8 each)
    if (8 * 8 > ctx->p.max_noise_sq) return fail(ctx, TAC_ERR_NOISE, "NoiseTooBig: the GF(2^128) product needs max_noise_level_squared >= 64");
    return TAC_OK;
}

// H = E_K(0) of K keys (key_idx NULL: the single schedule) and its powers H^1..H^w into table [K][w][128][L].  H comes
// out of one public-block call and a refresh.  Pass j computes H^(2^j+1) … H^(2^(j+1)): even powers square an earlier
// power (a linear map, at most 5 terms per bit, then a refresh), odd ones are the products H^(2^j) · H^(e − 2^j) of all
// keys in one gf128_mul_dev call.
int gcm_hash_key_build(tac_ctx* ctx, const uint64_t* keys, const int32_t* key_idx, int K, int w, uint64_t* table) {
    TRY(ensure_aes_luts(ctx));
    const size_t L = (size_t)ctx->big() + 1;
    auto row = [&](int k, int e, int bit) { return (uint32_t)(((size_t)k * w + (e - 1)) * 128 + bit); };
    TRY(ensure(ctx, ctx->gcm_pub, (size_t)K * 128 * L * 8));
    std::vector<uint8_t> zero((size_t)K * 16, 0);
    TRY(aes_blocks_dev(ctx, AesDir::Forward, keys, key_idx, K, 10, 0, nullptr, zero.data(), nullptr, ctx->gcm_pub.as<uint64_t>()));
    {
        std::vector<LinRow> rows((size_t)K * 128);
        std::vector<uint32_t> orow(rows.size());
        for (int k = 0; k < K; k++)
            for (int j = 0; j < 128; j++) {
                rows[(size_t)k * 128 + j].terms.push_back(LinTerm{lin_id(0, (size_t)k * 128 + j), 9, 0});
                orow[(size_t)k * 128 + j] = row(k, 1, j);
            }
        LinPlan plan;
        TRY(lin_plan_build(rows, ctx->p.max_noise_sq, 1, 1, plan) ? fail(ctx, TAC_ERR_NOISE, "GHASH key: refresh") : TAC_OK);
        TRY(lin_run(ctx, plan, {ctx->gcm_pub.as<uint64_t>()}, &orow, table));
    }
    std::vector<std::vector<int>> sq(128);            // bit r of y^2: XOR of y's bits sq[r]
    for (int l = 0; l < 128; l++)
        for (int r : gf128_fold(2 * l)) sq[r].push_back(l);
    for (int lo = 1; lo < w; lo *= 2) {
        std::vector<LinRow> rows;
        std::vector<uint32_t> orow, a_rows, b_rows, prow;
        for (int k = 0; k < K; k++)
            for (int e = lo + 1; e <= 2 * lo; e++)
                for (int j = 0; j < 128; j++) {
                    if (e % 2 == 0) {
                        LinRow r;
                        for (int l : sq[j]) r.terms.push_back(LinTerm{lin_id(0, row(k, e / 2, l)), 1, 0});
                        rows.push_back(r);
                        orow.push_back(row(k, e, j));
                    } else {
                        a_rows.push_back(row(k, lo, j));
                        b_rows.push_back(row(k, e - lo, j));
                        prow.push_back(row(k, e, j));
                    }
                }
        LinPlan plan;
        TRY(lin_plan_build(rows, ctx->p.max_noise_sq, 1, 1, plan) ? fail(ctx, TAC_ERR_NOISE, "GHASH key: squares") : TAC_OK);
        TRY(lin_run(ctx, plan, {table}, &orow, table));
        const int nprod = (int)(a_rows.size() / 128);
        if (nprod) {
            TRY(ensure(ctx, ctx->gf_ops, (size_t)2 * nprod * 128 * L * 8));
            uint64_t* ops = ctx->gf_ops.as<uint64_t>();
            TRY(gather_rows(ctx, table, a_rows, nullptr, ops));
            TRY(gather_rows(ctx, table, b_rows, nullptr, ops + (size_t)nprod * 128 * L));
            TRY(gf128_mul_dev(ctx, nprod, ops, ops + (size_t)nprod * 128 * L, table, &prow));
        }
    }
    return TAC_OK;
}

// the GHASH key table of the single schedule or (keyed) of every key table entry, built for `depth` powers
int gcm_hash_key(tac_ctx* ctx, bool keyed, int depth, uint64_t* out_host) {
    if (depth < 1 || depth > 1024 || (depth & (depth - 1))) return fail(ctx, TAC_ERR_ARG, "GHASH key depth must be a power of two in [1, 1024]");
    if (!ctx->keys_valid) return fail(ctx, TAC_ERR_STATE, "evaluation keys not uploaded");
    KeySet* ks;
    TRY(keys_for(ctx, AesDir::Forward, keyed, nullptr, 0, &ks));
    TRY(aes_noise_check(ctx, 0, 10));
    if (depth > 1) TRY(gf_noise_check(ctx));
    GcmTable& t = ks->gcm;
    const int K = ks->n;
    const size_t L = (size_t)ctx->big() + 1, bytes = (size_t)K * depth * 128 * L * 8;
    t.valid = false;
    TRY(ensure(ctx, t.buf, bytes, ("a GHASH key table of " + std::to_string(K) + " keys × " + std::to_string(depth) + " powers").c_str()));
    std::vector<int32_t> kidx(K);
    for (int k = 0; k < K; k++) kidx[k] = k;
    TRY(gcm_hash_key_build(ctx, ks->w.as<uint64_t>(), keyed ? kidx.data() : nullptr, K, depth, t.buf.as<uint64_t>()));
    if (out_host) CU(cudaMemcpyAsync(out_host, t.buf.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    t.depth = depth; t.valid = true;
    return TAC_OK;
}

// every check of an AES-GCM call
int gcm_check(tac_ctx* ctx, int n_msgs, const int32_t* key_idx, const tac_ccm_msg* msgs, const uint64_t* pt_out, const uint64_t* valid_out,
              KeySet** ks, uint64_t* pt_bytes) {
    TRY(records_check(ctx, n_msgs, key_idx, msgs, gcm_shape, "AES-GCM record",
                      "need a 12-byte IV, a tag length in {4, 8, 12, 13, 14, 15, 16}, data_len >= tag_len, a payload of at most 2^36 − 32 "
                      "bytes, AAD below 2^61 bytes and no NULL pointer with a non-zero length",
                      0, ks, pt_bytes));
    if (!(*ks)->gcm.valid) return fail(ctx, TAC_ERR_STATE, (*ks)->no_gcm);
    return outputs_check(ctx, n_msgs, *pt_bytes, pt_out, valid_out);
}

// AES-GCM transciphering of n records.  1. One public-block call over J0 of every record (rows 0..n−1, sorted order) and
// inc32^i(J0), i = 1..m, with XOR bytes C (the plaintext rows).  2. GHASH in Horner form over chunks of w blocks, the first
// chunk the short one: Y_c = Y_(c−1) · H^w ⊕ Σ_(i in chunk c) X_i · H^(pos); records are sorted by chunk count, descending,
// so step c runs over a prefix of them: one batched product (from step 1 on), then one linear layer whose rows are Y_c
// (squared noise <= max) or, in a record's last step, the tag difference D = MSB_t(E(J0) ⊕ S) ⊕ T (bytes >= t trivial
// zero).  3. CCM's three zero-test passes reduce D to the validity bit.
int aes_gcm_dev(tac_ctx* ctx, int n_msgs, const int32_t* key_idx, const tac_ccm_msg* msgs, uint64_t* pt_out, uint64_t* valid_out) {
    KeySet* ks;
    uint64_t pt_bytes;
    TRY(gcm_check(ctx, n_msgs, key_idx, msgs, pt_out, valid_out, &ks, &pt_bytes));
    if (n_msgs == 0) return TAC_OK;
    const GcmTable& tab = ks->gcm;
    const int n = n_msgs, w = tab.depth, maxn = ctx->p.max_noise_sq;
    std::vector<GcmShape> sh(n);
    std::vector<int64_t> chunks(n);
    for (int c = 0; c < n; c++) {
        gcm_shape(msgs[c], sh[c]);
        chunks[c] = (sh[c].M + w - 1) / w;
    }
    if (chunks.size() && *std::max_element(chunks.begin(), chunks.end()) > 1) TRY(gf_noise_check(ctx));
    TRY(ensure_ccm_luts(ctx));
    std::vector<int32_t> order(n), rank(n);
    for (int c = 0; c < n; c++) order[c] = c;
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return chunks[a] > chunks[b]; });
    for (int r = 0; r < n; r++) rank[order[r]] = r;
    const size_t L = (size_t)ctx->big() + 1, byte_words = 8 * L, blk = 16 * byte_words;
    // the public call: [J0 rows][counter rows of every record], sorted order
    int64_t rows = n;
    std::vector<int64_t> pt_row(n);
    for (int r = 0; r < n; r++) { pt_row[order[r]] = rows; rows += sh[order[r]].m; }
    std::vector<uint8_t> blocks((size_t)rows * 16), xr((size_t)rows * 16, 0);
    std::vector<int32_t> kidx(key_idx ? rows : 0);
    for (int r = 0; r < n; r++) {
        const int c = order[r];
        gcm_ctr_block(msgs[c], 1, &blocks[(size_t)r * 16]);
        for (int64_t i = 1; i <= sh[c].m; i++) gcm_ctr_block(msgs[c], (uint32_t)(1 + i), &blocks[(size_t)(pt_row[c] + i - 1) * 16]);
        if (sh[c].p) std::memcpy(&xr[(size_t)pt_row[c] * 16], msgs[c].data, (size_t)sh[c].p);
        if (key_idx) {
            kidx[r] = key_idx[c];
            for (int64_t i = 0; i < sh[c].m; i++) kidx[(size_t)(pt_row[c] + i)] = key_idx[c];
        }
    }
    TRY(ensure(ctx, ctx->gcm_pub, (size_t)rows * blk * 8));
    TRY(ensure(ctx, ctx->gcm_dy, (size_t)2 * n * blk * 8));
    TRY(ensure(ctx, ctx->ccm_work, (size_t)n * 18 * L * 8));
    uint64_t* pub = ctx->gcm_pub.as<uint64_t>();
    uint64_t* dy = ctx->gcm_dy.as<uint64_t>();             // [n][128]: D in caller order, then [n][128]: Y in sorted order
    TRY(aes_blocks_dev(ctx, AesDir::Forward, ks->w.as<uint64_t>(), key_idx ? kidx.data() : nullptr, (int)rows, 10, 0, nullptr, blocks.data(), xr.data(),
                       pub));
    // GHASH steps
    std::vector<std::vector<uint8_t>> X(n);
    for (int c = 0; c < n; c++) {
        X[c].resize((size_t)sh[c].M * 16);
        gcm_ghash_blocks(msgs[c], sh[c], X[c].data());
    }
    const int64_t steps = chunks[order[0]];
    for (int64_t s = 0; s < steps; s++) {
        int a = 0;
        while (a < n && chunks[order[a]] > s) a++;
        if (s > 0) {
            std::vector<uint32_t> hw((size_t)a * 128);
            for (int r = 0; r < a; r++)
                for (int j = 0; j < 128; j++)
                    hw[(size_t)r * 128 + j] = (uint32_t)(((size_t)(key_idx ? key_idx[order[r]] : 0) * w + (w - 1)) * 128 + j);
            TRY(ensure(ctx, ctx->gf_ops, (size_t)a * 128 * L * 8));
            TRY(ensure(ctx, ctx->gf_prod, (size_t)a * 128 * L * 8));
            TRY(gather_rows(ctx, tab.buf.as<uint64_t>(), hw, nullptr, ctx->gf_ops.as<uint64_t>()));
            TRY(gf128_mul_dev(ctx, a, dy + (size_t)n * 128 * L, ctx->gf_ops.as<uint64_t>(), ctx->gf_prod.as<uint64_t>()));
        }
        std::vector<LinRow> lrows((size_t)a * 128);
        std::vector<uint32_t> orow((size_t)a * 128);
        for (int r = 0; r < a; r++) {
            const int c = order[r];
            const int64_t first = sh[c].M - (chunks[c] - 1) * w;                       // blocks in chunk 0
            const int64_t b0 = s == 0 ? 0 : first + (s - 1) * w, b1 = s == 0 ? first : first + s * w;
            std::vector<int> exps;
            for (int64_t i = b0; i < b1; i++) exps.push_back((int)(b1 - i));
            const uint64_t base = (uint64_t)(key_idx ? key_idx[c] : 0) * w * 128;
            LinRow* rr = &lrows[(size_t)r * 128];
            ghash_terms(&X[c][(size_t)b0 * 16], (int)(b1 - b0), exps.data(), 0, base, (int64_t)r << 20, rr);
            const int64_t own = ((int64_t)r << 20) | 0xFFFFF;
            for (int j = 0; j < 128; j++)
                if (s > 0) rr[j].terms.push_back(LinTerm{lin_id(1, (size_t)r * 128 + j), 1, own});
            const bool last = s == chunks[c] - 1;
            for (int j = 0; j < 128; j++) {
                orow[(size_t)r * 128 + j] = (uint32_t)(last ? (size_t)c * 128 + j : (size_t)(n + r) * 128 + j);
                if (!last) continue;
                if (j >= 8 * sh[c].t) { rr[j] = LinRow{}; continue; }
                rr[j].terms.push_back(LinTerm{lin_id(2, (size_t)r * 128 + j), 9, own - 1});          // E(J0)
                rr[j].cbit = (msgs[c].data[sh[c].p + j / 8] >> (7 - j % 8)) & 1;                    // T
            }
        }
        LinPlan plan;
        if (lin_plan_build(lrows, maxn, maxn, 3, plan)) return fail(ctx, TAC_ERR_NOISE, "GHASH: the sums do not fit max_noise_level_squared");
        TRY(lin_run(ctx, plan, {tab.buf.as<uint64_t>(), ctx->gf_prod.p ? ctx->gf_prod.as<uint64_t>() : pub, pub}, &orow, dy));
    }
    TRY(tag_validity(ctx, n, dy, ctx->ccm_work.as<uint64_t>(), valid_out));
    // plaintext: the first p bytes of a record's counter rows, contiguous, into its place in the caller's order
    uint64_t off = 0;
    for (int c = 0; c < n; c++) {
        if (sh[c].p)
            CU(cudaMemcpyAsync(pt_out + off * byte_words, pub + (size_t)pt_row[c] * blk, sh[c].p * byte_words * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        off += sh[c].p;
    }
    return TAC_OK;
}

// host form of tac_aes_{ccm,gcm}_transcipher: check (ccm_check / gcm_check) against the host outputs, dev
// (aes_ccm_dev / aes_gcm_dev) into ws_out, then the plaintext and validity bits back
using RecordCheck = int (*)(tac_ctx*, int, const int32_t*, const tac_ccm_msg*, const uint64_t*, const uint64_t*, KeySet**, uint64_t*);
using RecordDev = int (*)(tac_ctx*, int, const int32_t*, const tac_ccm_msg*, uint64_t*, uint64_t*);
int records_host(tac_ctx* ctx, RecordCheck check, RecordDev dev, int n_msgs, const int32_t* key_idx, const tac_ccm_msg* msgs, uint64_t* pt_out_host,
                 uint64_t* valid_out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    KeySet* ks;
    uint64_t pt_bytes;
    TRY(check(ctx, n_msgs, key_idx, msgs, pt_out_host, valid_out_host, &ks, &pt_bytes));
    if (n_msgs == 0) return TAC_OK;
    const size_t L = (size_t)ctx->big() + 1, pt_words = (size_t)pt_bytes * 8 * L, valid_words = (size_t)n_msgs * L;
    TRY(ensure(ctx, ctx->ws_out, (pt_words + valid_words) * 8));
    uint64_t* pt = ctx->ws_out.as<uint64_t>();
    TRY(dev(ctx, n_msgs, key_idx, msgs, pt, pt + pt_words));
    if (pt_words) CU(cudaMemcpyAsync(pt_out_host, pt, pt_words * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(valid_out_host, pt + pt_words, valid_words * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}

}  // namespace

// =================================================================================================== C ABI
extern "C" {

const char* tac_last_error(tac_ctx*) { return g_error.c_str(); }

tac_ctx* tac_ctx_create(const tac_params* pp, int device) {
    tac_ctx* ctx = nullptr;     // for the CU macro's fail(ctx, …) before allocation
    auto bail = [&](const std::string& m) -> tac_ctx* { g_error = m; delete ctx; return nullptr; };
    const TacParams p = *reinterpret_cast<const TacParams*>(pp);
    if (!supported_shape(p)) return bail("unsupported (polynomial_size, glwe_dimension): kernels are instantiated for (512,4) and (1024,2)");
    {   // everything else the kernels assume about a caller-supplied parameter block (the four presets satisfy all of it)
        const std::string why = unsupported_params(p);
        if (!why.empty()) return bail("unsupported parameter set: " + why);
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return bail(std::string("no CUDA device: ") + cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return bail("device index out of range");
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail(std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e));
    if (prop.major != 10) return bail("this library is built for sm_100a (B200) only; found sm_" + std::to_string(prop.major) + std::to_string(prop.minor));
    ctx = new tac_ctx();
    ctx->p = p; ctx->device = device; ctx->sm_count = prop.multiProcessorCount;
    ctx->ops = (p.N == 512) ? shape_ops_n512_k4() : shape_ops_n1024_k2();
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(std::string("cudaStreamCreate: ") + cudaGetErrorString(e));
    ctx->own_stream = true;
    if (const char* s = getenv("TAC_MAX_CTS")) { const long v = atol(s); if (v > 0) ctx->max_cts = (size_t)v; }
    if (const char* s = getenv("TAC_FIX_CAP")) { const long v = atol(s); if (v >= 0 && (uint32_t)v <= kFixCap) ctx->fix_cap = (uint32_t)v; }
    // combined twist/twiddle table in extended precision
    std::vector<cplx> w(tab_len(p.N));
    build_wT(p.N, w.data());
    if (ensure(ctx, ctx->wT, w.size() * sizeof(cplx))) return bail("cudaMalloc(tables) failed");
    cudaMemcpy(ctx->wT.p, w.data(), w.size() * sizeof(cplx), cudaMemcpyHostToDevice);
    return ctx;
}

void tac_ctx_destroy(tac_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (auto& l : ctx->luts) cudaFree(l.dev);
    for (auto& r : ctx->prof_pool) for (auto& ev : r.ev) cudaEventDestroy(ev);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;             // the DevBufs free the rest
}

int tac_ctx_set_stream(tac_ctx* ctx, void* s) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (ctx->own_stream && ctx->stream) { CU(cudaStreamSynchronize(ctx->stream)); CU(cudaStreamDestroy(ctx->stream)); }
    ctx->stream = reinterpret_cast<cudaStream_t>(s);
    ctx->own_stream = false;
    return TAC_OK;
}
int tac_ctx_sync(tac_ctx* ctx) { LOCK(ctx); CU(cudaSetDevice(ctx->device)); CU(cudaStreamSynchronize(ctx->stream)); return TAC_OK; }
int tac_ctx_sm_count(tac_ctx* ctx) { return ctx->sm_count; }
int tac_ctx_set_profiling(tac_ctx* ctx, int on) { LOCK(ctx); ctx->profiling = on != 0; return TAC_OK; }
int tac_ctx_stage_times(tac_ctx* ctx, float out_ms[5], int* n_passes) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    for (int s = 0; s < ST_COUNT; s++) out_ms[s] = 0.f;
    for (size_t r = 0; r < ctx->prof_used; r++)
        for (int s = 0; s < ST_COUNT; s++) {
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, ctx->prof_pool[r].ev[s], ctx->prof_pool[r].ev[s + 1]));
            out_ms[s] += ms;
        }
    if (n_passes) *n_passes = (int)ctx->prof_used;
    ctx->prof_used = 0;
    return TAC_OK;
}
// FP64 FMA pipe peak of this GPU (the roofline denominator of the PBS kernel; not in MEASURED_PEAKS.json)
int tac_bench_fp64_peak(tac_ctx* ctx, double* tflops) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    TRY(ensure(ctx, ctx->ws_misc, 1 << 20));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    const int iters = 4096, blocks = ctx->sm_count * 8, threads = 256;
    double best = 0.0;
    for (int rep = 0; rep < 4; rep++) {
        CU(cudaEventRecord(e0, ctx->stream));
        dfma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->ws_misc.as<double>(), iters, 1.0000001);
        CU(cudaEventRecord(e1, ctx->stream));
        CU(cudaEventSynchronize(e1));
        TRY(post_launch(ctx, "dfma_peak_kernel"));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 16.0 * (double)iters * blocks * threads;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *tflops = best;
    return TAC_OK;
}
uint64_t tac_ctx_launch_count(tac_ctx* ctx) { LOCK(ctx); return ctx->launches; }

int tac_ctx_alloc_keys(tac_ctx* ctx) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (ctx->keys_allocated) return TAC_OK;
    const int Kd = (ctx->big() + 1) * ctx->p.pfks_l, nkb = (Kd + UG_KB - 1) / UG_KB;
    const int W = ctx->G() * ctx->p.N, tiles = (W + UG_NT - 1) / UG_NT;
    const int Kd_ks = ctx->big() * ctx->p.ks_l, nkb_ks = (Kd_ks + UG_KB - 1) / UG_KB, tiles_ks = (ctx->p.n + 1 + UG_NT - 1) / UG_NT;
    TRY(ensure(ctx, ctx->bsk_f, ctx->bsk_cplx() * sizeof(cplx), "the bootstrapping key"));
    TRY(ensure(ctx, ctx->ksk, ctx->ksk_words() * 8, "the keyswitching key"));
    TRY(ensure(ctx, ctx->pfpksk, ctx->pfpksk_words() * 8, "the private functional packing keyswitching keys"));
    TRY(ensure(ctx, ctx->ks_corr, (size_t)(ctx->p.n + 1) * 8));
    TRY(ensure(ctx, ctx->pfks_corr, (size_t)ctx->G() * ctx->G() * ctx->p.N * 8));
    TRY(ensure(ctx, ctx->pfks_planes, (size_t)ctx->G() * tiles * nkb * UG_B_BYTES));
    TRY(ensure(ctx, ctx->pfks_fix, 8 + (size_t)kFixCap * 8));
    TRY(ensure(ctx, ctx->ks_planes, (size_t)tiles_ks * nkb_ks * UG_B_BYTES));
    ctx->keys_allocated = true;
    return TAC_OK;
}
int tac_ctx_key_buffer(tac_ctx* ctx, int which, void** dev_ptr, size_t* bytes) {
    LOCK(ctx);
    if (!ctx->keys_allocated) return fail(ctx, TAC_ERR_STATE, "key buffers not allocated");
    switch (which) {
        case 0: *dev_ptr = ctx->bsk_f.p; *bytes = ctx->bsk_cplx() * sizeof(cplx); return TAC_OK;
        case 1: *dev_ptr = ctx->ksk.p; *bytes = ctx->ksk_words() * 8; return TAC_OK;
        case 2: *dev_ptr = ctx->pfpksk.p; *bytes = ctx->pfpksk_words() * 8; return TAC_OK;
        default: return fail(ctx, TAC_ERR_ARG, "key buffer index");
    }
}
// correction rows: corr[col] = (B/2)·Σ_k key[k][col], obtained by running the GEMM on constant digits B/2
int tac_ctx_keys_ready(tac_ctx* ctx) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!ctx->keys_allocated) return fail(ctx, TAC_ERR_STATE, "key buffers not allocated");
    const TacParams& p = ctx->p;
    const int Kd_ks = ctx->big() * p.ks_l, Kd_pf = (ctx->big() + 1) * p.pfks_l;
    const int Kmax = std::max(Kd_ks, Kd_pf);
    TRY(ensure(ctx, ctx->ws_misc, (size_t)Kmax * 4));
    std::vector<uint32_t> h(Kmax);
    std::fill(h.begin(), h.end(), 1u << (p.ks_b - 1));
    CU(cudaMemcpyAsync(ctx->ws_misc.p, h.data(), (size_t)Kd_ks * 4, cudaMemcpyHostToDevice, ctx->stream));
    TRY(gemm(ctx, ctx->ws_misc.as<uint32_t>(), 1, Kd_ks, ctx->ksk.as<uint64_t>(), p.n + 1, 1, nullptr, nullptr, 0, ctx->ks_corr.as<uint64_t>()));
    negate_kernel<<<grid1d(p.n + 1, 256, ctx->sm_count), 256, 0, ctx->stream>>>(ctx->ks_corr.as<uint64_t>(), (size_t)p.n + 1);
    TRY(post_launch(ctx, "negate_kernel"));
    CU(cudaStreamSynchronize(ctx->stream));
    std::fill(h.begin(), h.end(), 1u << (p.pfks_b - 1));
    CU(cudaMemcpyAsync(ctx->ws_misc.p, h.data(), (size_t)Kd_pf * 4, cudaMemcpyHostToDevice, ctx->stream));
    const size_t W = (size_t)ctx->G() * p.N;
    TRY(gemm(ctx, ctx->ws_misc.as<uint32_t>(), 1, Kd_pf, ctx->pfpksk.as<uint64_t>(), (int)W, ctx->G(), nullptr, nullptr, 0, ctx->pfks_corr.as<uint64_t>()));
    negate_kernel<<<grid1d(W * ctx->G(), 256, ctx->sm_count), 256, 0, ctx->stream>>>(ctx->pfks_corr.as<uint64_t>(), W * ctx->G());
    TRY(post_launch(ctx, "negate_kernel"));
    CU(cudaStreamSynchronize(ctx->stream));
    {   // byte-plane tiles of the PFPKSK and the KSK for the tcgen05 GEMM
        const int nkb = (Kd_pf + UG_KB - 1) / UG_KB, tiles = ((int)W + UG_NT - 1) / UG_NT;
        const size_t units = (size_t)ctx->G() * tiles * nkb * 2 * UG_NT;
        umma_key_tiles_kernel<<<grid1d(units, 256, ctx->sm_count), 256, 0, ctx->stream>>>(ctx->pfpksk.as<uint64_t>(), ctx->G(), Kd_pf, (int)W, nkb, ctx->pfks_planes.as<uint8_t>());
        TRY(post_launch(ctx, "umma_key_tiles_kernel(pfks)"));
        const int nkb_ks = (Kd_ks + UG_KB - 1) / UG_KB, tiles_ks = (p.n + 1 + UG_NT - 1) / UG_NT;
        const size_t units_ks = (size_t)tiles_ks * nkb_ks * 2 * UG_NT;
        umma_key_tiles_kernel<<<grid1d(units_ks, 256, ctx->sm_count), 256, 0, ctx->stream>>>(ctx->ksk.as<uint64_t>(), 1, Kd_ks, p.n + 1, nkb_ks, ctx->ks_planes.as<uint8_t>());
        TRY(post_launch(ctx, "umma_key_tiles_kernel(ks)"));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    ctx->keys_valid = true;
    return TAC_OK;
}
int tac_ctx_upload_keys(tac_ctx* ctx, const uint64_t* bsk_std, const uint64_t* ksk, const uint64_t* pfpksk) {
    LOCK(ctx);
    TRY(tac_ctx_alloc_keys(ctx));
    const TacParams& p = ctx->p;
    CU(cudaMemcpyAsync(ctx->ksk.p, ksk, ctx->ksk_words() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->pfpksk.p, pfpksk, ctx->pfpksk_words() * 8, cudaMemcpyHostToDevice, ctx->stream));
    // BSK: standard → Fourier on the device, in slices ([U] fft64/crypto/bootstrap.rs::fill_with_forward_fourier)
    const size_t polys = (size_t)p.n * p.pbs_l * ctx->G() * ctx->G();
    const size_t slice = 16384;
    TRY(ensure(ctx, ctx->ws_misc, slice * p.N * 8));
    for (size_t q = 0; q < polys; q += slice) {
        const size_t cnt = std::min(slice, polys - q);
        CU(cudaMemcpyAsync(ctx->ws_misc.p, bsk_std + q * p.N, cnt * p.N * 8, cudaMemcpyHostToDevice, ctx->stream));
        TRY(poly_fft(ctx, ctx->ws_misc.as<uint64_t>(), cnt, ctx->bsk_f.as<cplx>() + q * (p.N / 2)));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    return tac_ctx_keys_ready(ctx);
}

// evaluation keys straight from a key file (wire.cpp): sections 3-5 must be present and belong to this parameter set
int tac_ctx_load_keys(tac_ctx* ctx, const char* path) {
    LOCK(ctx);
    tac_params fp;
    uint32_t present = 0;
    if (int rc = tac_keys_load_params(path, &fp, &present)) return fail(ctx, rc, std::string("cannot read key file ") + (path ? path : "(null)"));
    if (memcmp(&fp, &ctx->p, sizeof fp) != 0) return fail(ctx, TAC_ERR_ARG, "key file was written for another parameter set");
    if ((present & 0x38u) != 0x38u) return fail(ctx, TAC_ERR_STATE, "key file lacks evaluation-key sections (3 BSK, 4 KSK, 5 PFPKSK)");
    std::vector<uint64_t> bsk(tac_key_len(&fp, 2)), ksk(tac_key_len(&fp, 3)), pf(tac_key_len(&fp, 4));
    if (int rc = tac_keys_load(path, &fp, nullptr, nullptr, bsk.data(), ksk.data(), pf.data())) return fail(ctx, rc, "key file truncated or corrupted (checksum)");
    return tac_ctx_upload_keys(ctx, bsk.data(), ksk.data(), pf.data());
}

int tac_lut_register(tac_ctx* ctx, int n_in, int n_out, const uint64_t* table, size_t len) {
    LOCK(ctx);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return fail(ctx, TAC_ERR_CUDA, "cudaSetDevice");
    const size_t per = tac_lut_len(n_in, ctx->p.N);
    if (n_in <= 0 || n_in > 16 || n_out <= 0 || n_out > 64 || len != per * (size_t)n_out) return fail(ctx, TAC_ERR_ARG, "LUT shape does not match (n_in, n_out, N)");
    Lut l{n_in, n_out, per, nullptr};
    if (cudaMalloc(&l.dev, len * 8) != cudaSuccess) return fail(ctx, TAC_ERR_CUDA, "cudaMalloc(LUT)");
    if (cudaMemcpy(l.dev, table, len * 8, cudaMemcpyHostToDevice) != cudaSuccess) return fail(ctx, TAC_ERR_CUDA, "cudaMemcpy(LUT)");
    ctx->luts.push_back(l);
    return (int)ctx->luts.size() - 1;
}

int tac_wopbs_batch_dev(tac_ctx* ctx, int lut_id, int batch, const uint64_t* in_dev, uint64_t* out_dev) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    const Lut* lut; TRY(get_lut(ctx, lut_id, &lut));
    if (batch < 0) return fail(ctx, TAC_ERR_ARG, "negative batch");
    if (batch == 0) return TAC_OK;
    return wopbs_dev(ctx, *lut, batch, in_dev, out_dev);
}
int tac_wopbs_batch(tac_ctx* ctx, int lut_id, int batch, const uint64_t* in_host, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    const Lut* lut; TRY(get_lut(ctx, lut_id, &lut));
    if (batch < 0) return fail(ctx, TAC_ERR_ARG, "negative batch");
    if (batch == 0) return TAC_OK;
    const size_t big1 = (size_t)ctx->big() + 1;
    const size_t in_b = (size_t)batch * lut->n_in * big1 * 8, out_b = (size_t)batch * lut->n_out * big1 * 8;
    TRY(ensure(ctx, ctx->ws_in, in_b));
    TRY(ensure(ctx, ctx->ws_out, out_b));
    CU(cudaMemcpyAsync(ctx->ws_in.p, in_host, in_b, cudaMemcpyHostToDevice, ctx->stream));
    TRY(wopbs_dev(ctx, *lut, batch, ctx->ws_in.as<uint64_t>(), ctx->ws_out.as<uint64_t>()));
    CU(cudaMemcpyAsync(out_host, ctx->ws_out.p, out_b, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}

// Coalescing form of tac_wopbs_batch for callers that arrive one SBOX at a time from many threads (the reference's rayon
// fan-out over 16 bytes × blocks).  The first caller to find no leader becomes the leader: it waits `window` µs for
// company, takes everything queued, runs ONE batched pass per LUT and hands the results back; callers that arrive while a
// pass is running queue up for the next leader.  Every caller blocks until its own request is done.
int tac_ctx_set_coalescing(tac_ctx* ctx, int window_us, int max_batch) {
    std::lock_guard<std::mutex> lk(ctx->q_mu);
    if (window_us < 0 || max_batch < 1) return fail(ctx, TAC_ERR_ARG, "coalescing window / batch out of range");
    ctx->q_window_us = window_us; ctx->q_max_batch = max_batch;
    return TAC_OK;
}
int tac_ctx_coalescing_stats(tac_ctx* ctx, uint64_t* requests, uint64_t* passes) {
    std::lock_guard<std::mutex> lk(ctx->q_mu);
    if (requests) *requests = ctx->q_requests;
    if (passes) *passes = ctx->q_passes;
    return TAC_OK;
}
static void run_coalesced_group(tac_ctx* ctx, std::vector<PendingWopbs*>& grp) {
    LOCK(ctx);
    auto finish = [&](int rc) { for (auto* r : grp) { r->rc = rc; if (rc) r->err = g_error; } };
    if (cudaSetDevice(ctx->device) != cudaSuccess) return finish(fail(ctx, TAC_ERR_CUDA, "cudaSetDevice"));
    const Lut* lut;
    if (int rc = get_lut(ctx, grp[0]->lut_id, &lut)) return finish(rc);
    const size_t big1 = (size_t)ctx->big() + 1, in_ct = (size_t)lut->n_in * big1 * 8, out_ct = (size_t)lut->n_out * big1 * 8;
    size_t total = 0;
    for (auto* r : grp) total += (size_t)r->batch;
    if (int rc = ensure(ctx, ctx->ws_in, total * in_ct)) return finish(rc);
    if (int rc = ensure(ctx, ctx->ws_out, total * out_ct)) return finish(rc);
    auto cu = [&](cudaError_t e, const char* what) { return e == cudaSuccess ? 0 : fail(ctx, TAC_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e)); };
    size_t off = 0;
    for (auto* r : grp) {
        if (int rc = cu(cudaMemcpyAsync(ctx->ws_in.as<uint8_t>() + off * in_ct, r->in, (size_t)r->batch * in_ct, cudaMemcpyHostToDevice, ctx->stream), "H2D")) return finish(rc);
        off += (size_t)r->batch;
    }
    if (int rc = wopbs_dev(ctx, *lut, (int)total, ctx->ws_in.as<uint64_t>(), ctx->ws_out.as<uint64_t>())) return finish(rc);
    off = 0;
    for (auto* r : grp) {
        if (int rc = cu(cudaMemcpyAsync(r->out, ctx->ws_out.as<uint8_t>() + off * out_ct, (size_t)r->batch * out_ct, cudaMemcpyDeviceToHost, ctx->stream), "D2H")) return finish(rc);
        off += (size_t)r->batch;
    }
    finish(cu(cudaStreamSynchronize(ctx->stream), "cudaStreamSynchronize"));
}
int tac_wopbs_coalesced(tac_ctx* ctx, int lut_id, int batch, const uint64_t* in_host, uint64_t* out_host) {
    if (batch < 0) return fail(ctx, TAC_ERR_ARG, "negative batch");
    if (batch == 0) return TAC_OK;
    PendingWopbs me{lut_id, batch, in_host, out_host};
    std::unique_lock<std::mutex> lk(ctx->q_mu);
    ctx->q_pending.push_back(&me);
    ctx->q_requests++;
    ctx->q_cv.notify_all();
    for (;;) {
        ctx->q_cv.wait(lk, [&] { return me.done || !ctx->q_leader; });
        if (me.done) break;
        // become the leader of the next pass
        ctx->q_leader = true;
        if (ctx->q_window_us > 0) {
            const auto deadline = std::chrono::steady_clock::now() + std::chrono::microseconds(ctx->q_window_us);
            size_t seen = 0;
            // keep waiting while requests are still arriving, at most `window` after the last arrival check
            while (ctx->q_cv.wait_until(lk, deadline, [&] { return ctx->q_pending.size() != seen; })) {
                seen = ctx->q_pending.size();
                size_t cts = 0;
                for (auto* r : ctx->q_pending) cts += (size_t)r->batch;
                if (cts >= (size_t)ctx->q_max_batch) break;
            }
        }
        std::vector<PendingWopbs*> mine;
        mine.swap(ctx->q_pending);
        lk.unlock();
        // one pass per distinct LUT, in arrival order
        std::vector<bool> used(mine.size(), false);
        size_t n_groups = 0;
        for (size_t i = 0; i < mine.size(); i++) {
            if (used[i]) continue;
            std::vector<PendingWopbs*> grp;
            for (size_t j = i; j < mine.size(); j++)
                if (!used[j] && mine[j]->lut_id == mine[i]->lut_id) { used[j] = true; grp.push_back(mine[j]); }
            run_coalesced_group(ctx, grp);
            n_groups++;
        }
        lk.lock();
        ctx->q_passes += n_groups;
        for (auto* r : mine) r->done = true;
        ctx->q_leader = false;
        ctx->q_cv.notify_all();
    }
    if (me.rc) g_error = me.err;
    return me.rc;
}

int tac_lwe_add_batch_dev(tac_ctx* ctx, uint64_t* a, const uint64_t* b, size_t n_cts) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    const size_t total = n_cts * ((size_t)ctx->big() + 1);
    if (total == 0) return TAC_OK;
    lwe_add_kernel<<<grid1d(total, 256, ctx->sm_count), 256, 0, ctx->stream>>>(a, b, total);
    return post_launch(ctx, "lwe_add_kernel");
}
int tac_lwe_add_batch(tac_ctx* ctx, uint64_t* a_host, const uint64_t* b_host, size_t n_cts) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    const size_t bytes = n_cts * ((size_t)ctx->big() + 1) * 8;
    if (bytes == 0) return TAC_OK;
    TRY(ensure(ctx, ctx->ws_in, bytes));
    TRY(ensure(ctx, ctx->ws_out, bytes));
    CU(cudaMemcpyAsync(ctx->ws_in.p, a_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->ws_out.p, b_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    TRY(tac_lwe_add_batch_dev(ctx, ctx->ws_in.as<uint64_t>(), ctx->ws_out.as<uint64_t>(), n_cts));
    CU(cudaMemcpyAsync(a_host, ctx->ws_in.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}

// ------------------------------------------------------------------------------------------------ fused AES
int tac_aes_set_key_schedule(tac_ctx* ctx, const uint64_t* ks_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    return ks_set(ctx, ctx->single, 1, ks_host);
}
int tac_aes_key_schedule_buffer(tac_ctx* ctx, void** dev_ptr, size_t* bytes) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    TRY(ks_set(ctx, ctx->single, 1, nullptr));
    *dev_ptr = ctx->single.w.p; *bytes = key_sched_bytes(ctx);
    return TAC_OK;
}

int tac_aes_encrypt_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_dev, uint64_t* out_dev) {
    return aes_call(ctx, AesDir::Forward, false, nullptr, n_blocks, rounds, in_noise_sq, in_dev, nullptr, nullptr, out_dev, false);
}
int tac_aes_encrypt_blocks(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_host, uint64_t* out_host) {
    return aes_call(ctx, AesDir::Forward, false, nullptr, n_blocks, rounds, in_noise_sq, in_host, nullptr, nullptr, out_host, true);
}
// trivial input: no noise of its own
int tac_aes_encrypt_public_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_dev) {
    return aes_call(ctx, AesDir::Forward, false, nullptr, n_blocks, rounds, 0, nullptr, blocks_host, xor_host, out_dev, false);
}
int tac_aes_encrypt_public_blocks(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_host) {
    return aes_call(ctx, AesDir::Forward, false, nullptr, n_blocks, rounds, 0, nullptr, blocks_host, xor_host, out_host, true);
}

// ------------------------------------------------------------------------------------ AES decryption (FIPS-197 §5.3.5)
// Equivalent inverse cipher (aes_blocks_dev, AesDir::Inverse).  InvS·{14, 11, 13, 9} comes out of one 8 → 32 circuit
// bootstrap per byte, so a middle round sums 4 outputs of squared noise 8 and one round key of level 1: 33, as in the
// forward direction.  Round keys are read from dk only.
int tac_aes_decrypt_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_dev, uint64_t* out_dev) {
    return aes_call(ctx, AesDir::Inverse, false, nullptr, n_blocks, rounds, in_noise_sq, in_dev, nullptr, nullptr, out_dev, false);
}
int tac_aes_decrypt_blocks(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_host, uint64_t* out_host) {
    return aes_call(ctx, AesDir::Inverse, false, nullptr, n_blocks, rounds, in_noise_sq, in_host, nullptr, nullptr, out_host, true);
}

// decryption of PUBLIC ciphertext blocks (AES-ECB / AES-CBC transciphering): state0 = dk[40..43] + trivial(block), the
// plan runs along the inverse dependence rule, xor_host (the previous ciphertext blocks for CBC) joins the final round
int tac_aes_decrypt_public_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_dev) {
    return aes_call(ctx, AesDir::Inverse, false, nullptr, n_blocks, rounds, 0, nullptr, blocks_host, xor_host, out_dev, false);
}
int tac_aes_decrypt_public_blocks(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_host) {
    return aes_call(ctx, AesDir::Inverse, false, nullptr, n_blocks, rounds, 0, nullptr, blocks_host, xor_host, out_host, true);
}

// inverse key schedule on the device from the resident encryption schedule (inv_key_expand with one key)
int tac_aes_inv_key_schedule(tac_ctx* ctx, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    return ks_invert(ctx, ctx->single, out_host);
}
int tac_aes_set_inv_key_schedule(tac_ctx* ctx, const uint64_t* dk_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!dk_host) return fail(ctx, TAC_ERR_ARG, "NULL inverse key schedule");
    return ks_set_inv(ctx, ctx->single, 1, dk_host);
}

// fhe_sbox_gal_mul_pbs::key_schedule (:134-164): key_expand with one key, into the single schedule
int tac_aes_key_schedule(tac_ctx* ctx, const uint64_t* key_bits_host, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!key_bits_host) return fail(ctx, TAC_ERR_ARG, "NULL key bits");
    return ks_expand(ctx, ctx->single, 1, key_bits_host, out_host);
}

// ------------------------------------------------------------------------------------------------ AES under many keys
// A table of key schedules beside the single one.  Block b of a keyed call runs under entry key_idx[b]; its output equals,
// word for word, the single-key entry point's for that block with that entry resident (every stage gives the same words
// whatever the batch).
int tac_aes_key_table(tac_ctx* ctx, int n_keys, const uint64_t* key_bits_host, uint64_t* key_scheds_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (n_keys < 1 || !key_bits_host) return fail(ctx, TAC_ERR_ARG, "need n_keys >= 1 and key bits");
    return ks_expand(ctx, ctx->table, n_keys, key_bits_host, key_scheds_host);
}
int tac_aes_set_key_table(tac_ctx* ctx, int n_keys, const uint64_t* key_scheds_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (n_keys < 1 || !key_scheds_host) return fail(ctx, TAC_ERR_ARG, "need n_keys >= 1 and key schedules");
    return ks_set(ctx, ctx->table, n_keys, key_scheds_host);
}
int tac_aes_inv_key_table(tac_ctx* ctx, uint64_t* inv_key_scheds_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    return ks_invert(ctx, ctx->table, inv_key_scheds_host);
}
int tac_aes_set_inv_key_table(tac_ctx* ctx, const uint64_t* inv_key_scheds_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (ctx->table.n < 1) return fail(ctx, TAC_ERR_STATE, ctx->table.absent);
    if (!inv_key_scheds_host) return fail(ctx, TAC_ERR_ARG, "NULL inverse key schedules");
    return ks_set_inv(ctx, ctx->table, ctx->table.n, inv_key_scheds_host);
}

int tac_aes_encrypt_blocks_keyed_dev(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const int32_t* key_idx_host, const uint64_t* in_dev,
                                     uint64_t* out_dev) {
    return aes_call(ctx, AesDir::Forward, true, key_idx_host, n_blocks, rounds, in_noise_sq, in_dev, nullptr, nullptr, out_dev, false);
}
int tac_aes_encrypt_blocks_keyed(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const int32_t* key_idx_host, const uint64_t* in_host,
                                 uint64_t* out_host) {
    return aes_call(ctx, AesDir::Forward, true, key_idx_host, n_blocks, rounds, in_noise_sq, in_host, nullptr, nullptr, out_host, true);
}
int tac_aes_encrypt_public_blocks_keyed_dev(tac_ctx* ctx, int n_blocks, int rounds, const int32_t* key_idx_host, const uint8_t* blocks_host,
                                            const uint8_t* xor_host, uint64_t* out_dev) {
    return aes_call(ctx, AesDir::Forward, true, key_idx_host, n_blocks, rounds, 0, nullptr, blocks_host, xor_host, out_dev, false);
}
int tac_aes_encrypt_public_blocks_keyed(tac_ctx* ctx, int n_blocks, int rounds, const int32_t* key_idx_host, const uint8_t* blocks_host,
                                        const uint8_t* xor_host, uint64_t* out_host) {
    return aes_call(ctx, AesDir::Forward, true, key_idx_host, n_blocks, rounds, 0, nullptr, blocks_host, xor_host, out_host, true);
}
int tac_aes_decrypt_blocks_keyed_dev(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const int32_t* key_idx_host, const uint64_t* in_dev,
                                     uint64_t* out_dev) {
    return aes_call(ctx, AesDir::Inverse, true, key_idx_host, n_blocks, rounds, in_noise_sq, in_dev, nullptr, nullptr, out_dev, false);
}
int tac_aes_decrypt_blocks_keyed(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const int32_t* key_idx_host, const uint64_t* in_host,
                                 uint64_t* out_host) {
    return aes_call(ctx, AesDir::Inverse, true, key_idx_host, n_blocks, rounds, in_noise_sq, in_host, nullptr, nullptr, out_host, true);
}
int tac_aes_decrypt_public_blocks_keyed_dev(tac_ctx* ctx, int n_blocks, int rounds, const int32_t* key_idx_host, const uint8_t* blocks_host,
                                            const uint8_t* xor_host, uint64_t* out_dev) {
    return aes_call(ctx, AesDir::Inverse, true, key_idx_host, n_blocks, rounds, 0, nullptr, blocks_host, xor_host, out_dev, false);
}
int tac_aes_decrypt_public_blocks_keyed(tac_ctx* ctx, int n_blocks, int rounds, const int32_t* key_idx_host, const uint8_t* blocks_host,
                                        const uint8_t* xor_host, uint64_t* out_host) {
    return aes_call(ctx, AesDir::Inverse, true, key_idx_host, n_blocks, rounds, 0, nullptr, blocks_host, xor_host, out_host, true);
}

// ------------------------------------------------------------------------------------------------ AES-CCM / AES-GCM transciphering
// key_idx NULL: every record under the single resident schedule, else record i under key table entry key_idx[i].  The
// context lock is taken here only.
int tac_aes_ccm_transcipher_dev(tac_ctx* ctx, int n_msgs, const int32_t* key_idx, const tac_ccm_msg* msgs, uint64_t* pt_out_dev,
                                uint64_t* valid_out_dev) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    return aes_ccm_dev(ctx, n_msgs, key_idx, msgs, pt_out_dev, valid_out_dev);
}
int tac_aes_ccm_transcipher(tac_ctx* ctx, int n_msgs, const int32_t* key_idx, const tac_ccm_msg* msgs, uint64_t* pt_out_host,
                            uint64_t* valid_out_host) {
    return records_host(ctx, ccm_check, aes_ccm_dev, n_msgs, key_idx, msgs, pt_out_host, valid_out_host);
}
int tac_aes_gcm_hash_key(tac_ctx* ctx, int depth, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    return gcm_hash_key(ctx, false, depth, out_host);
}
int tac_aes_gcm_hash_key_table(tac_ctx* ctx, int depth, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    return gcm_hash_key(ctx, true, depth, out_host);
}
int tac_aes_gcm_transcipher_dev(tac_ctx* ctx, int n_msgs, const int32_t* key_idx, const tac_ccm_msg* msgs, uint64_t* pt_out_dev,
                                uint64_t* valid_out_dev) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    return aes_gcm_dev(ctx, n_msgs, key_idx, msgs, pt_out_dev, valid_out_dev);
}
int tac_aes_gcm_transcipher(tac_ctx* ctx, int n_msgs, const int32_t* key_idx, const tac_ccm_msg* msgs, uint64_t* pt_out_host,
                            uint64_t* valid_out_host) {
    return records_host(ctx, gcm_check, aes_gcm_dev, n_msgs, key_idx, msgs, pt_out_host, valid_out_host);
}

// ------------------------------------------------------------------------------------------------ single stages
int tac_stage_keyswitch(tac_ctx* ctx, int n, const uint64_t* in_host, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!ctx->keys_valid) return fail(ctx, TAC_ERR_STATE, "evaluation keys not uploaded");
    if (n <= 0) return n == 0 ? TAC_OK : fail(ctx, TAC_ERR_ARG, "negative count");
    const size_t ib = (size_t)n * (ctx->big() + 1) * 8, ob = (size_t)n * (ctx->p.n + 1) * 8;
    TRY(ensure(ctx, ctx->ws_in, ib)); TRY(ensure(ctx, ctx->ws_small, ob));
    CU(cudaMemcpyAsync(ctx->ws_in.p, in_host, ib, cudaMemcpyHostToDevice, ctx->stream));
    TRY(stage_ks(ctx, ctx->ws_in.as<uint64_t>(), n, ctx->ws_small.as<uint64_t>()));
    CU(cudaMemcpyAsync(out_host, ctx->ws_small.p, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}
// n products a·b in GF(2^128) (GCM's field and bit order), a, b, out [n][128][kN+1]; outputs at squared noise 1
int tac_gf128_mul(tac_ctx* ctx, int n, const uint64_t* a_host, const uint64_t* b_host, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!ctx->keys_valid) return fail(ctx, TAC_ERR_STATE, "evaluation keys not uploaded");
    if (n <= 0) return n == 0 ? TAC_OK : fail(ctx, TAC_ERR_ARG, "negative count");
    if (!a_host || !b_host || !out_host) return fail(ctx, TAC_ERR_ARG, "NULL operand or output");
    TRY(gf_noise_check(ctx));
    const size_t words = (size_t)n * 128 * (ctx->big() + 1);
    TRY(ensure(ctx, ctx->ws_in, 2 * words * 8));
    TRY(ensure(ctx, ctx->ws_out, words * 8));
    CU(cudaMemcpyAsync(ctx->ws_in.p, a_host, words * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->ws_in.as<uint64_t>() + words, b_host, words * 8, cudaMemcpyHostToDevice, ctx->stream));
    TRY(gf128_mul_dev(ctx, n, ctx->ws_in.as<uint64_t>(), ctx->ws_in.as<uint64_t>() + words, ctx->ws_out.as<uint64_t>()));
    CU(cudaMemcpyAsync(out_host, ctx->ws_out.p, words * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}
int tac_stage_pbs(tac_ctx* ctx, int n, const uint64_t* in_host, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!ctx->keys_valid) return fail(ctx, TAC_ERR_STATE, "evaluation keys not uploaded");
    if (n <= 0) return n == 0 ? TAC_OK : fail(ctx, TAC_ERR_ARG, "negative count");
    const size_t ib = (size_t)n * (ctx->p.n + 1) * 8, ob = (size_t)n * (ctx->big() + 1) * 8;
    TRY(ensure(ctx, ctx->ws_small, ib)); TRY(ensure(ctx, ctx->ws_pbs, ob));
    CU(cudaMemcpyAsync(ctx->ws_small.p, in_host, ib, cudaMemcpyHostToDevice, ctx->stream));
    TRY(pbs(ctx, ctx->ws_small.as<uint64_t>(), n, ctx->ws_pbs.as<uint64_t>()));
    CU(cudaMemcpyAsync(out_host, ctx->ws_pbs.p, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}
// [U] fft64/crypto/wop_pbs.rs::extract_bits — WopbsKey::extract_bits(DeltaLog, ct, ExtractedBitsCount): the general chain
// keyswitch → bootstrap of the sign → subtract, least significant bit first; output list most significant bit first.
// The AES path calls it with (63, 1), which is the keyswitch alone (reference shortint_woppbs_1bit.rs:342-349).
int tac_extract_bits(tac_ctx* ctx, int delta_log, int n_bits, int n_cts, const uint64_t* in_host, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!ctx->keys_valid) return fail(ctx, TAC_ERR_STATE, "evaluation keys not uploaded");
    if (n_bits < 1 || delta_log < 1 || delta_log + n_bits > 64) return fail(ctx, TAC_ERR_ARG, "need 1 <= delta_log and delta_log + n_bits <= 64");
    if (n_cts <= 0) return n_cts == 0 ? TAC_OK : fail(ctx, TAC_ERR_ARG, "negative count");
    const size_t L = (size_t)ctx->big() + 1, S = (size_t)ctx->p.n + 1, total = (size_t)n_cts * L;
    TRY(ensure(ctx, ctx->ws_in, total * 8));                 // remaining
    TRY(ensure(ctx, ctx->ws_state, total * 8));              // shifted
    TRY(ensure(ctx, ctx->ws_pbs, total * 8));                // bootstrapped bit
    TRY(ensure(ctx, ctx->ws_small, (size_t)n_cts * S * 8));
    TRY(ensure(ctx, ctx->ws_out, (size_t)n_cts * n_bits * S * 8));
    uint64_t* rem = ctx->ws_in.as<uint64_t>();
    uint64_t* shifted = ctx->ws_state.as<uint64_t>();
    CU(cudaMemcpyAsync(rem, in_host, total * 8, cudaMemcpyHostToDevice, ctx->stream));
    const int g = grid1d(total, 256, ctx->sm_count);
    for (int i = 0; i < n_bits; i++) {
        lwe_shl_kernel<<<g, 256, 0, ctx->stream>>>(rem, 64 - delta_log - i - 1, total, shifted);
        TRY(post_launch(ctx, "lwe_shl_kernel"));
        TRY(stage_ks(ctx, shifted, n_cts, ctx->ws_small.as<uint64_t>()));
        CU(cudaMemcpy2DAsync(ctx->ws_out.as<uint64_t>() + (size_t)(n_bits - 1 - i) * S, (size_t)n_bits * S * 8, ctx->ws_small.p, S * 8, S * 8, (size_t)n_cts,
                             cudaMemcpyDeviceToDevice, ctx->stream));
        if (i == n_bits - 1) break;
        TRY(pbs(ctx, ctx->ws_small.as<uint64_t>(), n_cts, ctx->ws_pbs.as<uint64_t>(), 1ull << (delta_log + i - 1)));
        lwe_sub_kernel<<<g, 256, 0, ctx->stream>>>(rem, ctx->ws_pbs.as<uint64_t>(), total);
        TRY(post_launch(ctx, "lwe_sub_kernel"));
    }
    CU(cudaMemcpyAsync(out_host, ctx->ws_out.p, (size_t)n_cts * n_bits * S * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}
int tac_stage_pfks(tac_ctx* ctx, int n, const uint64_t* in_host, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!ctx->keys_valid) return fail(ctx, TAC_ERR_STATE, "evaluation keys not uploaded");
    if (n <= 0) return n == 0 ? TAC_OK : fail(ctx, TAC_ERR_ARG, "negative count");
    const size_t ib = (size_t)n * (ctx->big() + 1) * 8, ob = (size_t)n * ctx->G() * ctx->G() * ctx->p.N * 8;
    TRY(ensure(ctx, ctx->ws_pbs, ib)); TRY(ensure(ctx, ctx->ws_ggsw, ob));
    CU(cudaMemcpyAsync(ctx->ws_pbs.p, in_host, ib, cudaMemcpyHostToDevice, ctx->stream));
    TRY(stage_pfks(ctx, ctx->ws_pbs.as<uint64_t>(), n, ctx->ws_ggsw.as<uint64_t>()));
    CU(cudaMemcpyAsync(out_host, ctx->ws_ggsw.p, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}
int tac_stage_vertical_packing(tac_ctx* ctx, int lut_id, int batch, const uint64_t* ggsw_std_host, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    const Lut* lut; TRY(get_lut(ctx, lut_id, &lut));
    if (batch <= 0) return batch == 0 ? TAC_OK : fail(ctx, TAC_ERR_ARG, "negative batch");
    const int G = ctx->G(), M = ctx->p.N / 2;
    const size_t nct = (size_t)batch * lut->n_in * ctx->p.cbs_l;              // GGSW level matrices
    const size_t ib = nct * G * G * ctx->p.N * 8, ob = (size_t)batch * lut->n_out * (ctx->big() + 1) * 8;
    TRY(ensure(ctx, ctx->ws_ggsw, ib)); TRY(ensure(ctx, ctx->ws_ggswf, nct * G * G * M * sizeof(cplx))); TRY(ensure(ctx, ctx->ws_out, ob));
    CU(cudaMemcpyAsync(ctx->ws_ggsw.p, ggsw_std_host, ib, cudaMemcpyHostToDevice, ctx->stream));
    TRY(poly_fft(ctx, ctx->ws_ggsw.as<uint64_t>(), nct * G * G, ctx->ws_ggswf.as<cplx>()));
    TRY(vertical_packing(ctx, *lut, ctx->ws_ggswf.as<cplx>(), batch, ctx->ws_out.as<uint64_t>()));
    CU(cudaMemcpyAsync(out_host, ctx->ws_out.p, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}

int tac_stage_poly_fft(tac_ctx* ctx, size_t n_polys, const uint64_t* polys_host, double* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (n_polys == 0) return TAC_OK;
    const size_t N = ctx->p.N, M = N / 2;
    TRY(ensure(ctx, ctx->ws_ggsw, n_polys * N * 8)); TRY(ensure(ctx, ctx->ws_ggswf, n_polys * M * sizeof(cplx)));
    CU(cudaMemcpyAsync(ctx->ws_ggsw.p, polys_host, n_polys * N * 8, cudaMemcpyHostToDevice, ctx->stream));
    TRY(poly_fft(ctx, ctx->ws_ggsw.as<uint64_t>(), n_polys, ctx->ws_ggswf.as<cplx>()));
    CU(cudaMemcpyAsync(out_host, ctx->ws_ggswf.p, n_polys * M * sizeof(cplx), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}
int tac_fft_slot_frequencies(int polynomial_size, int32_t* freq) {
    if (polynomial_size != 512 && polynomial_size != 1024) return TAC_ERR_ARG;
    const int M = polynomial_size / 2, P = M / 16;
    for (int q = 0; q < P; q++)
        for (int r = 0; r < 16; r++) freq[slot_of(q, r)] = q + P * r;
    return TAC_OK;
}
int tac_stage_sample_extract(tac_ctx* ctx, size_t n_glwe, const uint64_t* glwe_host, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (n_glwe == 0) return TAC_OK;
    const size_t ib = n_glwe * ctx->G() * ctx->p.N * 8, ob = n_glwe * ((size_t)ctx->big() + 1) * 8;
    TRY(ensure(ctx, ctx->ws_ggsw, ib)); TRY(ensure(ctx, ctx->ws_out, ob));
    CU(cudaMemcpyAsync(ctx->ws_ggsw.p, glwe_host, ib, cudaMemcpyHostToDevice, ctx->stream));
    TRY(check_launch(ctx, ctx->ops->sample_extract(klaunch(ctx), ctx->ws_ggsw.as<uint64_t>(), n_glwe, ctx->ws_out.as<uint64_t>()), "sample_extract_kernel"));
    CU(cudaMemcpyAsync(out_host, ctx->ws_out.p, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}

int tac_stage_cmux_rotate(tac_ctx* ctx, int levels, int base_log, const uint64_t* ggsw_std_host, int n_acc, const int32_t* rot, uint64_t* acc_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (n_acc <= 0) return n_acc == 0 ? TAC_OK : fail(ctx, TAC_ERR_ARG, "negative count");
    const TacParams& p = ctx->p;
    const int G = ctx->G(), M = p.N / 2;
    const size_t polys = (size_t)levels * G * G;
    const size_t ab = (size_t)n_acc * G * p.N * 8;
    TRY(ensure(ctx, ctx->ws_ggsw, polys * p.N * 8)); TRY(ensure(ctx, ctx->ws_ggswf, polys * M * sizeof(cplx)));
    TRY(ensure(ctx, ctx->ws_out, ab)); TRY(ensure(ctx, ctx->ws_misc, (size_t)n_acc * 4));
    CU(cudaMemcpyAsync(ctx->ws_ggsw.p, ggsw_std_host, polys * p.N * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->ws_out.p, acc_host, ab, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->ws_misc.p, rot, (size_t)n_acc * 4, cudaMemcpyHostToDevice, ctx->stream));
    TRY(poly_fft(ctx, ctx->ws_ggsw.as<uint64_t>(), polys, ctx->ws_ggswf.as<cplx>()));
    TRY(check_launch(ctx, ctx->ops->cmux_test(klaunch(ctx), levels, ctx->ws_ggswf.as<cplx>(), ctx->ws_misc.as<int>(), base_log, n_acc, ctx->ws_out.as<uint64_t>()),
                     "cmux_rotate_test_kernel"));
    CU(cudaMemcpyAsync(acc_host, ctx->ws_out.p, ab, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}

}  // extern "C"
