// capi.cu — device context, key upload, the batched circuit-bootstrap pipeline and the fused AES paths behind the C ABI
// of include/tfhe_aes_cuda.h.  No CPU fallback: every entry point that computes fails with TAC_ERR_CUDA when there is
// no usable CUDA device.
#include "../../include/tfhe_aes_cuda.h"
#include "kernels_common.cuh"
#include "aes_plan.h"
#include "kernels_gemm_umma.cuh"
#include "ep_step.cuh"
#include "shape_launch.h"

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

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
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
    cplx* bsk_f = nullptr;
    uint64_t* ksk = nullptr;
    uint64_t* pfpksk = nullptr;
    uint64_t* ks_corr = nullptr;
    uint64_t* pfks_corr = nullptr;
    uint8_t* ks_planes = nullptr;        // byte planes of the KSK
    uint8_t* pfks_planes = nullptr;      // byte-plane tiles of the PFPKSK for the tcgen05 GEMM (kernels_gemm_umma.cuh)
    uint32_t* pfks_fix = nullptr;        // [0] = count, then uint2 (ct, k) entries
    bool keys_allocated = false, keys_valid = false;
    // tables
    cplx* wT = nullptr;            // combined twist/twiddle table (ep_core.cuh)
    const ShapeOps* ops = nullptr; // kernels of this (N, k)
    // LUTs
    std::vector<Lut> luts;
    int aes_lut24 = -1, aes_lut8 = -1, aes_lut1 = -1;
    int aes_lut_inv32 = -1, aes_lut_inv8 = -1, aes_lut_key32 = -1;   // decryption: InvS·{14,11,13,9}, InvS, b·{14,11,13,9}
    // AES key schedule
    uint64_t* key_sched = nullptr;
    uint64_t* inv_key_sched = nullptr;   // equivalent inverse cipher's schedule dk, same layout [44 words][4][8][kN+1]
    bool inv_key_sched_valid = false;    // dk belongs to the resident key_sched (cleared by tac_aes_set_key_schedule)
    uint64_t* rc_rows = nullptr;     // trivial(RC[1..10]) as byte ciphertexts [10][8][kN+1], uploaded once
    // workspace
    DevBuf ws_in, ws_out, ws_small, ws_ksdig, ws_pbs, ws_pfdig, ws_ggsw, ws_ggswf, ws_tree_a, ws_tree_b, ws_state, ws_muls, ws_misc;
    DevBuf ws_plan, ws_rep;          // public-block AES: uploaded plan tables / public bytes, compact S-box inputs
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

int ensure(tac_ctx* ctx, DevBuf& b, size_t bytes) {
    if (b.cap >= bytes) return TAC_OK;
    if (b.p) CU(cudaFree(b.p));
    b.p = nullptr; b.cap = 0;
    CU(cudaMalloc(&b.p, bytes));
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
KLaunch klaunch(tac_ctx* ctx) { return KLaunch{ctx->stream, ctx->wT, ctx->sm_count}; }
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
    return check_launch(ctx, ctx->ops->pbs(klaunch(ctx), p.pbs_l, small, nct, p.n, ctx->bsk_f, p.pbs_b, alpha, out), "pbs kernel");
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
    umma_digit_tiles_kernel<<<grid1d((size_t)mpad * nkb * 2, 256, ctx->sm_count), 256, 0, ctx->stream>>>(
        in, nct, mpad, big + 1, p.ks_b, p.ks_l, Kd, nkb, 1, DA, ctx->pfks_fix, reinterpret_cast<uint2*>(ctx->pfks_fix + 2), 0);
    TRY(post_launch(ctx, "umma_digit_tiles_kernel(ks)"));
    return gemm_umma<1>(ctx, DA, nct, ctx->ks_planes, W, 1, nkb, ctx->ks_corr, in + big, (size_t)big + 1, small);
}
// PFKS with all k+1 keys on the tensor cores: in [nct][big+1] → ggsw_std [nct][G][G·N]
int stage_pfks(tac_ctx* ctx, const uint64_t* in, int nct, uint64_t* ggsw) {
    const TacParams& p = ctx->p;
    const int big1 = ctx->big() + 1, Kd = big1 * p.pfks_l, nkb = (Kd + UG_KB - 1) / UG_KB;
    const int W = ctx->G() * p.N, mpad = ((nct + UG_MT - 1) / UG_MT) * UG_MT;
    if (p.pfks_b > 16) {       // digits wider than 16 bits (params_sqrd_lvl_1: base 2^24): 64-bit integer-pipe GEMM
        TRY(ensure(ctx, ctx->ws_pfdig, (size_t)nct * Kd * 4));
        pfks_digits_kernel<<<grid1d((size_t)nct * big1, 256, ctx->sm_count), 256, 0, ctx->stream>>>(in, nct, big1, p.pfks_b, p.pfks_l, ctx->ws_pfdig.as<uint32_t>());
        TRY(post_launch(ctx, "pfks_digits_kernel"));
        return gemm(ctx, ctx->ws_pfdig.as<uint32_t>(), nct, Kd, ctx->pfpksk, W, ctx->G(), ctx->pfks_corr, nullptr, 0, ggsw);
    }
    TRY(ensure(ctx, ctx->ws_pfdig, (size_t)2 * nkb * 2 * mpad * 16));
    CU(cudaMemsetAsync(ctx->pfks_fix, 0, 4, ctx->stream));
    uint8_t* DA = ctx->ws_pfdig.as<uint8_t>();
    umma_digit_tiles_kernel<<<grid1d((size_t)mpad * nkb * 2, 256, ctx->sm_count), 256, 0, ctx->stream>>>(
        in, nct, mpad, big1, p.pfks_b, p.pfks_l, Kd, nkb, 0, DA, ctx->pfks_fix, reinterpret_cast<uint2*>(ctx->pfks_fix + 2), ctx->fix_cap);
    TRY(post_launch(ctx, "umma_digit_tiles_kernel(pfks)"));
    TRY(gemm_umma<2>(ctx, DA, nct, ctx->pfks_planes, W, ctx->G(), nkb, ctx->pfks_corr, nullptr, 0, ggsw));
    pfks_fixup_kernel<<<64, 256, 0, ctx->stream>>>(ctx->pfks_fix, reinterpret_cast<const uint2*>(ctx->pfks_fix + 2), ctx->fix_cap, ctx->pfpksk, Kd, W, ctx->G(), ggsw);
    TRY(post_launch(ctx, "pfks_fixup_kernel"));
    // more ties than the list holds (crafted / trivial inputs): this kernel re-derives them all; otherwise it returns at once
    pfks_fixup_scan_kernel<<<dim3((ctx->G() * W + 255) / 256, std::min(nct, 2 * ctx->sm_count)), 256, 0, ctx->stream>>>(
        ctx->pfks_fix, ctx->fix_cap, in, nct, big1, p.pfks_b, p.pfks_l, ctx->pfpksk, Kd, W, ctx->G(), ggsw);
    return post_launch(ctx, "pfks_fixup_scan_kernel");
}

// the whole circuit bootstrap for `nbox` boxes resident on the device
int wopbs_dev(tac_ctx* ctx, const Lut& lut, int nbox, const uint64_t* in, uint64_t* out) {
    const TacParams& p = ctx->p;
    if (!ctx->keys_valid) return fail(ctx, TAC_ERR_STATE, "evaluation keys not uploaded");
    const int big1 = ctx->big() + 1, G = ctx->G(), M = p.N / 2, lc = p.cbs_l;
    const size_t ggsw_words = (size_t)G * G * p.N;
    const int max_boxes = (int)std::max<size_t>(1, ctx->max_cts / ((size_t)lut.n_in * lc));
    for (int b0 = 0; b0 < nbox; b0 += max_boxes) {
        const int nb = std::min(max_boxes, nbox - b0);
        const int nct = nb * lut.n_in;
        const uint64_t* cin = in + (size_t)b0 * lut.n_in * big1;
        uint64_t* cout = out + (size_t)b0 * lut.n_out * big1;
        TRY(ensure(ctx, ctx->ws_small, (size_t)nct * (p.n + 1) * 8));
        TRY(ensure(ctx, ctx->ws_pbs, (size_t)nct * lc * big1 * 8));
        TRY(ensure(ctx, ctx->ws_ggsw, (size_t)nct * lc * ggsw_words * 8));
        TRY(ensure(ctx, ctx->ws_ggswf, (size_t)nct * lc * G * G * M * sizeof(cplx)));
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
        TRY(poly_fft(ctx, ctx->ws_ggsw.as<uint64_t>(), (size_t)nct * lc * G * G, ctx->ws_ggswf.as<cplx>()));   // fill_with_forward_fourier
        TRY(stage_event(ctx, 4));
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
int aes_blocks_dev(tac_ctx* ctx, AesDir dir, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_dev, const uint8_t* blocks_host,
                   const uint8_t* xor_host, uint64_t* out_dev) {
    const bool fwd = dir == AesDir::Forward, pub = in_dev == nullptr;
    std::vector<AesRoundPlan> plan;
    if (pub) {
        if (aes_public_plan_build(n_blocks, rounds, blocks_host, dir, plan)) return fail(ctx, TAC_ERR_ARG, "n_blocks / rounds out of range, or NULL blocks");
    } else {
        if (n_blocks < 0 || rounds < 1 || rounds > 10) return fail(ctx, TAC_ERR_ARG, "n_blocks / rounds out of range");
        plan.assign(rounds, AesRoundPlan{16 * (int64_t)n_blocks, true});
    }
    if (n_blocks == 0) return TAC_OK;
    TRY(aes_noise_check(ctx, in_noise_sq, rounds));
    TRY(fwd ? ensure_aes_luts(ctx) : ensure_aes_inv_luts(ctx));
    const size_t L = (size_t)ctx->big() + 1, byte_words = 8 * L, blk = 16 * byte_words;
    const size_t npos = (size_t)n_blocks * 16, total = (size_t)n_blocks * blk;
    // per direction: S-box LUTs S·{1,2,3} / S or InvS·{14,11,13,9} / InvS, round keys, (Inv)ShiftRows kernels
    const uint64_t* keys = fwd ? ctx->key_sched : ctx->inv_key_sched;
    const Lut& lut_mid = ctx->luts[fwd ? ctx->aes_lut24 : ctx->aes_lut_inv32];
    const Lut& lut_last = ctx->luts[fwd ? ctx->aes_lut8 : ctx->aes_lut_inv8];
    const uint64_t* k_first = fwd ? keys : keys + (size_t)10 * blk;
    const uint64_t* k_last = fwd ? keys + (size_t)10 * blk : keys;
    const auto mix_columns = fwd ? aes_mix_columns_kernel<true> : aes_mix_columns_kernel<false>;
    const auto final_round = fwd ? aes_final_round_kernel<true> : aes_final_round_kernel<false>;
    // public input: one upload of the blocks, the XOR bytes, then rep_pos / idx of every round that shares
    std::vector<size_t> off_rep(rounds, 0), off_idx(rounds, 0);
    std::vector<uint8_t> host;
    size_t max_rep = 0;
    if (pub) {
        size_t bytes = 2 * npos;
        for (int r = 0; r < rounds; r++) {
            if (plan[r].identity) continue;
            off_rep[r] = bytes; bytes += (size_t)plan[r].boxes * 4;
            off_idx[r] = bytes; bytes += npos * 4;
            max_rep = std::max(max_rep, (size_t)plan[r].boxes);
        }
        host.assign(bytes, 0);
        std::memcpy(host.data(), blocks_host, npos);
        if (xor_host) std::memcpy(host.data() + npos, xor_host, npos);
        for (int r = 0; r < rounds; r++) {
            if (plan[r].identity) continue;
            std::memcpy(host.data() + off_rep[r], plan[r].rep_pos.data(), (size_t)plan[r].boxes * 4);
            std::memcpy(host.data() + off_idx[r], plan[r].idx.data(), npos * 4);
        }
        TRY(ensure(ctx, ctx->ws_plan, bytes));
    }
    TRY(ensure(ctx, ctx->ws_state, total * 8));
    TRY(ensure(ctx, ctx->ws_muls, total * (fwd ? 3 : 4) * 8));
    if (pub) {
        TRY(ensure(ctx, ctx->ws_rep, std::max<size_t>(1, max_rep) * byte_words * 8));
        // pageable source: the call returns once the bytes are staged, so `host` may go out of scope before the copy lands
        CU(cudaMemcpyAsync(ctx->ws_plan.p, host.data(), host.size(), cudaMemcpyHostToDevice, ctx->stream));
    }
    const uint8_t* d_plan = ctx->ws_plan.as<uint8_t>();
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
            aes_add_round_key_kernel<<<g, 256, 0, ctx->stream>>>(in_dev, k_first, blk, total, state);          // :96-99
            TRY(post_launch(ctx, "aes_add_round_key_kernel"));
            *in = state;
        } else if (rd == 1) {
            uint64_t* dst = plan[r].identity ? state : rep;
            aes_public_round1_kernel<<<grid1d(n_words, 256, ctx->sm_count), 256, 0, ctx->stream>>>(k_first, d_plan, rep_pos(r), (int)L, n_words, dst);
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
        mix_columns<<<g, 256, 0, ctx->stream>>>(muls, keys + (size_t)(fwd ? rd : rounds - rd) * blk, (int)L, total, state, idx(rd - 1));
        TRY(post_launch(ctx, "aes_mix_columns_kernel"));
    }
    TRY(sbox_inputs(rounds, &in));
    TRY(wopbs_dev(ctx, lut_last, (int)plan[rounds - 1].boxes, in, muls));                                     // sub_bytes :51-58
    final_round<<<g, 256, 0, ctx->stream>>>(muls, k_last, (int)L, total, out_dev, idx(rounds - 1), xor_host ? d_plan + npos : nullptr);
    return post_launch(ctx, "aes_final_round_kernel");
}

// host-buffer form of an AES _dev entry point: ciphertext input (ct_in) through ws_in, the output through ws_out;
// dev_call(in_dev, out_dev) runs the _dev entry point
template <class DevCall>
int aes_blocks_host(tac_ctx* ctx, int n_blocks, bool ct_in, const uint64_t* in_host, uint64_t* out_host, DevCall dev_call) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (n_blocks <= 0) return n_blocks == 0 ? TAC_OK : fail(ctx, TAC_ERR_ARG, "negative n_blocks");
    const size_t bytes = (size_t)n_blocks * 128 * (ctx->big() + 1) * 8;
    if (ct_in) TRY(ensure(ctx, ctx->ws_in, bytes));
    TRY(ensure(ctx, ctx->ws_out, bytes));
    if (ct_in) CU(cudaMemcpyAsync(ctx->ws_in.p, in_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    TRY(dev_call(ctx->ws_in.as<const uint64_t>(), ctx->ws_out.as<uint64_t>()));
    CU(cudaMemcpyAsync(out_host, ctx->ws_out.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
}

// dk present and made from (or uploaded for) the resident encryption schedule
int inv_key_sched_check(tac_ctx* ctx) {
    if (!ctx->inv_key_sched || !ctx->inv_key_sched_valid)
        return fail(ctx, TAC_ERR_STATE, "no inverse key schedule for the resident key schedule (tac_aes_inv_key_schedule or tac_aes_set_inv_key_schedule)");
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
    if (cudaMalloc(&ctx->wT, w.size() * sizeof(cplx)) != cudaSuccess) return bail("cudaMalloc(tables) failed");
    cudaMemcpy(ctx->wT, w.data(), w.size() * sizeof(cplx), cudaMemcpyHostToDevice);
    return ctx;
}

void tac_ctx_destroy(tac_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (void* p : {(void*)ctx->bsk_f, (void*)ctx->ksk, (void*)ctx->pfpksk, (void*)ctx->ks_corr, (void*)ctx->pfks_corr, (void*)ctx->pfks_planes, (void*)ctx->ks_planes, (void*)ctx->pfks_fix, (void*)ctx->wT,
                    (void*)ctx->key_sched, (void*)ctx->inv_key_sched, (void*)ctx->rc_rows})
        if (p) cudaFree(p);
    for (auto& l : ctx->luts) cudaFree(l.dev);
    for (DevBuf* b : {&ctx->ws_in, &ctx->ws_out, &ctx->ws_small, &ctx->ws_ksdig, &ctx->ws_pbs, &ctx->ws_pfdig, &ctx->ws_ggsw, &ctx->ws_ggswf,
                      &ctx->ws_tree_a, &ctx->ws_tree_b, &ctx->ws_state, &ctx->ws_muls, &ctx->ws_misc, &ctx->ws_plan, &ctx->ws_rep})
        if (b->p) cudaFree(b->p);
    for (auto& r : ctx->prof_pool) for (auto& ev : r.ev) cudaEventDestroy(ev);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
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
    CU(cudaMalloc(&ctx->bsk_f, ctx->bsk_cplx() * sizeof(cplx)));
    CU(cudaMalloc(&ctx->ksk, ctx->ksk_words() * 8));
    CU(cudaMalloc(&ctx->pfpksk, ctx->pfpksk_words() * 8));
    CU(cudaMalloc(&ctx->ks_corr, (size_t)(ctx->p.n + 1) * 8));
    CU(cudaMalloc(&ctx->pfks_corr, (size_t)ctx->G() * ctx->G() * ctx->p.N * 8));
    {
        const int Kd = (ctx->big() + 1) * ctx->p.pfks_l, nkb = (Kd + UG_KB - 1) / UG_KB;
        const int W = ctx->G() * ctx->p.N, tiles = (W + UG_NT - 1) / UG_NT;
        CU(cudaMalloc(&ctx->pfks_planes, (size_t)ctx->G() * tiles * nkb * UG_B_BYTES));
        CU(cudaMalloc(&ctx->pfks_fix, 8 + (size_t)kFixCap * 8));
        const int Kd_ks = ctx->big() * ctx->p.ks_l, nkb_ks = (Kd_ks + UG_KB - 1) / UG_KB, tiles_ks = (ctx->p.n + 1 + UG_NT - 1) / UG_NT;
        CU(cudaMalloc(&ctx->ks_planes, (size_t)tiles_ks * nkb_ks * UG_B_BYTES));
    }
    ctx->keys_allocated = true;
    return TAC_OK;
}
int tac_ctx_key_buffer(tac_ctx* ctx, int which, void** dev_ptr, size_t* bytes) {
    LOCK(ctx);
    if (!ctx->keys_allocated) return fail(ctx, TAC_ERR_STATE, "key buffers not allocated");
    switch (which) {
        case 0: *dev_ptr = ctx->bsk_f; *bytes = ctx->bsk_cplx() * sizeof(cplx); return TAC_OK;
        case 1: *dev_ptr = ctx->ksk; *bytes = ctx->ksk_words() * 8; return TAC_OK;
        case 2: *dev_ptr = ctx->pfpksk; *bytes = ctx->pfpksk_words() * 8; return TAC_OK;
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
    TRY(gemm(ctx, ctx->ws_misc.as<uint32_t>(), 1, Kd_ks, ctx->ksk, p.n + 1, 1, nullptr, nullptr, 0, ctx->ks_corr));
    negate_kernel<<<grid1d(p.n + 1, 256, ctx->sm_count), 256, 0, ctx->stream>>>(ctx->ks_corr, (size_t)p.n + 1);
    TRY(post_launch(ctx, "negate_kernel"));
    CU(cudaStreamSynchronize(ctx->stream));
    std::fill(h.begin(), h.end(), 1u << (p.pfks_b - 1));
    CU(cudaMemcpyAsync(ctx->ws_misc.p, h.data(), (size_t)Kd_pf * 4, cudaMemcpyHostToDevice, ctx->stream));
    const size_t W = (size_t)ctx->G() * p.N;
    TRY(gemm(ctx, ctx->ws_misc.as<uint32_t>(), 1, Kd_pf, ctx->pfpksk, (int)W, ctx->G(), nullptr, nullptr, 0, ctx->pfks_corr));
    negate_kernel<<<grid1d(W * ctx->G(), 256, ctx->sm_count), 256, 0, ctx->stream>>>(ctx->pfks_corr, W * ctx->G());
    TRY(post_launch(ctx, "negate_kernel"));
    CU(cudaStreamSynchronize(ctx->stream));
    {   // byte-plane tiles of the PFPKSK and the KSK for the tcgen05 GEMM
        const int nkb = (Kd_pf + UG_KB - 1) / UG_KB, tiles = ((int)W + UG_NT - 1) / UG_NT;
        const size_t units = (size_t)ctx->G() * tiles * nkb * 2 * UG_NT;
        umma_key_tiles_kernel<<<grid1d(units, 256, ctx->sm_count), 256, 0, ctx->stream>>>(ctx->pfpksk, ctx->G(), Kd_pf, (int)W, nkb, ctx->pfks_planes);
        TRY(post_launch(ctx, "umma_key_tiles_kernel(pfks)"));
        const int nkb_ks = (Kd_ks + UG_KB - 1) / UG_KB, tiles_ks = (p.n + 1 + UG_NT - 1) / UG_NT;
        const size_t units_ks = (size_t)tiles_ks * nkb_ks * 2 * UG_NT;
        umma_key_tiles_kernel<<<grid1d(units_ks, 256, ctx->sm_count), 256, 0, ctx->stream>>>(ctx->ksk, 1, Kd_ks, p.n + 1, nkb_ks, ctx->ks_planes);
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
    CU(cudaMemcpyAsync(ctx->ksk, ksk, ctx->ksk_words() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->pfpksk, pfpksk, ctx->pfpksk_words() * 8, cudaMemcpyHostToDevice, ctx->stream));
    // BSK: standard → Fourier on the device, in slices ([U] fft64/crypto/bootstrap.rs::fill_with_forward_fourier)
    const size_t polys = (size_t)p.n * p.pbs_l * ctx->G() * ctx->G();
    const size_t slice = 16384;
    TRY(ensure(ctx, ctx->ws_misc, slice * p.N * 8));
    for (size_t q = 0; q < polys; q += slice) {
        const size_t cnt = std::min(slice, polys - q);
        CU(cudaMemcpyAsync(ctx->ws_misc.p, bsk_std + q * p.N, cnt * p.N * 8, cudaMemcpyHostToDevice, ctx->stream));
        TRY(poly_fft(ctx, ctx->ws_misc.as<uint64_t>(), cnt, ctx->bsk_f + q * (p.N / 2)));
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
    const size_t bytes = (size_t)44 * 32 * (ctx->big() + 1) * 8;
    if (!ctx->key_sched) CU(cudaMalloc(&ctx->key_sched, bytes));
    ctx->inv_key_sched_valid = false;        // an inverse schedule belongs to the encryption schedule it was made from
    if (ks_host) {
        CU(cudaMemcpyAsync(ctx->key_sched, ks_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    return TAC_OK;
}
int tac_aes_key_schedule_buffer(tac_ctx* ctx, void** dev_ptr, size_t* bytes) {
    LOCK(ctx);
    TRY(tac_aes_set_key_schedule(ctx, nullptr));
    *dev_ptr = ctx->key_sched; *bytes = (size_t)44 * 32 * (ctx->big() + 1) * 8;
    return TAC_OK;
}

int tac_aes_encrypt_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_dev, uint64_t* out_dev) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!ctx->key_sched) return fail(ctx, TAC_ERR_STATE, "no key schedule on the device (tac_aes_set_key_schedule)");
    return aes_blocks_dev(ctx, AesDir::Forward, n_blocks, rounds, in_noise_sq, in_dev, nullptr, nullptr, out_dev);
}
int tac_aes_encrypt_blocks(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_host, uint64_t* out_host) {
    return aes_blocks_host(ctx, n_blocks, true, in_host, out_host, [&](const uint64_t* in, uint64_t* out) {
        return tac_aes_encrypt_blocks_dev(ctx, n_blocks, rounds, in_noise_sq, in, out);
    });
}

int tac_aes_encrypt_public_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_dev) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!ctx->key_sched) return fail(ctx, TAC_ERR_STATE, "no key schedule on the device (tac_aes_set_key_schedule)");
    return aes_blocks_dev(ctx, AesDir::Forward, n_blocks, rounds, 0, nullptr, blocks_host, xor_host, out_dev);   // trivial input: no noise of its own
}
int tac_aes_encrypt_public_blocks(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_host) {
    return aes_blocks_host(ctx, n_blocks, false, nullptr, out_host, [&](const uint64_t*, uint64_t* out) {
        return tac_aes_encrypt_public_blocks_dev(ctx, n_blocks, rounds, blocks_host, xor_host, out);
    });
}

// ------------------------------------------------------------------------------------ AES decryption (FIPS-197 §5.3.5)
// Equivalent inverse cipher (aes_blocks_dev, AesDir::Inverse).  InvS·{14, 11, 13, 9} comes out of one 8 → 32 circuit
// bootstrap per byte, so a middle round sums 4 outputs of squared noise 8 and one round key of level 1: 33, as in the
// forward direction.  Round keys are read from dk only.
int tac_aes_decrypt_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_dev, uint64_t* out_dev) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    TRY(inv_key_sched_check(ctx));
    return aes_blocks_dev(ctx, AesDir::Inverse, n_blocks, rounds, in_noise_sq, in_dev, nullptr, nullptr, out_dev);
}
int tac_aes_decrypt_blocks(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_host, uint64_t* out_host) {
    return aes_blocks_host(ctx, n_blocks, true, in_host, out_host, [&](const uint64_t* in, uint64_t* out) {
        return tac_aes_decrypt_blocks_dev(ctx, n_blocks, rounds, in_noise_sq, in, out);
    });
}

// decryption of PUBLIC ciphertext blocks (AES-ECB / AES-CBC transciphering): state0 = dk[40..43] + trivial(block), the
// plan runs along the inverse dependence rule, xor_host (the previous ciphertext blocks for CBC) joins the final round
int tac_aes_decrypt_public_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_dev) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    TRY(inv_key_sched_check(ctx));
    return aes_blocks_dev(ctx, AesDir::Inverse, n_blocks, rounds, 0, nullptr, blocks_host, xor_host, out_dev);   // trivial input: no noise of its own
}
int tac_aes_decrypt_public_blocks(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_host) {
    return aes_blocks_host(ctx, n_blocks, false, nullptr, out_host, [&](const uint64_t*, uint64_t* out) {
        return tac_aes_decrypt_public_blocks_dev(ctx, n_blocks, rounds, blocks_host, xor_host, out);
    });
}

// inverse key schedule on the device from the resident encryption schedule: dk[0..3] = w[0..3], dk[40..43] = w[40..43],
// dk[4rd..4rd+3] = InvMixColumns(w[4rd..4rd+3]) for rd = 1..9.  One 8 → 32 circuit bootstrap (b·{14, 11, 13, 9}) of the
// 144 key bytes, the InvMixColumns sums (squared noise 32), then one 1-bit bootstrap per sum bit back to level 1 (as
// boot_word does in the forward key schedule).
int tac_aes_inv_key_schedule(tac_ctx* ctx, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!ctx->key_sched) return fail(ctx, TAC_ERR_STATE, "no key schedule on the device (tac_aes_set_key_schedule)");
    if (4 * 8 > ctx->p.max_noise_sq) return fail(ctx, TAC_ERR_NOISE, "NoiseTooBig: the inverse key schedule needs max_noise_level_squared >= 32");
    TRY(ensure_aes_luts(ctx));
    TRY(ensure_aes_inv_luts(ctx));
    const size_t L = (size_t)ctx->big() + 1, byte = 8 * L, word = 4 * byte, bytes = 44 * word * 8;
    const int n_key_bytes = 9 * 16;                          // round keys 1..9
    if (!ctx->inv_key_sched) CU(cudaMalloc(&ctx->inv_key_sched, bytes));
    ctx->inv_key_sched_valid = false;
    uint64_t* dk = ctx->inv_key_sched;
    const uint64_t* w = ctx->key_sched;
    TRY(ensure(ctx, ctx->ws_muls, (size_t)n_key_bytes * 32 * L * 8));
    TRY(ensure(ctx, ctx->ws_state, (size_t)n_key_bytes * byte * 8));
    CU(cudaMemcpyAsync(dk, w, 4 * word * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    CU(cudaMemcpyAsync(dk + 40 * word, w + 40 * word, 4 * word * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    uint64_t* muls = ctx->ws_muls.as<uint64_t>();
    uint64_t* sums = ctx->ws_state.as<uint64_t>();
    TRY(wopbs_dev(ctx, ctx->luts[ctx->aes_lut_key32], n_key_bytes, w + 4 * word, muls));
    const size_t total = (size_t)n_key_bytes * byte;
    aes_inv_mix_key_kernel<<<grid1d(total, 256, ctx->sm_count), 256, 0, ctx->stream>>>(muls, (int)L, total, sums);
    TRY(post_launch(ctx, "aes_inv_mix_key_kernel"));
    TRY(wopbs_dev(ctx, ctx->luts[ctx->aes_lut1], n_key_bytes * 8, sums, dk + 4 * word));
    if (out_host) CU(cudaMemcpyAsync(out_host, dk, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->inv_key_sched_valid = true;
    return TAC_OK;
}
int tac_aes_set_inv_key_schedule(tac_ctx* ctx, const uint64_t* dk_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (!dk_host) return fail(ctx, TAC_ERR_ARG, "NULL inverse key schedule");
    const size_t bytes = (size_t)44 * 32 * (ctx->big() + 1) * 8;
    if (!ctx->inv_key_sched) CU(cudaMalloc(&ctx->inv_key_sched, bytes));
    ctx->inv_key_sched_valid = false;
    CU(cudaMemcpyAsync(ctx->inv_key_sched, dk_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->inv_key_sched_valid = true;
    return TAC_OK;
}

// fhe_sbox_gal_mul_pbs::key_schedule (:134-164) with boot_word (:166-180) and sub_word (:182-191) on the device
int tac_aes_key_schedule(tac_ctx* ctx, const uint64_t* key_bits_host, uint64_t* out_host) {
    LOCK(ctx);
    CU(cudaSetDevice(ctx->device));
    if (8 + 1 > ctx->p.max_noise_sq) return fail(ctx, TAC_ERR_NOISE, "NoiseTooBig: key schedule needs max_noise_level_squared >= 9");
    TRY(ensure_aes_luts(ctx));
    TRY(tac_aes_set_key_schedule(ctx, nullptr));
    const size_t L = (size_t)ctx->big() + 1, byte = 8 * L, word = 4 * byte;
    uint64_t* ek = ctx->key_sched;
    TRY(ensure(ctx, ctx->ws_state, 3 * word * 8));
    uint64_t* rot = ctx->ws_state.as<uint64_t>();       // rotated previous word / its SBOX image
    uint64_t* sub = rot + word;
    uint64_t* acc = sub + word;
    CU(cudaMemcpyAsync(ek, key_bits_host, 4 * word * 8, cudaMemcpyHostToDevice, ctx->stream));
    // trivial(RC) constants: body += encode_bit(1) on the set bits of RC[i/4], byte 0 (:154; Byte::trivial data_model.rs:35-43).
    // All ten rows are uploaded once per context, so the 40 steps below enqueue without a host synchronisation.
    if (!ctx->rc_rows) {
        static const uint8_t RC[11] = {0x00, 0x01, 0x02, 0x04, 0x08, 0x10, 0x20, 0x40, 0x80, 0x1B, 0x36};
        std::vector<uint64_t> rows((size_t)10 * byte, 0ull);
        for (int r = 1; r <= 10; r++)
            for (int bit = 0; bit < 8; bit++)
                if (RC[r] & (0x80 >> bit)) rows[(size_t)(r - 1) * byte + (size_t)bit * L + (L - 1)] = tac_encode_bit(1);
        CU(cudaMalloc(&ctx->rc_rows, rows.size() * 8));
        CU(cudaMemcpy(ctx->rc_rows, rows.data(), rows.size() * 8, cudaMemcpyHostToDevice));
    }
    for (int i = 4; i < 44; i++) {
        uint64_t* cur = ek + (size_t)i * word;
        const uint64_t* prev = ek + (size_t)(i - 1) * word;
        const uint64_t* addend = prev;
        if (i % 4 == 0) {
            // rotate_left(1): bytes [1,2,3,0]
            CU(cudaMemcpyAsync(rot, prev + byte, 3 * byte * 8, cudaMemcpyDeviceToDevice, ctx->stream));
            CU(cudaMemcpyAsync(rot + 3 * byte, prev, byte * 8, cudaMemcpyDeviceToDevice, ctx->stream));
            TRY(wopbs_dev(ctx, ctx->luts[ctx->aes_lut8], 4, rot, sub));                                       // sub_word
            TRY(tac_lwe_add_batch_dev(ctx, sub, ctx->rc_rows + (size_t)(i / 4 - 1) * byte, 8));
            addend = sub;
        }
        CU(cudaMemcpyAsync(acc, ek + (size_t)(i - 4) * word, word * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        TRY(tac_lwe_add_batch_dev(ctx, acc, addend, 32));
        TRY(wopbs_dev(ctx, ctx->luts[ctx->aes_lut1], 32, acc, cur));                                          // boot_word → bootstrap_assign
    }
    if (out_host) CU(cudaMemcpyAsync(out_host, ek, 44 * word * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return TAC_OK;
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
