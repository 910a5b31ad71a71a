// libvqa_b200.so -- C ABI + host-side orchestration of the CLIP-FlanT5 VQAScore forward on one B200.
// The forward is a fixed sequence of kernel launches on the caller's stream; no torch, no cuBLAS.
#include "../../include/vqa_b200.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <unordered_map>
#include <vector>

#include "ptx.cuh"
#include "gemm_sm100.cuh"
#include "elementwise.cuh"
#include "attention.cuh"
#include "attention_sm100.cuh"
#include "qwen_kernels.cuh"
#include "preprocess.cuh"

using namespace vqa;
typedef __nv_bfloat16 bf16;

// bits of vqa_clipt5_config::emulate_bf16_rounding (see include/vqa_b200.h)
constexpr int VQA_FLAG_ROUND_DECODER = 1, VQA_FLAG_ROUND_ATTN_SCORES = 2, VQA_FLAG_FUSE_NORMS = 4;

// ------------------------------------------------------------------------------------------------ handle
struct BoundTensor {
    const void* data = nullptr;
    int64_t shape[4] = {0, 0, 0, 0};
    int ndim = 0;
    int dtype = 0;
};

struct VitLayerW {
    const bf16 *ln1_w, *ln1_b, *qkv_w, *qkv_b, *out_w, *out_b, *ln2_w, *ln2_b, *fc1_w, *fc1_b, *fc2_w, *fc2_b;
};
struct T5EncLayerW {
    const bf16 *ln0, *qkv, *o, *ln1, *wi, *wo;
    const bf16 *qkv_g = nullptr, *wi_g = nullptr;   // fused-norm mode: qkv . diag(ln0), wi . diag(ln1) (gamma folded into the weight's K axis)
};
struct T5DecLayerW {
    const bf16 *ln0, *qkv, *o, *ln1, *cq, *ckv, *co, *ln2, *wi, *wo;
    const bf16* ckT;   // Wk^T [d_model, inner] for the absorbed cross-attention (optional)
};

struct QwenState;
struct vqa_handle {
    int kind = 0;               // 0: CLIP-FlanT5, 1: Qwen2.5-VL
    QwenState* qwen = nullptr;
    vqa_clipt5_config cfg;
    int device = 0;
    int num_sms = 148;
    std::string err;
    std::unordered_map<std::string, BoundTensor> tensors;
    bool finalized = false;
    int64_t launches = 0;
    int kpad = 0;  // padded K of the patch-embedding GEMM
    // resolved weights
    const bf16 *patch_w = nullptr, *cls = nullptr, *pos = nullptr, *pre_ln_w = nullptr, *pre_ln_b = nullptr;
    std::vector<VitLayerW> vit;
    const bf16 *proj0_w = nullptr, *proj0_b = nullptr, *proj2_w = nullptr, *proj2_b = nullptr;
    const bf16 *shared = nullptr, *enc_rel = nullptr, *dec_rel = nullptr, *enc_final_ln = nullptr,
               *dec_final_ln = nullptr, *lm_head = nullptr;
    std::vector<T5EncLayerW> enc;
    std::vector<T5DecLayerW> dec;
    // relative-position bucket LUTs (device), index rel + max_dist, rel clamped to [-max_dist, max_dist]
    int* lut_bidir = nullptr;
    int* lut_unidir = nullptr;
    // optional per-category device timing (vqa_set_profile): CUDA events around every launch of the forward
    bool profile = false;
    std::vector<cudaEvent_t> ev_pool;
    struct ProfRec { int cat; double flops; double bytes; int ev0, ev1; };
    std::vector<ProfRec> prof;
    size_t ev_used = 0;
};

enum ProfCat { CAT_GEMM = 0, CAT_ATTENTION = 1, CAT_NORM = 2, CAT_OTHER = 3, CAT_COUNT = 4 };

// Records an event pair around the launches issued in its lifetime (only in profile mode).
struct ProfScope {
    vqa_handle* h; cudaStream_t st; int idx = -1;
    ProfScope(vqa_handle* h_, int cat, double flops, cudaStream_t st_, double bytes = 0.0) : h(h_), st(st_) {
        if (!h->profile) return;
        while (h->ev_pool.size() < h->ev_used + 2) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) return;
            h->ev_pool.push_back(e);
        }
        vqa_handle::ProfRec r{cat, flops, bytes, (int)h->ev_used, (int)h->ev_used + 1};
        h->ev_used += 2;
        cudaEventRecord(h->ev_pool[r.ev0], st);
        idx = (int)h->prof.size();
        h->prof.push_back(r);
    }
    ~ProfScope() {
        if (idx >= 0) cudaEventRecord(h->ev_pool[h->prof[idx].ev1], st);
    }
};

static thread_local std::string g_global_err;

static int fail(vqa_handle* h, int code, const std::string& msg) {
    if (h) h->err = msg; else g_global_err = msg;
    return code;
}
#define PROF(h, cat, flops, st, expr)              \
    do {                                           \
        ProfScope _ps(h, cat, flops, st);          \
        CUDA_TRY(h, expr);                         \
    } while (0)
#define CUDA_TRY(h, expr)                                                                          \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return fail(h, VQA_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));      \
    } while (0)

// ------------------------------------------------------------------------------------------------ GEMM dispatch
static int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && v[0]) ? atoi(v) : dflt;
}

template <int EPI>
static cudaError_t gemm_dispatch_variant(const GemmLaunch& g, int variant, int num_sms, cudaStream_t st) {
    switch (variant) {
        case 2562: return launch_gemm_t<256, 2, EPI>(g, num_sms, st);
        case 2561: return launch_gemm_t<256, 1, EPI>(g, num_sms, st);
        case 1282: return launch_gemm_t<128, 2, EPI>(g, num_sms, st);
        case 1281: return launch_gemm_t<128, 1, EPI>(g, num_sms, st);
        case 641:  return launch_gemm_t<64, 1, EPI>(g, num_sms, st);
        case 321:
            if constexpr (epi_is_gated(EPI)) return cudaErrorInvalidValue;
            else return launch_gemm_t<32, 1, EPI>(g, num_sms, st);
        default:   return cudaErrorInvalidValue;
    }
}

static int pick_variant(int M, int N, int epi) {
    static const int forced = env_int("VQA_GEMM_VARIANT", 0);
    if (forced) return forced;
    if (M <= 128) {
        // skinny (decoder rows): pure weight streaming; favour many CTAs. The gated epilogue pairs two half tiles of
        // BLOCK_N/2 >= 32 columns, so it needs BLOCK_N >= 64.
        if (epi_is_gated(epi)) return N <= 16384 ? 641 : 1281;
        if (N <= 4096) return 321;
        if (N <= 12288) return 641;
        return 1281;
    }
    if (M <= 256 * 16 && N <= 1024) return 1281;
    return 2562;
}

// partial sums per row that a residual-writing GEMM with this tile variant emits for N output columns (GemmParams::ssq_out)
static int ssq_parts_for(int variant, int N) {
    switch (variant) {
        case 2562: return gemm_ssq_parts<256, 2>(N);
        case 2561: return gemm_ssq_parts<256, 1>(N);
        case 1282: return gemm_ssq_parts<128, 2>(N);
        case 1281: return gemm_ssq_parts<128, 1>(N);
        case 641:  return gemm_ssq_parts<64, 1>(N);
        default:   return gemm_ssq_parts<32, 1>(N);
    }
}

// Sum of squares of every row of x (bf16 [rows, D]) into slot 0 of its partial-sum row (the other slots are zero): seeds the fused
// RMSNorm chain for the encoder's input embeddings. One warp per row.
__global__ void __launch_bounds__(256) row_ssq_kernel(const bf16* __restrict__ x, float* __restrict__ ssq, int rows, int D, int stride) {
    pdl_launch_dependents();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const uint4* xr = reinterpret_cast<const uint4*>(x + (size_t)row * D);
    float ss = 0.f;
    for (int i = lane; i < D / 8; i += 32) {
        const uint4 v = xr[i];
        const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 f = unpack_bf16x2(u[e]);
            ss = fmaf(f.x, f.x, ss);
            ss = fmaf(f.y, f.y, ss);
        }
    }
    ss = warp_sum(ss);
    if (lane == 0) ssq[(size_t)row * stride] = ss;
}

// Launch C = epi(A W^T). Returns cudaError_t. `launch_counter` is incremented per kernel.
struct NormFuse {            // fused RMSNorm hooks of one GEMM launch (see GemmParams::ssq_*)
    float* ssq_out = nullptr;       // producer: partial sums of squares of the rows this GEMM writes ([M, ssq_stride])
    const float* ssq_in = nullptr;  // consumer: partial sums of the rows of A
    int stride = 0;                 // floats per row in both buffers (multiple of 4; unused slots are zero)
    float inv_dim = 0.f, eps = 0.f;
};
static cudaError_t run_gemm(const bf16* A, int lda, const bf16* W, int ldw, int w_rows, bf16* C, int ldc, int M, int N,
                            int K, const bf16* bias, const bf16* residual, int ldr, int epi, int gate_up_offset,
                            int variant, int num_sms, cudaStream_t st, int64_t* launch_counter, bool c_f32 = false,
                            const NormFuse* nf = nullptr, int c_group_in = 0, int c_group_out = 0) {
    GemmLaunch g;
    g.A = A; g.lda = lda; g.W = W; g.ldw = ldw; g.w_rows = w_rows;
    memset(&g.p, 0, sizeof(g.p));
    g.p.M = M; g.p.N = N; g.p.K = K; g.p.C = C; g.p.ldc = ldc; g.p.bias = bias; g.p.residual = residual;
    g.p.ldr = ldr; g.p.gate_up_offset = gate_up_offset;
    if (c_f32 && epi != EPI_STORE) return cudaErrorInvalidValue;
    g.p.c_f32 = c_f32 ? 1 : 0;
    if (c_group_in > 0) {   // narrow output column groups written into wider slots (GemmParams::c_group_in)
        if (epi != EPI_STORE || residual || c_f32 || (c_group_in & 7) || (c_group_out & 7) || c_group_out < c_group_in || N % c_group_in)
            return cudaErrorInvalidValue;
        g.p.c_group_in = c_group_in; g.p.c_group_out = c_group_out;
    }
    if (nf) {
        g.p.ssq_out = nf->ssq_out; g.p.ssq_in = nf->ssq_in; g.p.ssq_out_parts = g.p.ssq_in_parts = nf->stride;
        g.p.ssq_inv_dim = nf->inv_dim; g.p.ssq_eps = nf->eps;
        if (nf->ssq_out && (epi != EPI_STORE || c_f32)) return cudaErrorInvalidValue;
    }
    if (launch_counter) ++*launch_counter;
    if (variant == 0) variant = pick_variant(M, N, epi);
    switch (epi) {
        case EPI_STORE:      return gemm_dispatch_variant<EPI_STORE>(g, variant, num_sms, st);
        case EPI_QUICK_GELU: return gemm_dispatch_variant<EPI_QUICK_GELU>(g, variant, num_sms, st);
        case EPI_GELU_ERF:   return gemm_dispatch_variant<EPI_GELU_ERF>(g, variant, num_sms, st);
        case EPI_GATED_GELU: return gemm_dispatch_variant<EPI_GATED_GELU>(g, variant, num_sms, st);
        case EPI_RELU:       return gemm_dispatch_variant<EPI_RELU>(g, variant, num_sms, st);
        case EPI_GATED_SILU: return gemm_dispatch_variant<EPI_GATED_SILU>(g, variant, num_sms, st);
        default:             return cudaErrorInvalidValue;
    }
}

// Batched launch: `nb` independent GEMMs sharing one tensor map per operand (see GemmParams::num_batches).
struct BatchSpec {
    int nb; int a_row_off, a_k_off, w_row_off, w_k_off; long long c_stride;
    long long a_rows, a_cols, w_rows, w_cols;   // full extents visible to TMA
};
static cudaError_t run_gemm_batched(const bf16* A, int lda, const bf16* W, int ldw, bf16* C, int ldc, int M, int N, int K,
                                    const BatchSpec& bs, int variant, int num_sms, cudaStream_t st, int64_t* launch_counter) {
    GemmLaunch g;
    g.A = A; g.lda = lda; g.W = W; g.ldw = ldw; g.w_rows = (int)bs.w_rows;
    g.a_rows = bs.a_rows; g.a_cols = bs.a_cols; g.w_cols = bs.w_cols;
    memset(&g.p, 0, sizeof(g.p));
    g.p.M = M; g.p.N = N; g.p.K = K; g.p.C = C; g.p.ldc = ldc;
    g.p.num_batches = bs.nb; g.p.a_row_off = bs.a_row_off; g.p.a_k_off = bs.a_k_off; g.p.w_row_off = bs.w_row_off;
    g.p.w_k_off = bs.w_k_off; g.p.c_batch_stride = bs.c_stride;
    if (launch_counter) ++*launch_counter;
    return gemm_dispatch_variant<EPI_STORE>(g, variant, num_sms, st);
}

// Split-K for skinny GEMMs (M <= 128 decoder rows x a 4096-row weight): 32 N tiles alone leave 116 SMs idle and stream the weight at ~1 TB/s
// (profiles/r02_small_batch.md), so the K range is cut into `splits` slices that run as the batches of ONE launch (fp32 partial tiles in `ws`),
// and this kernel adds the slices: C = [residual +] bf16(sum_s partial_s + bias) -- the Linear's bf16 output, then the residual add, like EPI_STORE.
__global__ void splitk_reduce_kernel(const float* __restrict__ part, int splits, int M, int N, const bf16* __restrict__ bias,
                                     const bf16* __restrict__ residual, int ldr, bf16* __restrict__ C, int ldc) {
    pdl_launch_dependents();
    const int nv = N / 8;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)M * nv) return;
    const int m = (int)(i / nv), n = (int)(i % nv) * 8;
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int s = 0; s < splits; ++s) {
        const float4* src = reinterpret_cast<const float4*>(part + ((size_t)s * M + m) * N + n);
        const float4 a = src[0], b = src[1];
        acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w; acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
    }
    if (bias) {
        const uint4 bb = __ldg(reinterpret_cast<const uint4*>(bias + n));
        const float2 b0 = unpack_bf16x2(bb.x), b1 = unpack_bf16x2(bb.y), b2 = unpack_bf16x2(bb.z), b3 = unpack_bf16x2(bb.w);
        acc[0] += b0.x; acc[1] += b0.y; acc[2] += b1.x; acc[3] += b1.y; acc[4] += b2.x; acc[5] += b2.y; acc[6] += b3.x; acc[7] += b3.y;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = bf16_round(acc[e]);
    if (residual) {
        const uint4 rr = *reinterpret_cast<const uint4*>(residual + (size_t)m * ldr + n);
        const float2 r0 = unpack_bf16x2(rr.x), r1 = unpack_bf16x2(rr.y), r2 = unpack_bf16x2(rr.z), r3 = unpack_bf16x2(rr.w);
        acc[0] += r0.x; acc[1] += r0.y; acc[2] += r1.x; acc[3] += r1.y; acc[4] += r2.x; acc[5] += r2.y; acc[6] += r3.x; acc[7] += r3.y;
    }
    *reinterpret_cast<uint4*>(C + (size_t)m * ldc + n) = make_uint4(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]),
                                                                     pack_bf16x2(acc[4], acc[5]), pack_bf16x2(acc[6], acc[7]));
}

// number of K slices a skinny store-GEMM is cut into (1 = not worth it / not possible)
static int splitk_slices(int M, int N, int K, int num_sms) {
    static const int off = env_int("VQA_GEMM_SPLITK", 1) == 0;
    if (off || M > 128 || N % 8 || K < 2048) return 1;
    const int n_tiles = (N + 127) / 128;
    int s = num_sms / n_tiles;
    if (s > 8) s = 8;
    while (s >= 2 && K % (s * 64) != 0) --s;
    return s >= 2 ? s : 1;
}
static size_t splitk_workspace_bytes(int M, int N, int K, int num_sms) {
    const int s = splitk_slices(M, N, K, num_sms);
    return s > 1 ? (size_t)s * M * N * 4 : 0;
}
static cudaError_t run_gemm_splitk(const bf16* A, int lda, const bf16* W, int ldw, int w_rows, bf16* C, int ldc, int M, int N, int K,
                                   const bf16* bias, const bf16* residual, int ldr, int splits, float* ws, int num_sms, cudaStream_t st,
                                   int64_t* launch_counter) {
    GemmLaunch g;
    g.A = A; g.lda = lda; g.W = W; g.ldw = ldw; g.w_rows = w_rows;
    g.a_rows = M; g.a_cols = K; g.w_cols = K;
    memset(&g.p, 0, sizeof(g.p));
    const int Ks = K / splits;
    g.p.M = M; g.p.N = N; g.p.K = Ks; g.p.C = reinterpret_cast<bf16*>(ws); g.p.ldc = N; g.p.c_f32 = 2;
    g.p.num_batches = splits; g.p.a_k_off = Ks; g.p.w_k_off = Ks; g.p.c_batch_stride = (long long)M * N;
    if (launch_counter) *launch_counter += 2;
    cudaError_t e = gemm_dispatch_variant<EPI_STORE>(g, 1281, num_sms, st);
    if (e != cudaSuccess) return e;
    const long long n = (long long)M * (N / 8);
    splitk_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ws, splits, M, N, bias, residual, ldr, C, ldc);
    return cudaGetLastError();
}

constexpr int LMHEAD_BN = 128;
constexpr int LMHEAD_PARTS = GemmConfig<LMHEAD_BN, 1>::LSE_PARTS;   // (max, sum) partials per (row, n tile)
static cudaError_t run_lmhead(const bf16* H, int ldh, const bf16* W, int ldw, int M, int N, int K, const int* labels,
                              float* lse_max, float* lse_sum, float* label_logit, int num_sms, cudaStream_t st,
                              int64_t* launch_counter, float logit_scale = 1.0f, const uint32_t* penalty_bitmap = nullptr,
                              int penalty_words = 0, float penalty = 1.0f) {
    GemmLaunch g;
    g.A = H; g.lda = ldh; g.W = W; g.ldw = ldw; g.w_rows = N;
    memset(&g.p, 0, sizeof(g.p));
    g.p.M = M; g.p.N = N; g.p.K = K;
    g.p.lse_max = lse_max; g.p.lse_sum = lse_sum; g.p.labels = labels; g.p.label_logit = label_logit;
    g.p.lse_scale = logit_scale;
    g.p.penalty_bitmap = penalty_bitmap; g.p.penalty_words = penalty_words; g.p.penalty = penalty;
    if (launch_counter) ++*launch_counter;
    return launch_gemm_t<LMHEAD_BN, 1, EPI_LSE>(g, num_sms, st);
}

static cudaError_t run_rmsnorm(const bf16* x, const bf16* w, bf16* y, int rows, int D, float eps, cudaStream_t st,
                               int64_t* lc) {
    if (lc) ++*lc;
    if (rows <= 0) return cudaSuccess;
    if (D % 256 == 0 && D < 4096) {
        const int blocks = (rows + 7) / 8;      // one warp per row
#define VQA_RMS_CASE(NV) case NV: t5_rmsnorm_warp_kernel<NV><<<blocks, 256, 0, st>>>(x, w, y, rows, eps); break;
        switch (D / 256) {
            VQA_RMS_CASE(1) VQA_RMS_CASE(2) VQA_RMS_CASE(3) VQA_RMS_CASE(4) VQA_RMS_CASE(5) VQA_RMS_CASE(6) VQA_RMS_CASE(7) VQA_RMS_CASE(8)
            VQA_RMS_CASE(9) VQA_RMS_CASE(10) VQA_RMS_CASE(11) VQA_RMS_CASE(12) VQA_RMS_CASE(13) VQA_RMS_CASE(14) VQA_RMS_CASE(15)
        }
#undef VQA_RMS_CASE
        return cudaGetLastError();
    }
    const int nvec = D / 8;
    if (D % 8) return cudaErrorInvalidValue;
    if (nvec <= 256)       t5_rmsnorm_kernel<1><<<rows, 256, 0, st>>>(x, w, y, D, eps);
    else if (nvec <= 512)  t5_rmsnorm_kernel<2><<<rows, 256, 0, st>>>(x, w, y, D, eps);
    else if (nvec <= 1024) t5_rmsnorm_kernel<4><<<rows, 256, 0, st>>>(x, w, y, D, eps);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}
// LayerNorm of an fp32 stream (the CLIP residual under autocast) -> bf16
static cudaError_t run_layernorm_f32(const float* x, const bf16* g, const bf16* b, bf16* y, int rows, int D, float eps,
                                     cudaStream_t st, int64_t* lc) {
    if (lc) ++*lc;
    const int blocks = (rows + 7) / 8;
    if (D == 1024)      layernorm_kernel<1024, float><<<blocks, 256, 0, st>>>(x, g, b, y, rows, eps);
    else if (D == 256)  layernorm_kernel<256, float><<<blocks, 256, 0, st>>>(x, g, b, y, rows, eps);
    else if (D == 512)  layernorm_kernel<512, float><<<blocks, 256, 0, st>>>(x, g, b, y, rows, eps);
    else if (D == 768)  layernorm_kernel<768, float><<<blocks, 256, 0, st>>>(x, g, b, y, rows, eps);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}
static cudaError_t run_layernorm(const bf16* x, const bf16* g, const bf16* b, bf16* y, int rows, int D, float eps,
                                 cudaStream_t st, int64_t* lc) {
    if (lc) ++*lc;
    const int blocks = (rows + 7) / 8;
    if (D == 1024)      layernorm_kernel<1024><<<blocks, 256, 0, st>>>(x, g, b, y, rows, eps);
    else if (D == 256)  layernorm_kernel<256><<<blocks, 256, 0, st>>>(x, g, b, y, rows, eps);
    else if (D == 512)  layernorm_kernel<512><<<blocks, 256, 0, st>>>(x, g, b, y, rows, eps);
    else if (D == 768)  layernorm_kernel<768><<<blocks, 256, 0, st>>>(x, g, b, y, rows, eps);
    else if (D == 1280) layernorm_kernel<1280><<<blocks, 256, 0, st>>>(x, g, b, y, rows, eps);
    else return cudaErrorInvalidValue;
    return cudaGetLastError();
}
// q, k, v are column slices of one packed buffer (they always are on this path). bias_const_from: see launch_attn_tc.
static cudaError_t run_flash(const bf16* q, const bf16* k, const bf16* v, int ldqkv, bf16* o, int ldo, int B, int S,
                             int H, const int* seq_lens, const float* bias_table, float scale, int bias_const_from, bool round_scores,
                             cudaStream_t st, int64_t* lc) {
    if (lc) ++*lc;
    const int q_col0 = 0, k_col0 = (int)(k - q), v_col0 = (int)(v - q);
    return launch_attn_tc(q, ldqkv, q_col0, k_col0, v_col0, o, ldo, B, S, H, seq_lens, bias_table, scale, bias_const_from, round_scores, st);
}

// ------------------------------------------------------------------------------------------------ C ABI: lifecycle
extern "C" const char* vqa_version(void) {
    return "vqa_b200 abi=1 arch=sm_100a kernels=tcgen05-gemm,flash-d64,t5-norm,lmhead-lse";
}

// Host mirror of T5Attention._relative_position_bucket (modeling_t5.py:189-234), fp32 like torch.
static int host_rel_bucket(int rel, bool bidirectional, int num_buckets, int max_distance) {
    int bucket = 0;
    if (bidirectional) {
        num_buckets /= 2;
        if (rel > 0) bucket += num_buckets;
        rel = abs(rel);
    } else {
        rel = -std::min(rel, 0);
    }
    const int max_exact = num_buckets / 2;
    if (rel < max_exact) return bucket + rel;
    float v = logf((float)rel / (float)max_exact) / (float)log((double)max_distance / (double)max_exact) *
              (float)(num_buckets - max_exact);
    int large = max_exact + (int)v;
    large = std::min(large, num_buckets - 1);
    return bucket + large;
}

extern "C" int vqa_create_clipt5(const vqa_clipt5_config* cfg, int device, vqa_handle** out) {
    if (!cfg || !out) return fail(nullptr, VQA_ERR_INVALID_ARG, "null argument");
    if (cfg->vit_hidden % cfg->vit_heads || cfg->vit_hidden / cfg->vit_heads != 64)
        return fail(nullptr, VQA_ERR_UNSUPPORTED, "vision head_dim must be 64");
    if (cfg->image_size % cfg->patch_size) return fail(nullptr, VQA_ERR_INVALID_ARG, "image_size % patch_size != 0");
    if (cfg->d_model % 8 || cfg->d_ff % 64 || cfg->vit_hidden % 256)
        return fail(nullptr, VQA_ERR_UNSUPPORTED, "d_model % 8, d_ff % 64, vit_hidden % 256 must be 0");
    vqa_handle* h = new vqa_handle();
    h->cfg = *cfg;
    h->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) {
        g_global_err = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
        delete h;
        return VQA_ERR_CUDA;
    }
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess || prop.major != 10) {
        g_global_err = "vqa_b200 requires an sm_100 (B200) device";
        delete h;
        return VQA_ERR_UNSUPPORTED;
    }
    h->num_sms = prop.multiProcessorCount;
    const int kreal = 3 * cfg->patch_size * cfg->patch_size;
    h->kpad = (kreal + 63) / 64 * 64;
    // bucket LUTs
    const int md = cfg->rel_max_distance;
    std::vector<int> lb(2 * md + 1), lu(2 * md + 1);
    for (int r = -md; r <= md; ++r) {
        lb[r + md] = host_rel_bucket(r, true, cfg->rel_buckets, md);
        lu[r + md] = host_rel_bucket(r, false, cfg->rel_buckets, md);
    }
    if (cudaMalloc(&h->lut_bidir, lb.size() * 4) != cudaSuccess || cudaMalloc(&h->lut_unidir, lu.size() * 4) != cudaSuccess ||
        cudaMemcpy(h->lut_bidir, lb.data(), lb.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(h->lut_unidir, lu.data(), lu.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
        g_global_err = "LUT allocation failed";
        delete h;
        return VQA_ERR_CUDA;
    }
    *out = h;
    return VQA_OK;
}

extern "C" int vqa_bind_weights(vqa_handle* h, const vqa_tensor* tensors, int32_t n) {
    if (!h || (!tensors && n > 0)) return fail(h, VQA_ERR_INVALID_ARG, "null argument");
    for (int i = 0; i < n; ++i) {
        const vqa_tensor& t = tensors[i];
        if (!t.name || !t.data) return fail(h, VQA_ERR_INVALID_ARG, "tensor with null name/data");
        if (t.dtype != VQA_DTYPE_BF16) return fail(h, VQA_ERR_UNSUPPORTED, std::string(t.name) + ": weights must be bf16");
        if ((reinterpret_cast<uintptr_t>(t.data) & 15) != 0)
            return fail(h, VQA_ERR_INVALID_ARG, std::string(t.name) + ": pointer not 16-byte aligned");
        BoundTensor b;
        b.data = t.data; b.ndim = t.ndim; b.dtype = t.dtype;
        for (int d = 0; d < 4; ++d) b.shape[d] = (d < t.ndim) ? t.shape[d] : 1;
        h->tensors[t.name] = b;
    }
    h->finalized = false;
    return VQA_OK;
}

static const bf16* need(vqa_handle* h, const std::string& name, int64_t d0, int64_t d1, bool& ok) {
    auto it = h->tensors.find(name);
    if (it == h->tensors.end()) {
        if (ok) h->err = "missing weight: " + name;
        ok = false;
        return nullptr;
    }
    const BoundTensor& b = it->second;
    int64_t numel = 1;
    for (int d = 0; d < b.ndim; ++d) numel *= b.shape[d];
    if (numel != d0 * d1) {
        if (ok) {
            char buf[256];
            snprintf(buf, sizeof buf, "weight %s: expected %lld x %lld elements, got %lld", name.c_str(), (long long)d0,
                     (long long)d1, (long long)numel);
            h->err = buf;
        }
        ok = false;
        return nullptr;
    }
    return reinterpret_cast<const bf16*>(b.data);
}

static int qwen_finalize(vqa_handle* h, QwenState& q);
extern "C" int vqa_finalize_weights(vqa_handle* h) {
    if (!h) return VQA_ERR_INVALID_ARG;
    if (h->kind == 1) {
        int rc = qwen_finalize(h, *h->qwen);
        h->finalized = (rc == VQA_OK);
        return rc;
    }
    const vqa_clipt5_config& c = h->cfg;
    bool ok = true;
    const int P = (c.image_size / c.patch_size) * (c.image_size / c.patch_size);
    const int Dv = c.vit_hidden, Dm = c.d_model, inner = c.n_heads * 64;
    h->patch_w = need(h, "vit.patch_embed.weight", Dv, h->kpad, ok);
    h->cls = need(h, "vit.class_embedding", Dv, 1, ok);
    h->pos = need(h, "vit.position_embedding", P + 1, Dv, ok);
    h->pre_ln_w = need(h, "vit.pre_ln.weight", Dv, 1, ok);
    h->pre_ln_b = need(h, "vit.pre_ln.bias", Dv, 1, ok);
    h->vit.resize(c.vit_layers_run);
    for (int i = 0; i < c.vit_layers_run; ++i) {
        const std::string p = "vit.layers." + std::to_string(i) + ".";
        VitLayerW& L = h->vit[i];
        L.ln1_w = need(h, p + "ln1.weight", Dv, 1, ok); L.ln1_b = need(h, p + "ln1.bias", Dv, 1, ok);
        L.qkv_w = need(h, p + "qkv.weight", 3 * Dv, Dv, ok); L.qkv_b = need(h, p + "qkv.bias", 3 * Dv, 1, ok);
        L.out_w = need(h, p + "out.weight", Dv, Dv, ok); L.out_b = need(h, p + "out.bias", Dv, 1, ok);
        L.ln2_w = need(h, p + "ln2.weight", Dv, 1, ok); L.ln2_b = need(h, p + "ln2.bias", Dv, 1, ok);
        L.fc1_w = need(h, p + "fc1.weight", c.vit_mlp, Dv, ok); L.fc1_b = need(h, p + "fc1.bias", c.vit_mlp, 1, ok);
        L.fc2_w = need(h, p + "fc2.weight", Dv, c.vit_mlp, ok); L.fc2_b = need(h, p + "fc2.bias", Dv, 1, ok);
    }
    h->proj0_w = need(h, "proj.0.weight", Dm, Dv, ok); h->proj0_b = need(h, "proj.0.bias", Dm, 1, ok);
    h->proj2_w = need(h, "proj.2.weight", Dm, Dm, ok); h->proj2_b = need(h, "proj.2.bias", Dm, 1, ok);
    h->shared = need(h, "t5.shared", c.vocab, Dm, ok);
    h->enc_rel = need(h, "t5.enc.rel_bias", c.rel_buckets, c.n_heads, ok);
    h->dec_rel = need(h, "t5.dec.rel_bias", c.rel_buckets, c.n_heads, ok);
    h->enc_final_ln = need(h, "t5.enc.final_ln", Dm, 1, ok);
    h->dec_final_ln = need(h, "t5.dec.final_ln", Dm, 1, ok);
    h->lm_head = need(h, "t5.lm_head", c.vocab, Dm, ok);
    h->enc.resize(c.enc_layers);
    for (int i = 0; i < c.enc_layers; ++i) {
        const std::string p = "t5.enc." + std::to_string(i) + ".";
        T5EncLayerW& L = h->enc[i];
        L.ln0 = need(h, p + "ln0", Dm, 1, ok); L.qkv = need(h, p + "qkv", 3 * inner, Dm, ok);
        L.o = need(h, p + "o", Dm, inner, ok); L.ln1 = need(h, p + "ln1", Dm, 1, ok);
        L.wi = need(h, p + "wi", 2 * c.d_ff, Dm, ok); L.wo = need(h, p + "wo", Dm, c.d_ff, ok);
        if (c.emulate_bf16_rounding & VQA_FLAG_FUSE_NORMS) {
            L.qkv_g = need(h, p + "qkv_g", 3 * inner, Dm, ok);
            L.wi_g = need(h, p + "wi_g", 2 * c.d_ff, Dm, ok);
        }
    }
    h->dec.resize(c.dec_layers);
    for (int i = 0; i < c.dec_layers; ++i) {
        const std::string p = "t5.dec." + std::to_string(i) + ".";
        T5DecLayerW& L = h->dec[i];
        L.ln0 = need(h, p + "ln0", Dm, 1, ok); L.qkv = need(h, p + "qkv", 3 * inner, Dm, ok);
        L.o = need(h, p + "o", Dm, inner, ok); L.ln1 = need(h, p + "ln1", Dm, 1, ok);
        L.cq = need(h, p + "cq", inner, Dm, ok); L.ckv = need(h, p + "ckv", 2 * inner, Dm, ok);
        L.co = need(h, p + "co", Dm, inner, ok); L.ln2 = need(h, p + "ln2", Dm, 1, ok);
        L.wi = need(h, p + "wi", 2 * c.d_ff, Dm, ok); L.wo = need(h, p + "wo", Dm, c.d_ff, ok);
        L.ckT = nullptr;
        if (c.cross_attention_mode == 0) L.ckT = need(h, p + "ckT", Dm, inner, ok);
    }
    if (!ok) return VQA_ERR_MISSING_WEIGHT;
    h->finalized = true;
    return VQA_OK;
}

// ------------------------------------------------------------------------------------------------ workspace plan
struct Plan {
    size_t off = 0;
    size_t take(size_t bytes) {
        size_t o = off;
        off += (bytes + 255) & ~size_t(255);
        return o;
    }
};
struct ClipT5Workspace {
    // vision
    size_t patches, patch_out, hv, vn, vqkv, vattn, vmlp, proj1, proj2;
    // t5
    size_t x, xn, qkv, attn, ff, bias_table, seq_lens, ckv, ssq_a, ssq_b;
    size_t y, yn, dqkv, dattn, dq, dff, splitk, splitk_bytes;
    size_t xt, qt, csc, cctx;   // absorbed cross-attention: Xenc^T, q~ = Wk^T q, scores/probs, context sum p.h
    size_t lse_max, lse_sum, label_logit;
    size_t total;
};
static int ssq_stride(int d_model) { return (d_model / 32 + 3) / 4 * 4; }
static ClipT5Workspace plan_workspace(const vqa_handle* h, int B, int NI, int L, int T) {
    const vqa_clipt5_config& c = h->cfg;
    const int P = (c.image_size / c.patch_size) * (c.image_size / c.patch_size);
    const size_t Mv = (size_t)NI * (P + 1), Mp = (size_t)NI * P;
    const int S = L - 1 + P;
    const size_t M = (size_t)B * S, Md = (size_t)B * T;
    const size_t inner = (size_t)c.n_heads * 64;
    Plan pl;
    ClipT5Workspace w;
    w.patches = pl.take(Mp * h->kpad * 2);
    w.patch_out = pl.take(Mp * c.vit_hidden * 2);
    w.hv = pl.take(Mv * c.vit_hidden * 4);      // fp32: the vision tower's residual stream (see the vision loop)
    w.vn = pl.take(Mv * c.vit_hidden * 2);
    w.vqkv = pl.take(Mv * 3 * c.vit_hidden * 2);
    w.vattn = pl.take(Mv * c.vit_hidden * 2);
    w.vmlp = pl.take(Mv * c.vit_mlp * 2);
    w.proj1 = pl.take(Mv * c.d_model * 2);
    w.proj2 = pl.take(Mv * c.d_model * 2);
    w.x = pl.take(M * c.d_model * 2);
    w.xn = pl.take(M * c.d_model * 2);
    w.qkv = pl.take(M * 3 * inner * 2);
    w.attn = pl.take(M * inner * 2);
    w.ff = pl.take(M * c.d_ff * 2);
    // fused-norm mode: per-row partial sums of squares of the residual stream, two buffers (the stream is rewritten twice per layer);
    // worst case one partial per 32 output columns
    w.ssq_a = pl.take(M * (size_t)ssq_stride(c.d_model) * 4);
    w.ssq_b = pl.take(M * (size_t)ssq_stride(c.d_model) * 4);
    w.bias_table = pl.take((size_t)c.n_heads * (2 * S - 1) * 4);
    w.seq_lens = pl.take((size_t)B * 4);
    const size_t Sp = (size_t)(S + 7) / 8 * 8;
    const size_t TH = (size_t)T * c.n_heads;
    if (c.cross_attention_mode == 0) {
        w.ckv = 0;
        w.xt = pl.take((size_t)B * c.d_model * Sp * 2);
        w.qt = pl.take((size_t)B * TH * c.d_model * 2);
        w.csc = pl.take(((size_t)B * TH + 256) * Sp * 2);
        w.cctx = pl.take((size_t)B * TH * c.d_model * 2);
    } else {
        w.ckv = pl.take(M * 2 * inner * 2);
        w.xt = w.qt = w.csc = w.cctx = 0;
    }
    w.y = pl.take(Md * c.d_model * 2);
    w.yn = pl.take(Md * c.d_model * 2);
    w.dqkv = pl.take(Md * 3 * inner * 2);
    w.dattn = pl.take(Md * inner * 2);
    w.dq = pl.take(Md * inner * 2);
    w.dff = pl.take(Md * c.d_ff * 2);
    {   // fp32 partial tiles of the decoder's split-K GEMMs (largest of the eligible shapes; 0 when none is)
        size_t sk = 0;
        const int shapes[4][2] = {{(int)(3 * inner), c.d_model}, {c.d_model, (int)inner}, {(int)inner, c.d_model}, {c.d_model, c.d_ff}};
        for (const auto& nk : shapes) sk = std::max(sk, splitk_workspace_bytes((int)Md, nk[0], nk[1], h->num_sms));
        w.splitk = pl.take(sk);
        w.splitk_bytes = sk;
    }
    const size_t ntiles = (size_t)LMHEAD_PARTS * ((c.vocab + LMHEAD_BN - 1) / LMHEAD_BN);
    w.lse_max = pl.take(Md * ntiles * 4);
    w.lse_sum = pl.take(Md * ntiles * 4);
    w.label_logit = pl.take(Md * 4);
    w.total = pl.off;
    return w;
}

#include "qwen25vl.cuh"

extern "C" size_t vqa_clipt5_workspace_bytes(vqa_handle* h, int32_t batch, int32_t n_images, int32_t text_len,
                                             int32_t label_len) {
    if (!h || batch <= 0 || n_images <= 0 || text_len <= 0 || label_len <= 0) return 0;
    return plan_workspace(h, batch, n_images, text_len, label_len).total;
}

__global__ void identity_index_kernel(int* idx, int n) {
    pdl_launch_dependents();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) idx[i] = i;
}

// ------------------------------------------------------------------------------------------------ forward
extern "C" int vqa_clipt5_score(vqa_handle* h, const void* pixels, int32_t pixel_dtype, int32_t n_images,
                                const int32_t* image_index, const int32_t* input_ids, const int32_t* text_lens,
                                const int32_t* labels, int32_t B, int32_t L, int32_t T, float* out_scores,
                                float* out_logprobs, void* workspace, size_t workspace_bytes, void* stream) {
    if (!h) return VQA_ERR_INVALID_ARG;
    if (h->kind != 0) return fail(h, VQA_ERR_INVALID_ARG, "not a CLIP-FlanT5 handle");
    if (!h->finalized) return fail(h, VQA_ERR_MISSING_WEIGHT, "vqa_finalize_weights has not succeeded");
    if (!pixels || !input_ids || !text_lens || !labels || !out_scores || !workspace)
        return fail(h, VQA_ERR_INVALID_ARG, "null device pointer");
    if (B <= 0 || L <= 0 || T <= 0 || n_images <= 0) return fail(h, VQA_ERR_INVALID_ARG, "non-positive size");
    if (T > 256) return fail(h, VQA_ERR_UNSUPPORTED, "label_len > 256 not supported by the decoder kernels");
    if (T > 8 && h->cfg.cross_attention_mode != 0)
        return fail(h, VQA_ERR_UNSUPPORTED, "label_len > 8 needs the absorbed cross-attention (cross_attention_mode = 0)");
    if (!image_index && n_images != B) return fail(h, VQA_ERR_INVALID_ARG, "image_index == NULL requires n_images == batch");
    if (pixel_dtype != VQA_DTYPE_F32 && pixel_dtype != VQA_DTYPE_BF16)
        return fail(h, VQA_ERR_INVALID_ARG, "pixel_dtype must be F32 or BF16");
    const vqa_clipt5_config& c = h->cfg;
    const ClipT5Workspace w = plan_workspace(h, B, n_images, L, T);
    if (workspace_bytes < w.total) return fail(h, VQA_ERR_WORKSPACE, "workspace too small");
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return fail(h, VQA_ERR_INVALID_ARG, "workspace must be 256-byte aligned");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    auto P_ = [&](size_t off) { return reinterpret_cast<bf16*>(ws + off); };
    h->launches = 0;
    int64_t* lc = &h->launches;
    const int nsm = h->num_sms;
    const int rnd = c.emulate_bf16_rounding & VQA_FLAG_ROUND_DECODER;
    const bool round_attn = (c.emulate_bf16_rounding & VQA_FLAG_ROUND_ATTN_SCORES) != 0;
    const bool fuse_norms = (c.emulate_bf16_rounding & VQA_FLAG_FUSE_NORMS) != 0;

    const int grid_w = c.image_size / c.patch_size;
    const int P = grid_w * grid_w;
    const int Dv = c.vit_hidden, Dm = c.d_model, H = c.n_heads, inner = H * 64, Hv = c.vit_heads;
    const int Mp = n_images * P, Mv = n_images * (P + 1);
    const int S = L - 1 + P;
    const int M = B * S, Md = B * T;

    h->prof.clear();
    h->ev_used = 0;
#define TRY(x) do { int _rc = (x); if (_rc) return _rc; } while (0)
    auto cuda_ok = [&](cudaError_t e, const char* what) -> int {
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) return fail(h, VQA_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
        return 0;
    };
    auto gemm = [&](const bf16* A, int lda, const bf16* W, int ldw, int w_rows, bf16* C, int ldc, int M_, int N_, int K_,
                    const bf16* bias, const bf16* res, int ldr, int epi, int gate_off) -> int {
        // algorithmic bytes: A and W read once, C written once (+ residual read once)
        const double n_out = epi_is_gated(epi) ? N_ / 2 : N_;
        const double bytes = 2.0 * ((double)M_ * K_ + (double)N_ * K_ + (double)M_ * n_out * (res ? 2 : 1));
        ProfScope ps(h, CAT_GEMM, 2.0 * M_ * (double)N_ * K_, st, bytes);
        return cuda_ok(run_gemm(A, lda, W, ldw, w_rows, C, ldc, M_, N_, K_, bias, res, ldr, epi, gate_off, 0, nsm, st, lc), "gemm");
    };
    auto rms = [&](const bf16* x, const bf16* wgt, bf16* y, int rows) -> int {
        ProfScope ps(h, CAT_NORM, 0, st);
        return cuda_ok(run_rmsnorm(x, wgt, y, rows, Dm, c.t5_ln_eps, st, lc), "rmsnorm");
    };
    auto lnorm = [&](const float* x, const bf16* g, const bf16* b_, bf16* y, int rows) -> int {
        ProfScope ps(h, CAT_NORM, 0, st);
        return cuda_ok(run_layernorm_f32(x, g, b_, y, rows, Dv, c.vit_ln_eps, st, lc), "layernorm");
    };
    auto gemm_f32res = [&](const bf16* A, int lda, const bf16* W, int ldw, int w_rows, float* C, int M_, int N_, int K_, const bf16* bias) -> int {
        // C (fp32) = C + bf16(A W^T + bias): the residual stream is read and written in fp32
        const double bytes = 2.0 * ((double)M_ * K_ + (double)N_ * K_) + 8.0 * (double)M_ * N_;
        ProfScope ps(h, CAT_GEMM, 2.0 * M_ * (double)N_ * K_, st, bytes);
        return cuda_ok(run_gemm(A, lda, W, ldw, w_rows, reinterpret_cast<bf16*>(C), N_, M_, N_, K_, bias, reinterpret_cast<const bf16*>(C), N_,
                                EPI_STORE, 0, 0, nsm, st, lc, true), "gemm (fp32 residual)");
    };
    // Precision of the vision tower's residual stream: the reference runs CLIPVisionModel under torch.autocast(bf16). nn.LayerNorm is on
    // autocast's fp32 list, so pre_layrnorm hands the encoder an fp32 tensor, every `residual + hidden_states` (modeling_clip.py:371,
    // :376) promotes to fp32, and only the Linear inputs are cast to bf16. hidden_states[-2] is therefore an fp32 tensor, rounded to
    // bf16 once where the projector's first Linear consumes it. The engine keeps the same: hv is fp32, the out_proj / fc2 epilogues add
    // the bf16 Linear output into it unrounded, the LayerNorms read fp32 and write the bf16 GEMM operand.
    float* hv = reinterpret_cast<float*>(ws + w.hv);

    // ---------------- vision tower (CLIP ViT, layers 0 .. vit_layers_run-1; hidden_states[-2]) ----------------
    {
        ProfScope ps(h, CAT_OTHER, 0, st);
        ++*lc;
        if (pixel_dtype == VQA_DTYPE_F32)
            patchify_kernel<float><<<Mp, 128, 0, st>>>(reinterpret_cast<const float*>(pixels), P_(w.patches), n_images,
                                                      c.image_size, c.image_size, c.patch_size, h->kpad);
        else
            patchify_kernel<bf16><<<Mp, 128, 0, st>>>(reinterpret_cast<const bf16*>(pixels), P_(w.patches), n_images,
                                                     c.image_size, c.image_size, c.patch_size, h->kpad);
        TRY(cuda_ok(cudaSuccess, "patchify"));
    }
    TRY(gemm(P_(w.patches), h->kpad, h->patch_w, h->kpad, Dv, P_(w.patch_out), Dv, Mp, Dv, h->kpad, nullptr, nullptr, 0,
             EPI_STORE, 0));
    {
        ProfScope ps(h, CAT_NORM, 0, st);
        ++*lc;
        if (Dv == 1024)
            clip_embed_ln_kernel<1024><<<(Mv + 7) / 8, 256, 0, st>>>(P_(w.patch_out), h->cls, h->pos, h->pre_ln_w,
                                                                     h->pre_ln_b, hv, n_images, P, c.vit_ln_eps);
        else if (Dv == 256)
            clip_embed_ln_kernel<256><<<(Mv + 7) / 8, 256, 0, st>>>(P_(w.patch_out), h->cls, h->pos, h->pre_ln_w,
                                                                    h->pre_ln_b, hv, n_images, P, c.vit_ln_eps);
        else
            return fail(h, VQA_ERR_UNSUPPORTED, "vit_hidden must be 1024 or 256");
        TRY(cuda_ok(cudaSuccess, "clip_embed_ln"));
    }
    for (int l = 0; l < c.vit_layers_run; ++l) {
        const VitLayerW& Lw = h->vit[l];
        TRY(lnorm(hv, Lw.ln1_w, Lw.ln1_b, P_(w.vn), Mv));
        TRY(gemm(P_(w.vn), Dv, Lw.qkv_w, Dv, 3 * Dv, P_(w.vqkv), 3 * Dv, Mv, 3 * Dv, Dv, Lw.qkv_b, nullptr, 0, EPI_STORE, 0));
        {
            ProfScope ps(h, CAT_ATTENTION, 4.0 * n_images * (double)Hv * (P + 1) * (P + 1) * 64, st);
            TRY(cuda_ok(run_flash(P_(w.vqkv), P_(w.vqkv) + Dv, P_(w.vqkv) + 2 * Dv, 3 * Dv, P_(w.vattn), Dv, n_images, P + 1,
                                  Hv, nullptr, nullptr, 0.125f, 0, round_attn, st, lc), "vit attention"));
        }
        TRY(gemm_f32res(P_(w.vattn), Dv, Lw.out_w, Dv, Dv, hv, Mv, Dv, Dv, Lw.out_b));
        TRY(lnorm(hv, Lw.ln2_w, Lw.ln2_b, P_(w.vn), Mv));
        TRY(gemm(P_(w.vn), Dv, Lw.fc1_w, Dv, c.vit_mlp, P_(w.vmlp), c.vit_mlp, Mv, c.vit_mlp, Dv, Lw.fc1_b, nullptr, 0,
                 EPI_QUICK_GELU, 0));
        TRY(gemm_f32res(P_(w.vmlp), c.vit_mlp, Lw.fc2_w, c.vit_mlp, Dv, hv, Mv, Dv, c.vit_mlp, Lw.fc2_b));
    }
    {   // hidden_states[-2] -> bf16 (`.to(images.dtype)` / the projector Linear's autocast cast): the single rounding of the tower's output
        ProfScope ps(h, CAT_OTHER, 0, st);
        ++*lc;
        const size_t n = (size_t)Mv * Dv;
        cast_f32_bf16_kernel<<<(unsigned)((n / 4 + 255) / 256 + 1), 256, 0, st>>>(hv, P_(w.vn), n);
        TRY(cuda_ok(cudaSuccess, "vision output cast"));
    }
    // mlp2x_gelu projector (Linear -> GELU(erf) -> Linear), applied to every row; the CLS rows are simply not spliced
    TRY(gemm(P_(w.vn), Dv, h->proj0_w, Dv, Dm, P_(w.proj1), Dm, Mv, Dm, Dv, h->proj0_b, nullptr, 0, EPI_GELU_ERF, 0));
    TRY(gemm(P_(w.proj1), Dm, h->proj2_w, Dm, Dm, P_(w.proj2), Dm, Mv, Dm, Dm, h->proj2_b, nullptr, 0, EPI_STORE, 0));

    // ---------------- multimodal splice -> T5 encoder input ----------------
    int* seq_lens = reinterpret_cast<int*>(ws + w.seq_lens);
    float* bias_table = reinterpret_cast<float*>(ws + w.bias_table);
    {
        ProfScope ps(h, CAT_OTHER, 0, st);
        *lc += 2;
        // feature block of an image = P + 1 rows, first patch row = 1 (drop CLS: mm_vision_select_feature='patch')
        splice_embed_kernel<<<B * S, 128, 0, st>>>(input_ids, text_lens, image_index, h->shared, P_(w.proj2), Dm, 1, P + 1,
                                                   P_(w.x), seq_lens, B, L, S, P, Dm, c.image_token_id);
        bias_table_from_lut_kernel<<<(H * (2 * S - 1) + 255) / 256, 256, 0, st>>>(h->enc_rel, h->lut_bidir,
                                                                                  c.rel_max_distance, bias_table, H, S);
        TRY(cuda_ok(cudaSuccess, "splice / bias table"));
    }

    // ---------------- T5 encoder ----------------
    // fuse_norms: the two T5LayerNorms of a layer never run as kernels. The GEMMs that write the residual stream (o, wo) leave per-row
    // partial sums of squares of what they stored; the GEMMs that read it (qkv, wi) take x itself with gamma folded into their weights and
    // scale their accumulator rows by rsqrt(mean(x^2) + eps) in the epilogue (gemm_sm100.cuh, GemmParams::ssq_*).
    NormFuse nf_cons, nf_prod;
    float* ssq_cur = reinterpret_cast<float*>(ws + w.ssq_a);
    float* ssq_nxt = reinterpret_cast<float*>(ws + w.ssq_b);
    if (fuse_norms) {
        const int parts = ssq_parts_for(pick_variant(M, Dm, EPI_STORE), Dm);
        const int stride = (parts + 3) / 4 * 4;
        if (stride > ssq_stride(Dm)) return fail(h, VQA_ERR_UNSUPPORTED, "fused norms: partial-sum stride exceeds the workspace plan");
        nf_cons.stride = nf_prod.stride = stride;
        nf_cons.inv_dim = 1.0f / (float)Dm;
        nf_cons.eps = c.t5_ln_eps;
        ProfScope ps(h, CAT_NORM, 0, st);
        *lc += 3;
        TRY(cuda_ok(cudaMemsetAsync(ssq_cur, 0, (size_t)M * stride * 4, st), "ssq clear"));
        TRY(cuda_ok(cudaMemsetAsync(ssq_nxt, 0, (size_t)M * stride * 4, st), "ssq clear"));
        row_ssq_kernel<<<(M + 7) / 8, 256, 0, st>>>(P_(w.x), ssq_cur, M, Dm, stride);
        TRY(cuda_ok(cudaSuccess, "row ssq"));
    }
    auto gemm_nf = [&](const bf16* A, int lda, const bf16* W, int ldw, int w_rows, bf16* C, int ldc, int M_, int N_, int K_, const bf16* res, int ldr,
                       int epi, int gate_off, const NormFuse& nf) -> int {
        const double n_out = epi_is_gated(epi) ? N_ / 2 : N_;
        const double bytes = 2.0 * ((double)M_ * K_ + (double)N_ * K_ + (double)M_ * n_out * (res ? 2 : 1));
        ProfScope ps(h, CAT_GEMM, 2.0 * M_ * (double)N_ * K_, st, bytes);
        return cuda_ok(run_gemm(A, lda, W, ldw, w_rows, C, ldc, M_, N_, K_, nullptr, res, ldr, epi, gate_off, 0, nsm, st, lc, false, &nf), "gemm");
    };
    for (int l = 0; l < c.enc_layers; ++l) {
        const T5EncLayerW& Lw = h->enc[l];
        if (fuse_norms) {
            nf_cons.ssq_in = ssq_cur;
            TRY(gemm_nf(P_(w.x), Dm, Lw.qkv_g, Dm, 3 * inner, P_(w.qkv), 3 * inner, M, 3 * inner, Dm, nullptr, 0, EPI_STORE, 0, nf_cons));
        } else {
            TRY(rms(P_(w.x), Lw.ln0, P_(w.xn), M));
            TRY(gemm(P_(w.xn), Dm, Lw.qkv, Dm, 3 * inner, P_(w.qkv), 3 * inner, M, 3 * inner, Dm, nullptr, nullptr, 0, EPI_STORE, 0));
        }
        {
            ProfScope ps(h, CAT_ATTENTION, 4.0 * B * (double)H * S * S * 64, st);
            TRY(cuda_ok(run_flash(P_(w.qkv), P_(w.qkv) + inner, P_(w.qkv) + 2 * inner, 3 * inner, P_(w.attn), inner, B, S, H,
                                  seq_lens, bias_table, 1.0f, c.rel_max_distance, round_attn, st, lc), "t5 encoder attention"));
        }
        if (fuse_norms) {
            nf_prod.ssq_out = ssq_nxt;
            TRY(gemm_nf(P_(w.attn), inner, Lw.o, inner, Dm, P_(w.x), Dm, M, Dm, inner, P_(w.x), Dm, EPI_STORE, 0, nf_prod));
            std::swap(ssq_cur, ssq_nxt);
            nf_cons.ssq_in = ssq_cur;
            TRY(gemm_nf(P_(w.x), Dm, Lw.wi_g, Dm, 2 * c.d_ff, P_(w.ff), c.d_ff, M, 2 * c.d_ff, Dm, nullptr, 0, EPI_GATED_GELU, c.d_ff, nf_cons));
            nf_prod.ssq_out = ssq_nxt;
            TRY(gemm_nf(P_(w.ff), c.d_ff, Lw.wo, c.d_ff, Dm, P_(w.x), Dm, M, Dm, c.d_ff, P_(w.x), Dm, EPI_STORE, 0, nf_prod));
            std::swap(ssq_cur, ssq_nxt);
        } else {
            TRY(gemm(P_(w.attn), inner, Lw.o, inner, Dm, P_(w.x), Dm, M, Dm, inner, nullptr, P_(w.x), Dm, EPI_STORE, 0));
            TRY(rms(P_(w.x), Lw.ln1, P_(w.xn), M));
            TRY(gemm(P_(w.xn), Dm, Lw.wi, Dm, 2 * c.d_ff, P_(w.ff), c.d_ff, M, 2 * c.d_ff, Dm, nullptr, nullptr, 0, EPI_GATED_GELU,
                     c.d_ff));
            TRY(gemm(P_(w.ff), c.d_ff, Lw.wo, c.d_ff, Dm, P_(w.x), Dm, M, Dm, c.d_ff, nullptr, P_(w.x), Dm, EPI_STORE, 0));
        }
    }
    TRY(rms(P_(w.x), h->enc_final_ln, P_(w.xn), M));  // encoder output lives in xn from here on
    const int Sp = (S + 7) / 8 * 8;
    if (c.cross_attention_mode == 0) {
        ProfScope ps(h, CAT_OTHER, 0, st);
        ++*lc;
        transpose_bsd_kernel<<<dim3((Sp + 31) / 32, (Dm + 31) / 32, B), dim3(32, 8), 0, st>>>(P_(w.xn), P_(w.xt), S, Dm, Sp);
        TRY(cuda_ok(cudaSuccess, "encoder transpose"));
    }

    // ---------------- T5 decoder (T target rows per pair) ----------------
    {
        ProfScope ps(h, CAT_OTHER, 0, st);
        ++*lc;
        decoder_embed_kernel<<<Md, 128, 0, st>>>(labels, h->shared, P_(w.y), T, Dm, c.decoder_start_id, c.pad_token_id);
        TRY(cuda_ok(cudaSuccess, "decoder embed"));
    }
    // decoder store-GEMMs: M = B*T rows against 4096-row weights -> split-K when that fills the SMs (run_gemm_splitk), else the plain path
    auto dgemm = [&](const bf16* A, int lda, const bf16* W, int ldw, int w_rows, bf16* C, int ldc, int M_, int N_, int K_,
                     const bf16* bias, const bf16* res, int ldr, int epi, int gate_off) -> int {
        const int sl = epi == EPI_STORE ? splitk_slices(M_, N_, K_, nsm) : 1;
        if (sl <= 1 || (size_t)sl * M_ * N_ * 4 > w.splitk_bytes) return gemm(A, lda, W, ldw, w_rows, C, ldc, M_, N_, K_, bias, res, ldr, epi, gate_off);
        const double bytes = 2.0 * ((double)M_ * K_ + (double)N_ * K_ + (double)M_ * N_ * (res ? 2 : 1));
        ProfScope ps(h, CAT_GEMM, 2.0 * M_ * (double)N_ * K_, st, bytes);
        return cuda_ok(run_gemm_splitk(A, lda, W, ldw, w_rows, C, ldc, M_, N_, K_, bias, res, ldr, sl, reinterpret_cast<float*>(ws + w.splitk), nsm, st, lc),
                       "split-K gemm");
    };
    for (int l = 0; l < c.dec_layers; ++l) {
        const T5DecLayerW& Lw = h->dec[l];
        // self-attention
        TRY(rms(P_(w.y), Lw.ln0, P_(w.yn), Md));
        TRY(dgemm(P_(w.yn), Dm, Lw.qkv, Dm, 3 * inner, P_(w.dqkv), 3 * inner, Md, 3 * inner, Dm, nullptr, nullptr, 0, EPI_STORE, 0));
        {
            ProfScope ps(h, CAT_ATTENTION, 4.0 * B * (double)H * T * T * 64, st);
            ++*lc;
            t5_decoder_self_attn_kernel<<<(B * H * T + 3) / 4, 128, 4 * T * sizeof(float), st>>>(P_(w.dqkv), P_(w.dattn), h->dec_rel, h->lut_unidir,
                                                                             c.rel_max_distance, B, T, H, rnd);
            TRY(cuda_ok(cudaSuccess, "decoder self attention"));
        }
        TRY(dgemm(P_(w.dattn), inner, Lw.o, inner, Dm, P_(w.y), Dm, Md, Dm, inner, nullptr, P_(w.y), Dm, EPI_STORE, 0));
        TRY(rms(P_(w.y), Lw.ln1, P_(w.yn), Md));
        TRY(dgemm(P_(w.yn), Dm, Lw.cq, Dm, inner, P_(w.dq), inner, Md, inner, Dm, nullptr, nullptr, 0, EPI_STORE, 0));
        if (c.cross_attention_mode != 0) {
            // reference association: K/V projection of all S encoder rows in every layer (modeling_t5.py:297-299)
            TRY(gemm(P_(w.xn), Dm, Lw.ckv, Dm, 2 * inner, P_(w.ckv), 2 * inner, M, 2 * inner, Dm, nullptr, nullptr, 0, EPI_STORE, 0));
            ProfScope ps(h, CAT_ATTENTION, 4.0 * B * (double)H * T * S * 64, st);
            ++*lc;
            t5_cross_attn_kernel<8><<<B * H, 128, 0, st>>>(P_(w.dq), P_(w.ckv), P_(w.dattn), seq_lens, 2 * inner, B, T, S, H, rnd);
            TRY(cuda_ok(cudaSuccess, "cross attention"));
        } else {
            // absorbed association (exact in real arithmetic; 30x fewer FLOPs because only T rows per pair attend):
            //   q.(Wk x_s) = (Wk^T q).x_s          sum_s p_s (Wv x_s) = Wv (sum_s p_s x_s)
            const int TH = T * H;
            auto bgemm = [&](const bf16* A, int lda, const bf16* W, int ldw, bf16* C, int ldc, int M_, int N_, int K_,
                             const BatchSpec& bs, int variant) -> int {
                ProfScope ps(h, CAT_GEMM, 2.0 * bs.nb * (double)M_ * N_ * K_, st,
                             2.0 * bs.nb * ((double)M_ * K_ + (double)N_ * K_ + (double)M_ * N_));
                return cuda_ok(run_gemm_batched(A, lda, W, ldw, C, ldc, M_, N_, K_, bs, variant, nsm, st, lc), "batched gemm");
            };
            // (1) q~[b,t,h,:] = Wk[h]^T q[b,t,h,:]   -- per head: [B*T, 64] x ckT[:, h*64:(h+1)*64]^T -> rows (b*T+t)*H + h
            TRY(bgemm(P_(w.dq), inner, Lw.ckT, inner, P_(w.qt), H * Dm, Md, Dm, 64,
                      BatchSpec{H, 0, 64, 0, 64, (long long)Dm, Md, inner, Dm, inner}, Dm >= 256 ? 2561 : 1281));
            // (2) scores[b,(t,h),s] = q~[b,(t,h),:] . x[b,s,:]   -- per pair: [T*H, d] x [S, d]^T
            TRY(bgemm(P_(w.qt), Dm, P_(w.xn), Dm, P_(w.csc), Sp, TH, Sp, Dm,
                      BatchSpec{B, TH, 0, S, 0, (long long)TH * Sp, (long long)B * TH, Dm, (long long)B * S, Dm}, 1281));
            {
                ProfScope ps(h, CAT_ATTENTION, 0, st);
                ++*lc;
                cross_softmax_kernel<<<(B * TH + 7) / 8, 256, 0, st>>>(P_(w.csc), seq_lens, TH, B * TH, S, Sp);
                TRY(cuda_ok(cudaSuccess, "cross softmax"));
            }
            // (3) ctx[b,(t,h),:] = sum_s p[b,(t,h),s] x[b,s,:]   -- per pair: [T*H, Sp] x (x[b]^T)[d, Sp]^T
            TRY(bgemm(P_(w.csc), Sp, P_(w.xt), Sp, P_(w.cctx), Dm, TH, Dm, Sp,
                      BatchSpec{B, TH, 0, Dm, 0, (long long)TH * Dm, (long long)B * TH, Sp, (long long)B * Dm, Sp},
                      Dm >= 256 ? 2561 : 1281));
            // (4) o[b,t,h,:] = Wv[h] ctx[b,t,h,:]   -- per head: [B*T, d] (cols h*d..) x Wv[h*64:(h+1)*64, :]^T -> cols h*64..
            TRY(bgemm(P_(w.cctx), H * Dm, Lw.ckv + (size_t)inner * Dm, Dm, P_(w.dattn), inner, Md, 64, Dm,
                      BatchSpec{H, 0, Dm, 64, 0, 64, Md, (long long)H * Dm, inner, Dm}, 641));
        }
        TRY(dgemm(P_(w.dattn), inner, Lw.co, inner, Dm, P_(w.y), Dm, Md, Dm, inner, nullptr, P_(w.y), Dm, EPI_STORE, 0));
        // gated FFN
        TRY(rms(P_(w.y), Lw.ln2, P_(w.yn), Md));
        TRY(gemm(P_(w.yn), Dm, Lw.wi, Dm, 2 * c.d_ff, P_(w.dff), c.d_ff, Md, 2 * c.d_ff, Dm, nullptr, nullptr, 0, EPI_GATED_GELU,
                 c.d_ff));
        TRY(dgemm(P_(w.dff), c.d_ff, Lw.wo, c.d_ff, Dm, P_(w.y), Dm, Md, Dm, c.d_ff, nullptr, P_(w.y), Dm, EPI_STORE, 0));
    }
    TRY(rms(P_(w.y), h->dec_final_ln, P_(w.yn), Md));

    // ---------------- lm_head x hidden, fused log-sum-exp + label gather; logits never reach HBM ----------------
    float* lse_max = reinterpret_cast<float*>(ws + w.lse_max);
    float* lse_sum = reinterpret_cast<float*>(ws + w.lse_sum);
    float* label_logit = reinterpret_cast<float*>(ws + w.label_logit);
    const int ntiles = LMHEAD_PARTS * ((c.vocab + LMHEAD_BN - 1) / LMHEAD_BN);
    {
        ProfScope ps(h, CAT_GEMM, 2.0 * Md * (double)c.vocab * Dm, st, 2.0 * ((double)Md * Dm + (double)c.vocab * Dm));
        TRY(cuda_ok(run_lmhead(P_(w.yn), Dm, h->lm_head, Dm, Md, c.vocab, Dm, labels, lse_max, lse_sum, label_logit, nsm, st, lc),
                    "lm_head"));
    }
    {
        ProfScope ps(h, CAT_OTHER, 0, st);
        ++*lc;
        lse_finalize_kernel<<<(B + 3) / 4, 128, 0, st>>>(lse_max, lse_sum, label_logit, labels, out_scores, out_logprobs, B, T,
                                                        ntiles);
        TRY(cuda_ok(cudaSuccess, "lse finalize"));
    }
#undef TRY
    return VQA_OK;
}

// Byte offsets inside the caller's workspace of the tensors a parity investigation wants to look at after a call has completed.
extern "C" int vqa_clipt5_debug_layout(vqa_handle* h, int32_t batch, int32_t n_images, int32_t text_len, int32_t label_len,
                                       size_t* offsets, int32_t n) {
    if (!h || h->kind != 0 || !offsets || n < 6 || batch <= 0 || n_images <= 0 || text_len <= 0 || label_len <= 0)
        return fail(h, VQA_ERR_INVALID_ARG, "bad debug layout argument");
    const ClipT5Workspace w = plan_workspace(h, batch, n_images, text_len, label_len);
    offsets[0] = w.xn;      // encoder output after the final T5LayerNorm  [B*S, d_model] bf16
    offsets[1] = w.yn;      // decoder output after the final T5LayerNorm  [B*T, d_model] bf16
    offsets[2] = w.proj2;   // projector output                            [NI*(P+1), d_model] bf16 (row 0 of each image = CLS)
    offsets[3] = w.x;       // encoder residual stream before the final norm
    offsets[4] = w.y;       // decoder residual stream before the final norm
    offsets[5] = w.hv;      // vision tower hidden states of the last executed layer [NI*(P+1), vit_hidden] FP32
    return VQA_OK;
}

extern "C" int vqa_qwen25vl_debug_layout(vqa_handle* h, int32_t batch, int32_t seq_len, int32_t n_patches, size_t* offsets, int32_t n) {
    if (!h || h->kind != 1 || !offsets || n < 4 || batch <= 0 || seq_len <= 0 || n_patches <= 0)
        return fail(h, VQA_ERR_INVALID_ARG, "bad debug layout argument");
    const QwenWorkspace w = qwen_plan(h->qwen->cfg, batch, seq_len, n_patches);
    offsets[0] = w.lastn;       // last-position hidden state after the final RMSNorm [B, hidden] bf16
    offsets[1] = w.vfeat_orig;  // merged vision features in processor order         [n_patches / merge^2, out_hidden] bf16
    offsets[2] = w.x;           // language-model residual stream                     [B*S, hidden] bf16
    offsets[3] = w.last;        // last-position residual before the final norm       [B, hidden] bf16
    return VQA_OK;
}

// Process-wide override of the GEMM tile order (tuning / A-B measurements): group_rows > 0 = A rows per M group, chunk_rows > 0 = W rows
// per L2-resident chunk, chunk_rows < 0 = no chunking; 0 = automatic choice (gemm_sm100.cuh launch_gemm_t).
extern "C" int vqa_set_gemm_schedule(int32_t group_rows, int32_t chunk_rows) {
    g_gemm_group_rows_override = group_rows;
    g_gemm_chunk_rows_override = chunk_rows;
    return VQA_OK;
}

// How many clusters of `cluster_size` CTAs of the 256-wide cta_group::2 GEMM kernel (one CTA per SM: ~198 KB of shared memory) the current
// device can hold at once (cudaOccupancyMaxActiveClusters). 148 SMs do not always divide into GPC-local clusters of 4 or 8: this is the
// number a cluster-multicast variant of the GEMM has to be sized against. Returns the count, or a negative vqa_status.
extern "C" int vqa_debug_max_active_clusters(int32_t cluster_size) {
    if (cluster_size < 1 || cluster_size > 16) return VQA_ERR_INVALID_ARG;
    using Cfg = GemmConfig<256, 2>;
    auto kernel = gemm_bf16_sm100_kernel<256, 2, EPI_STORE>;
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES) != cudaSuccess) return VQA_ERR_CUDA;
    if (cluster_size > 8 && cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) return VQA_ERR_CUDA;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(sms / cluster_size * cluster_size));
    cfg.blockDim = dim3(Cfg::NUM_THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cudaLaunchAttribute attrs[1];
    attrs[0].id = cudaLaunchAttributeClusterDimension;
    attrs[0].val.clusterDim.x = (unsigned)cluster_size;
    attrs[0].val.clusterDim.y = 1;
    attrs[0].val.clusterDim.z = 1;
    cfg.attrs = attrs;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess) { cudaGetLastError(); return VQA_ERR_CUDA; }
    return n;
}

extern "C" int vqa_set_profile(vqa_handle* h, int32_t enable) {
    if (!h) return VQA_ERR_INVALID_ARG;
    h->profile = enable != 0;
    return VQA_OK;
}

// After the stream has been synchronised by the caller: device milliseconds, algorithmic FLOPs and launch-scope counts of
// the last vqa_clipt5_score call per category {0 gemm, 1 attention, 2 norm, 3 other}.
extern "C" int vqa_profile_read(vqa_handle* h, float* ms, double* flops, double* bytes, int64_t* scopes) {
    if (!h || !ms || !flops || !bytes || !scopes) return VQA_ERR_INVALID_ARG;
    for (int i = 0; i < CAT_COUNT; ++i) { ms[i] = 0.f; flops[i] = 0.0; bytes[i] = 0.0; scopes[i] = 0; }
    for (const auto& r : h->prof) {
        float t = 0.f;
        cudaError_t e = cudaEventElapsedTime(&t, h->ev_pool[r.ev0], h->ev_pool[r.ev1]);
        if (e != cudaSuccess) return fail(h, VQA_ERR_CUDA, std::string("cudaEventElapsedTime: ") + cudaGetErrorString(e));
        ms[r.cat] += t;
        flops[r.cat] += r.flops;
        bytes[r.cat] += r.bytes;
        scopes[r.cat] += 1;
    }
    return VQA_OK;
}

extern "C" int64_t vqa_last_launch_count(vqa_handle* h) { return h ? h->launches : 0; }
extern "C" const char* vqa_last_error(vqa_handle* h) { return h ? h->err.c_str() : g_global_err.c_str(); }
extern "C" void vqa_destroy(vqa_handle* h) {
    if (!h) return;
    if (h->lut_bidir) cudaFree(h->lut_bidir);
    if (h->lut_unidir) cudaFree(h->lut_unidir);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    if (h->qwen) {
        QwenState* q = h->qwen;
        if (q->text_axis) cudaFree(q->text_axis);
        if (q->vis_axis) cudaFree(q->vis_axis);
        if (q->text_inv_freq) cudaFree(q->text_inv_freq);
        if (q->vis_inv_freq) cudaFree(q->vis_inv_freq);
        delete q;
    }
    delete h;
}

// ------------------------------------------------------------------------------------------------ Qwen2.5-VL ABI
extern "C" int vqa_create_qwen25vl(const vqa_qwen25vl_config* cfg, int device, vqa_handle** out) {
    if (!cfg || !out) return fail(nullptr, VQA_ERR_INVALID_ARG, "null argument");
    if (cfg->heads % cfg->kv_heads) return fail(nullptr, VQA_ERR_INVALID_ARG, "heads % kv_heads != 0");
    if (cfg->vit_head_dim > 128 || cfg->vit_head_dim % 16 || cfg->vit_hidden != cfg->vit_heads * cfg->vit_head_dim)
        return fail(nullptr, VQA_ERR_UNSUPPORTED, "vision head_dim must be a multiple of 16, <= 128, and hidden = heads * head_dim");
    if (cfg->hidden % 8 || cfg->mlp % 128 || cfg->vit_hidden % 8 || cfg->patch_dim % 8)
        return fail(nullptr, VQA_ERR_UNSUPPORTED, "hidden % 8, mlp % 128, vit_hidden % 8, patch_dim % 8 must be 0");
    if (cfg->vit_depth > 64) return fail(nullptr, VQA_ERR_UNSUPPORTED, "vit_depth > 64");
    cudaError_t e = cudaSetDevice(device);
    cudaDeviceProp prop;
    if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess || prop.major != 10) return fail(nullptr, VQA_ERR_UNSUPPORTED, "vqa_b200 requires an sm_100 (B200) device");
    vqa_handle* h = new vqa_handle();
    h->kind = 1;
    h->device = device;
    h->num_sms = prop.multiProcessorCount;
    h->qwen = new QwenState();
    h->qwen->cfg = *cfg;
    *out = h;
    return VQA_OK;
}

extern "C" int vqa_qwen25vl_set_rope(vqa_handle* h, const float* text_inv_freq, const int32_t* text_axis, int32_t text_half,
                                     const float* vis_inv_freq, const int32_t* vis_axis, int32_t vis_half) {
    if (!h || h->kind != 1 || !text_inv_freq || !text_axis || !vis_inv_freq || !vis_axis)
        return fail(h, VQA_ERR_INVALID_ARG, "bad rope argument");
    QwenState& q = *h->qwen;
    if (text_half != 64 || vis_half != q.cfg.vit_head_dim / 2) return fail(h, VQA_ERR_INVALID_ARG, "rope table sizes do not match the config");
    auto up = [&](const void* src, size_t bytes, void** dst) -> bool {
        if (*dst) cudaFree(*dst);
        return cudaMalloc(dst, bytes) == cudaSuccess && cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
    };
    if (!up(text_inv_freq, 64 * 4, (void**)&q.text_inv_freq) || !up(text_axis, 64 * 4, (void**)&q.text_axis) ||
        !up(vis_inv_freq, vis_half * 4, (void**)&q.vis_inv_freq) || !up(vis_axis, vis_half * 4, (void**)&q.vis_axis))
        return fail(h, VQA_ERR_CUDA, "rope table upload failed");
    q.rope_set = true;
    return VQA_OK;
}

extern "C" size_t vqa_qwen25vl_workspace_bytes(vqa_handle* h, int32_t batch, int32_t seq_len, int32_t n_patches) {
    if (!h || h->kind != 1 || batch <= 0 || seq_len <= 0 || n_patches <= 0) return 0;
    return qwen_plan(h->qwen->cfg, batch, seq_len, n_patches).total;
}

extern "C" int vqa_qwen25vl_score(vqa_handle* h, const void* pixel_patches, int32_t pixel_dtype, int32_t n_patches,
                                  const int32_t* vis_pos_hw, const int32_t* window_index, const int32_t* reverse_index,
                                  const int32_t* cu_window, int32_t n_windows, int32_t max_window_len, const int32_t* cu_frames,
                                  int32_t n_frames, int32_t max_frame_len, const int32_t* input_ids, const int32_t* seq_lens,
                                  const int32_t* feat_index, const int32_t* position_ids, const int32_t* answer_ids, int32_t batch,
                                  int32_t seq_len, float temperature, float repetition_penalty, float* out_probs, float* out_logprobs,
                                  void* workspace,
                                  size_t workspace_bytes, void* stream) {
    if (!h || h->kind != 1) return fail(h, VQA_ERR_INVALID_ARG, "not a Qwen2.5-VL handle");
    if (!h->finalized) return fail(h, VQA_ERR_MISSING_WEIGHT, "vqa_finalize_weights has not succeeded");
    if (!pixel_patches || !vis_pos_hw || !window_index || !reverse_index || !cu_window || !cu_frames || !input_ids || !seq_lens ||
        !feat_index || !position_ids || !answer_ids || !out_probs || !workspace)
        return fail(h, VQA_ERR_INVALID_ARG, "null device pointer");
    const int unit = h->qwen->cfg.spatial_merge * h->qwen->cfg.spatial_merge;
    if (batch <= 0 || seq_len <= 0 || n_patches <= 0 || n_patches % unit || n_windows <= 0 || n_frames <= 0 || !(temperature > 0.f) ||
        !(repetition_penalty > 0.f))
        return fail(h, VQA_ERR_INVALID_ARG, "bad size / temperature / repetition penalty");
    if (pixel_dtype != VQA_DTYPE_F32 && pixel_dtype != VQA_DTYPE_BF16) return fail(h, VQA_ERR_INVALID_ARG, "pixel_dtype must be F32 or BF16");
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return fail(h, VQA_ERR_INVALID_ARG, "workspace must be 256-byte aligned");
    return qwen_score(h, *h->qwen, pixel_patches, pixel_dtype, n_patches, vis_pos_hw, window_index, reverse_index, cu_window, n_windows,
                      max_window_len, cu_frames, n_frames, max_frame_len, input_ids, seq_lens, feat_index, position_ids, answer_ids, batch,
                      seq_len, temperature, repetition_penalty, out_probs, out_logprobs, workspace, workspace_bytes,
                      reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int vqa_qwen25vl_topk(vqa_handle* h, int32_t batch, int64_t total_rows, int32_t n_patches, int32_t k, float temperature,
                                 float repetition_penalty, int32_t* out_ids, float* out_probs, void* workspace, size_t workspace_bytes, void* stream) {
    if (!h || h->kind != 1) return fail(h, VQA_ERR_INVALID_ARG, "not a Qwen2.5-VL handle");
    if (!h->finalized) return fail(h, VQA_ERR_MISSING_WEIGHT, "vqa_finalize_weights has not succeeded");
    if (!out_ids || !out_probs || !workspace || batch <= 0 || total_rows <= 0 || n_patches <= 0 || k <= 0 || k > TOPK_MAX || !(temperature > 0.f) ||
        !(repetition_penalty > 0.f))
        return fail(h, VQA_ERR_INVALID_ARG, "bad top-k argument (1 <= k <= 8)");
    return qwen_topk(h, *h->qwen, batch, (size_t)total_rows, n_patches, k, temperature, repetition_penalty, out_ids, out_probs, workspace,
                     workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" size_t vqa_qwen25vl_packed_workspace_bytes(vqa_handle* h, int32_t n_prompts, int64_t total_rows, int32_t n_patches) {
    if (!h || h->kind != 1 || n_prompts <= 0 || total_rows <= 0 || n_patches <= 0) return 0;
    return qwen_plan_rows(h->qwen->cfg, n_prompts, (size_t)total_rows, n_patches).total;
}

extern "C" int vqa_qwen25vl_score_packed(vqa_handle* h, const void* pixel_patches, int32_t pixel_dtype, int32_t n_patches,
                                         const int32_t* vis_pos_hw, const int32_t* window_index, const int32_t* reverse_index,
                                         const int32_t* cu_window, int32_t n_windows, int32_t max_window_len, const int32_t* cu_frames,
                                         int32_t n_frames, int32_t max_frame_len, const int32_t* input_ids, const int32_t* feat_index,
                                         const int32_t* position_ids, int32_t total_rows, const int32_t* cu_seqlens, const int32_t* kv_prefix,
                                         int32_t n_seq, int32_t max_seq_len, const int32_t* pair_row, const int32_t* pair_seq,
                                         const int32_t* answer_ids, int32_t n_prompts, int32_t max_prompt_len, float temperature,
                                         float repetition_penalty, float* out_probs, float* out_logprobs, void* workspace, size_t workspace_bytes,
                                         void* stream) {
    if (!h || h->kind != 1) return fail(h, VQA_ERR_INVALID_ARG, "not a Qwen2.5-VL handle");
    if (!h->finalized) return fail(h, VQA_ERR_MISSING_WEIGHT, "vqa_finalize_weights has not succeeded");
    if (!pixel_patches || !vis_pos_hw || !window_index || !reverse_index || !cu_window || !cu_frames || !input_ids || !feat_index || !position_ids ||
        !cu_seqlens || !kv_prefix || !pair_row || !pair_seq || !answer_ids || !out_probs || !workspace)
        return fail(h, VQA_ERR_INVALID_ARG, "null device pointer");
    const int unit = h->qwen->cfg.spatial_merge * h->qwen->cfg.spatial_merge;
    if (n_prompts <= 0 || total_rows <= 0 || n_seq <= 0 || max_seq_len <= 0 || max_prompt_len <= 0 || n_patches <= 0 || n_patches % unit ||
        n_windows <= 0 || n_frames <= 0 || !(temperature > 0.f) || !(repetition_penalty > 0.f))
        return fail(h, VQA_ERR_INVALID_ARG, "bad size / temperature / repetition penalty");
    if (pixel_dtype != VQA_DTYPE_F32 && pixel_dtype != VQA_DTYPE_BF16) return fail(h, VQA_ERR_INVALID_ARG, "pixel_dtype must be F32 or BF16");
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return fail(h, VQA_ERR_INVALID_ARG, "workspace must be 256-byte aligned");
    QwenPacked pk;
    pk.total_rows = total_rows; pk.n_seq = n_seq; pk.max_seq_len = max_seq_len; pk.max_prompt_len = max_prompt_len;
    pk.cu_seqlens = cu_seqlens; pk.kv_prefix = kv_prefix; pk.pair_row = pair_row; pk.pair_seq = pair_seq;
    return qwen_score(h, *h->qwen, pixel_patches, pixel_dtype, n_patches, vis_pos_hw, window_index, reverse_index, cu_window, n_windows,
                      max_window_len, cu_frames, n_frames, max_frame_len, input_ids, nullptr, feat_index, position_ids, answer_ids, n_prompts,
                      total_rows, temperature, repetition_penalty, out_probs, out_logprobs, workspace, workspace_bytes,
                      reinterpret_cast<cudaStream_t>(stream), &pk);
}

// ------------------------------------------------------------------------------------------------ kernel-level ABI
static int device_sms() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}

extern "C" int vqa_op_gemm_bf16(const void* A, int32_t lda, const void* W, int32_t ldw, int32_t w_rows, void* C,
                                int32_t ldc, int32_t M, int32_t N, int32_t K, const void* bias, const void* residual,
                                int32_t ldr, int32_t epilogue, int32_t gate_up_offset, int32_t variant, void* stream) {
    if (!A || !W || !C || M <= 0 || N <= 0 || K <= 0) return fail(nullptr, VQA_ERR_INVALID_ARG, "bad gemm argument");
    if (lda % 8 || ldw % 8 || ldc % 8 || N % 8 || K % 8) return fail(nullptr, VQA_ERR_INVALID_ARG, "gemm: ld/N/K must be multiples of 8");
    cudaError_t e = run_gemm((const bf16*)A, lda, (const bf16*)W, ldw, w_rows, (bf16*)C, ldc, M, N, K, (const bf16*)bias,
                             (const bf16*)residual, ldr, epilogue, gate_up_offset, variant, device_sms(),
                             (cudaStream_t)stream, nullptr);
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("gemm launch: ") + cudaGetErrorString(e));
    return VQA_OK;
}

// vqa_op_gemm_bf16 (plain store epilogue) whose output columns are written in groups: logical column c lands at (c / group_in) * group_out + c % group_in
// (heads narrower than the attention kernel's 128-wide slots are produced at their native width; the caller zeroes the slot padding).
extern "C" int vqa_op_gemm_bf16_grouped(const void* A, int32_t lda, const void* W, int32_t ldw, int32_t w_rows, void* C, int32_t ldc, int32_t M,
                                        int32_t N, int32_t K, const void* bias, int32_t group_in, int32_t group_out, int32_t variant, void* stream) {
    if (!A || !W || !C || M <= 0 || N <= 0 || K <= 0 || group_in <= 0) return fail(nullptr, VQA_ERR_INVALID_ARG, "bad gemm argument");
    if (lda % 8 || ldw % 8 || ldc % 8 || N % 8 || K % 8) return fail(nullptr, VQA_ERR_INVALID_ARG, "gemm: ld/N/K must be multiples of 8");
    cudaError_t e = run_gemm((const bf16*)A, lda, (const bf16*)W, ldw, w_rows, (bf16*)C, ldc, M, N, K, (const bf16*)bias, nullptr, 0, EPI_STORE, 0, variant,
                             device_sms(), (cudaStream_t)stream, nullptr, false, nullptr, group_in, group_out);
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("gemm launch: ") + cudaGetErrorString(e));
    return VQA_OK;
}

// Skinny GEMM (M <= 128) with the K range cut into slices that run as one launch, partial tiles in `workspace` (fp32, splits * M * N floats; the
// slice count the library would pick is returned in *splits_out when splits == 0): C = [residual +] bf16(A W^T + bias).
extern "C" int vqa_op_gemm_bf16_splitk(const void* A, int32_t lda, const void* W, int32_t ldw, int32_t w_rows, void* C, int32_t ldc, int32_t M, int32_t N,
                                       int32_t K, const void* bias, const void* residual, int32_t ldr, int32_t splits, void* workspace,
                                       size_t workspace_bytes, int32_t* splits_out, void* stream) {
    if (!A || !W || !C || M <= 0 || N <= 0 || K <= 0) return fail(nullptr, VQA_ERR_INVALID_ARG, "bad gemm argument");
    if (lda % 8 || ldw % 8 || ldc % 8 || N % 8 || K % 8) return fail(nullptr, VQA_ERR_INVALID_ARG, "gemm: ld/N/K must be multiples of 8");
    if (splits == 0) splits = splitk_slices(M, N, K, device_sms());
    if (splits_out) *splits_out = splits;
    if (splits < 1 || K % (splits * 64)) return fail(nullptr, VQA_ERR_INVALID_ARG, "split-K: K must be a multiple of splits * 64");
    if (!workspace || workspace_bytes < (size_t)splits * M * N * 4) return fail(nullptr, VQA_ERR_WORKSPACE, "split-K workspace too small");
    cudaError_t e = run_gemm_splitk((const bf16*)A, lda, (const bf16*)W, ldw, w_rows, (bf16*)C, ldc, M, N, K, (const bf16*)bias, (const bf16*)residual, ldr,
                                    splits, (float*)workspace, device_sms(), (cudaStream_t)stream, nullptr);
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("gemm launch: ") + cudaGetErrorString(e));
    return VQA_OK;
}

// vqa_op_gemm_bf16 with the fused-RMSNorm hooks (GemmParams::ssq_*): ssq_in [M, stride] partial sums of squares of the rows of A (the
// epilogue scales accumulator row m by rsqrt(sum / norm_dim + eps)), ssq_out [M, stride] receives this GEMM's partial sums of squares of the
// rows it stores (epilogue 0 only); either may be NULL. *parts_out (HOST, optional) = number of slots of ssq_out this launch writes.
extern "C" int vqa_op_gemm_bf16_normfuse(const void* A, int32_t lda, const void* W, int32_t ldw, int32_t w_rows, void* C, int32_t ldc, int32_t M,
                                         int32_t N, int32_t K, const void* residual, int32_t ldr, int32_t epilogue, int32_t gate_up_offset,
                                         const float* ssq_in, float* ssq_out, int32_t stride, int32_t norm_dim, float eps, int32_t* parts_out,
                                         void* stream) {
    if (!A || !W || !C || M <= 0 || N <= 0 || K <= 0 || stride <= 0 || stride % 4 || norm_dim <= 0)
        return fail(nullptr, VQA_ERR_INVALID_ARG, "bad gemm argument");
    if (lda % 8 || ldw % 8 || ldc % 8 || N % 8 || K % 8) return fail(nullptr, VQA_ERR_INVALID_ARG, "gemm: ld/N/K must be multiples of 8");
    const int variant = pick_variant(M, N, epilogue);
    const int parts = ssq_parts_for(variant, epi_is_gated(epilogue) ? N / 2 : N);
    if (parts_out) *parts_out = parts;
    if (ssq_out && parts > stride) return fail(nullptr, VQA_ERR_INVALID_ARG, "ssq stride smaller than the partial sums this launch writes");
    NormFuse nf;
    nf.ssq_in = ssq_in; nf.ssq_out = ssq_out; nf.stride = stride; nf.inv_dim = 1.0f / (float)norm_dim; nf.eps = eps;
    cudaError_t e = run_gemm((const bf16*)A, lda, (const bf16*)W, ldw, w_rows, (bf16*)C, ldc, M, N, K, nullptr, (const bf16*)residual, ldr, epilogue,
                             gate_up_offset, variant, device_sms(), (cudaStream_t)stream, nullptr, false, &nf);
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("gemm launch: ") + cudaGetErrorString(e));
    return VQA_OK;
}

extern "C" int vqa_op_lmhead_logprob(const void* Hs, int32_t ldh, const void* W, int32_t ldw, int32_t M, int32_t N,
                                     int32_t K, const int32_t* labels, float* logprob, float* scratch, void* stream) {
    if (!Hs || !W || !labels || !logprob || !scratch) return fail(nullptr, VQA_ERR_INVALID_ARG, "null pointer");
    const int ntiles = LMHEAD_PARTS * ((N + LMHEAD_BN - 1) / LMHEAD_BN);
    float* lse_max = scratch;
    float* lse_sum = scratch + (size_t)M * ntiles;
    float* label_logit = scratch + 2 * (size_t)M * ntiles;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = run_lmhead((const bf16*)Hs, ldh, (const bf16*)W, ldw, M, N, K, labels, lse_max, lse_sum, label_logit,
                               device_sms(), st, nullptr);
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("lmhead launch: ") + cudaGetErrorString(e));
    // T = 1: score buffer unused -> reuse finalize with logprobs output only
    lse_finalize_kernel<<<(M + 3) / 4, 128, 0, st>>>(lse_max, lse_sum, label_logit, labels, lse_max /*scratch scores*/,
                                                    logprob, M, 1, ntiles);
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("lse finalize: ") + cudaGetErrorString(e));
    return VQA_OK;
}

extern "C" int vqa_op_attention_d64(const void* qkv, void* out, int32_t B, int32_t S, int32_t H, const int32_t* seq_lens,
                                    const float* bias_table, float scale, int32_t bias_const_from, int32_t round_scores, void* stream) {
    if (!qkv || !out || B <= 0 || S <= 0 || H <= 0) return fail(nullptr, VQA_ERR_INVALID_ARG, "bad attention argument");
    const bf16* q = (const bf16*)qkv;
    cudaError_t e = run_flash(q, q + H * 64, q + 2 * H * 64, 3 * H * 64, (bf16*)out, H * 64, B, S, H, seq_lens, bias_table,
                              scale, bias_const_from, round_scores != 0, (cudaStream_t)stream, nullptr);
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("attention launch: ") + cudaGetErrorString(e));
    return VQA_OK;
}

extern "C" int vqa_op_attention_d128(const void* qkv, int32_t ld, int64_t rows, int32_t q_col0, int32_t k_col0, int32_t v_col0,
                                     void* out, int32_t ldo, int32_t n_seq, int32_t max_len, int32_t S, int32_t q_heads, int32_t kv_group,
                                     const int32_t* cu_seqlens, const int32_t* seq_lens, float scale, int32_t causal, void* stream) {
    if (!qkv || !out || n_seq <= 0 || max_len <= 0 || q_heads <= 0 || kv_group <= 0) return fail(nullptr, VQA_ERR_INVALID_ARG, "bad attention argument");
    cudaError_t e = launch_attn_tc128((const bf16*)qkv, ld, rows, q_col0, k_col0, v_col0, (bf16*)out, ldo, n_seq, max_len, S, q_heads, kv_group,
                                      cu_seqlens, seq_lens, scale, causal != 0, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("attention d128 launch: ") + cudaGetErrorString(e));
    return VQA_OK;
}

// The same kernel with its variable-length extras: a shared key/value prefix per sequence, two short sequences per 128-row tile, compact output heads.
extern "C" int vqa_op_attention_d128_ex(const void* qkv, int32_t ld, int64_t rows, int32_t q_col0, int32_t k_col0, int32_t v_col0,
                                        void* out, int32_t ldo, int32_t n_seq, int32_t max_len, int32_t q_heads, int32_t kv_group,
                                        const int32_t* cu_seqlens, const int32_t* kv_prefix, float scale, int32_t causal,
                                        int32_t pair_sequences, int32_t o_head_stride, int32_t d_out, void* stream) {
    if (!qkv || !out || !cu_seqlens || n_seq <= 0 || max_len <= 0 || q_heads <= 0 || kv_group <= 0)
        return fail(nullptr, VQA_ERR_INVALID_ARG, "bad attention argument");
    cudaError_t e = launch_attn_tc128((const bf16*)qkv, ld, rows, q_col0, k_col0, v_col0, (bf16*)out, ldo, n_seq, max_len, 0, q_heads, kv_group,
                                      cu_seqlens, nullptr, scale, causal != 0, (cudaStream_t)stream, kv_prefix, pair_sequences != 0, o_head_stride, d_out);
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("attention d128 launch: ") + cudaGetErrorString(e));
    return VQA_OK;
}

extern "C" int vqa_op_norm(const void* x, const void* gamma, const void* beta, void* y, int32_t rows, int32_t D, float eps,
                           void* stream) {
    if (!x || !gamma || !y) return fail(nullptr, VQA_ERR_INVALID_ARG, "null pointer");
    cudaError_t e = beta ? run_layernorm((const bf16*)x, (const bf16*)gamma, (const bf16*)beta, (bf16*)y, rows, D, eps,
                                         (cudaStream_t)stream, nullptr)
                         : run_rmsnorm((const bf16*)x, (const bf16*)gamma, (bf16*)y, rows, D, eps, (cudaStream_t)stream,
                                       nullptr);
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("norm launch: ") + cudaGetErrorString(e));
    return VQA_OK;
}

// ---------------------------------------------------------------------------------------------- image pre-processing (SURVEY 8(f)2)
extern "C" size_t vqa_clip_preprocess_workspace_bytes(const int32_t* heights, const int32_t* widths, int32_t n_images,
                                                      int32_t out_size, int32_t pad_to_square) {
    if (!heights || !widths || n_images <= 0 || out_size <= 0) return 0;
    PrePlan plan;
    std::vector<int64_t> off(n_images, 0);
    if (!pre_plan(heights, widths, off.data(), n_images, out_size, pad_to_square != 0, plan)) {
        fail(nullptr, VQA_ERR_INVALID_ARG, plan.error);
        return 0;
    }
    return plan.bytes();
}

template <int LAYOUT>
static int pre_launch(const PrePlan& plan, const void* src, int n_images, const uint8_t* background, const float* mean, const float* stdv,
                      PrePatchGeom geom, void* out, int32_t out_dtype, void* workspace, size_t workspace_bytes, void* host_staging,
                      cudaStream_t st) {
    if (workspace_bytes < plan.bytes()) return fail(nullptr, VQA_ERR_WORKSPACE, "pre-processing workspace too small");
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    cudaError_t e;
    if (host_staging) {
        // caller-owned (pinned) staging: one truly asynchronous copy; the caller keeps the buffer untouched until the stream passes it
        uint8_t* hs = static_cast<uint8_t*>(host_staging);
        memcpy(hs, plan.images.data(), plan.images.size() * sizeof(PreImage));
        memcpy(hs + plan.images_bytes(), plan.tables.data(), plan.tables.size() * sizeof(int));
        e = cudaMemcpyAsync(ws, hs, plan.bytes(), cudaMemcpyHostToDevice, st);
    } else {
        // pageable host -> device: the runtime stages the bytes before returning, so the plan may die with the caller's frame
        e = cudaMemcpyAsync(ws, plan.images.data(), plan.images.size() * sizeof(PreImage), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(ws + plan.images_bytes(), plan.tables.data(), plan.tables.size() * sizeof(int), cudaMemcpyHostToDevice, st);
    }
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("pre-processing table upload: ") + cudaGetErrorString(e));
    const PreImage* d_images = reinterpret_cast<const PreImage*>(ws);
    const int* d_tables = reinterpret_cast<const int*>(ws + plan.images_bytes());
    const uchar3 bg = make_uchar3(background[0], background[1], background[2]);
    const float3 mu = make_float3(mean[0], mean[1], mean[2]), sd = make_float3(stdv[0], stdv[1], stdv[2]);
    dim3 grid(plan.max_tiles, n_images);
    if (out_dtype == VQA_DTYPE_F32) {
        e = cudaFuncSetAttribute(image_preprocess_kernel<float, LAYOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PRE_MAX_SMEM);
        if (e == cudaSuccess)
            image_preprocess_kernel<float, LAYOUT><<<grid, PRE_THREADS, plan.smem, st>>>(static_cast<const uint8_t*>(src), d_images, d_tables, bg,
                                                                                        mu, sd, geom, static_cast<float*>(out));
    } else {
        e = cudaFuncSetAttribute(image_preprocess_kernel<bf16, LAYOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PRE_MAX_SMEM);
        if (e == cudaSuccess)
            image_preprocess_kernel<bf16, LAYOUT><<<grid, PRE_THREADS, plan.smem, st>>>(static_cast<const uint8_t*>(src), d_images, d_tables, bg,
                                                                                       mu, sd, geom, static_cast<bf16*>(out));
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return fail(nullptr, VQA_ERR_CUDA, std::string("pre-processing launch: ") + cudaGetErrorString(e));
    return VQA_OK;
}

extern "C" int vqa_clip_preprocess(const void* src, const int64_t* offsets, const int32_t* heights, const int32_t* widths,
                                   int32_t n_images, int32_t out_size, int32_t pad_to_square, const uint8_t* background,
                                   const float* mean, const float* stdv, void* out, int32_t out_dtype, void* workspace,
                                   size_t workspace_bytes, void* host_staging, void* stream) {
    if (!src || !offsets || !heights || !widths || !background || !mean || !stdv || !out || !workspace)
        return fail(nullptr, VQA_ERR_INVALID_ARG, "null pointer");
    if (n_images <= 0 || out_size <= 0) return fail(nullptr, VQA_ERR_INVALID_ARG, "bad size");
    if (out_dtype != VQA_DTYPE_F32 && out_dtype != VQA_DTYPE_BF16) return fail(nullptr, VQA_ERR_INVALID_ARG, "out_dtype must be f32 or bf16");
    PrePlan plan;
    if (!pre_plan(heights, widths, offsets, n_images, out_size, pad_to_square != 0, plan)) return fail(nullptr, VQA_ERR_INVALID_ARG, plan.error);
    return pre_launch<PRE_CHW>(plan, src, n_images, background, mean, stdv, PrePatchGeom{1, 1, 1}, out, out_dtype, workspace, workspace_bytes,
                               host_staging, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int vqa_qwen_preprocess_plan(const int32_t* heights, const int32_t* widths, int32_t n_images, int32_t patch, int32_t merge,
                                        int64_t min_pixels, int64_t max_pixels, int32_t* grid_hw, int64_t* total_patches,
                                        size_t* workspace_bytes) {
    if (!heights || !widths || n_images <= 0 || patch <= 0 || merge <= 0 || min_pixels <= 0 || max_pixels < min_pixels)
        return fail(nullptr, VQA_ERR_INVALID_ARG, "bad argument");
    PrePlan plan;
    std::vector<int64_t> off(n_images, 0);
    long long rows = 0;
    if (!pre_plan_qwen(heights, widths, off.data(), n_images, patch, merge, 1, min_pixels, max_pixels, plan, grid_hw, &rows))
        return fail(nullptr, VQA_ERR_INVALID_ARG, plan.error);
    if (total_patches) *total_patches = rows;
    if (workspace_bytes) *workspace_bytes = plan.bytes();
    return VQA_OK;
}

extern "C" int vqa_qwen_preprocess(const void* src, const int64_t* offsets, const int32_t* heights, const int32_t* widths, int32_t n_images,
                                   int32_t patch, int32_t temporal_patch, int32_t merge, int64_t min_pixels, int64_t max_pixels,
                                   const float* mean, const float* stdv, void* out, int32_t out_dtype, void* workspace,
                                   size_t workspace_bytes, void* host_staging, void* stream) {
    if (!src || !offsets || !heights || !widths || !mean || !stdv || !out || !workspace) return fail(nullptr, VQA_ERR_INVALID_ARG, "null pointer");
    if (n_images <= 0 || patch <= 0 || merge <= 0 || temporal_patch <= 0 || min_pixels <= 0 || max_pixels < min_pixels)
        return fail(nullptr, VQA_ERR_INVALID_ARG, "bad argument");
    if (out_dtype != VQA_DTYPE_F32 && out_dtype != VQA_DTYPE_BF16) return fail(nullptr, VQA_ERR_INVALID_ARG, "out_dtype must be f32 or bf16");
    PrePlan plan;
    if (!pre_plan_qwen(heights, widths, offsets, n_images, patch, merge, temporal_patch, min_pixels, max_pixels, plan, nullptr, nullptr))
        return fail(nullptr, VQA_ERR_INVALID_ARG, plan.error);
    const uint8_t no_bg[3] = {0, 0, 0};
    return pre_launch<PRE_QWEN_PATCHES>(plan, src, n_images, no_bg, mean, stdv, PrePatchGeom{patch, merge, temporal_patch}, out, out_dtype,
                                        workspace, workspace_bytes, host_staging, reinterpret_cast<cudaStream_t>(stream));
}

// Host-only: the fixed-point tap table of one resize axis, exactly as vqa_clip_preprocess builds it (for CPU tests of the host logic).
// bounds: [count][2] (first source index, taps used), kk: [count][ksize] with ksize = return value (call with kk = NULL to size it).
extern "C" int32_t vqa_resample_table(int32_t in_size, int32_t out_size, int32_t first, int32_t count, int32_t* bounds, int32_t* kk) {
    if (in_size <= 0 || out_size <= 0 || first < 0 || count <= 0 || first + count > out_size) {
        fail(nullptr, VQA_ERR_INVALID_ARG, "bad resample table request");
        return 0;
    }
    std::vector<int> tab;
    const int ksize = pre_build_table(in_size, out_size, first, count, tab);
    if (bounds) memcpy(bounds, tab.data(), (size_t)count * 2 * sizeof(int));
    if (kk) memcpy(kk, tab.data() + (size_t)count * 2, (size_t)count * ksize * sizeof(int));
    return ksize;
}

// ---------------------------------------------------------------------------------------------- Qwen video pre-processing
extern "C" int vqa_qwen_video_preprocess_plan(const int32_t* heights, const int32_t* widths, const int32_t* frames, const int32_t* policy,
                                              int32_t n_videos, int32_t patch, int32_t temporal_patch, int32_t merge,
                                              const int64_t* min_pixels, const int64_t* max_pixels, int32_t* grid_thw,
                                              int64_t* total_patches, size_t* workspace_bytes) {
    if (!heights || !widths || !frames || !policy || !min_pixels || !max_pixels || n_videos <= 0 || patch <= 0 || merge <= 0 ||
        temporal_patch <= 0)
        return fail(nullptr, VQA_ERR_INVALID_ARG, "bad argument");
    PrePlan plan;
    std::vector<int64_t> off(n_videos, 0);
    long long rows = 0;
    if (!pre_plan_qwen_video(heights, widths, frames, policy, off.data(), n_videos, patch, merge, temporal_patch, min_pixels, max_pixels,
                             plan, grid_thw, &rows))
        return fail(nullptr, VQA_ERR_INVALID_ARG, plan.error);
    if (total_patches) *total_patches = rows;
    if (workspace_bytes) *workspace_bytes = plan.bytes();
    return VQA_OK;
}

extern "C" int vqa_qwen_video_preprocess(const void* src, const int64_t* offsets, const int32_t* heights, const int32_t* widths,
                                         const int32_t* frames, const int32_t* policy, int32_t n_videos, int32_t patch,
                                         int32_t temporal_patch, int32_t merge, const int64_t* min_pixels, const int64_t* max_pixels,
                                         const float* mean, const float* stdv, void* out, int32_t out_dtype, void* workspace,
                                         size_t workspace_bytes, void* host_staging, void* stream) {
    if (!src || !offsets || !heights || !widths || !frames || !policy || !min_pixels || !max_pixels || !mean || !stdv || !out || !workspace)
        return fail(nullptr, VQA_ERR_INVALID_ARG, "null pointer");
    if (n_videos <= 0 || patch <= 0 || merge <= 0 || temporal_patch <= 0) return fail(nullptr, VQA_ERR_INVALID_ARG, "bad argument");
    if (out_dtype != VQA_DTYPE_F32 && out_dtype != VQA_DTYPE_BF16) return fail(nullptr, VQA_ERR_INVALID_ARG, "out_dtype must be f32 or bf16");
    PrePlan plan;
    if (!pre_plan_qwen_video(heights, widths, frames, policy, offsets, n_videos, patch, merge, temporal_patch, min_pixels, max_pixels, plan,
                             nullptr, nullptr))
        return fail(nullptr, VQA_ERR_INVALID_ARG, plan.error);
    const uint8_t no_bg[3] = {0, 0, 0};
    return pre_launch<PRE_QWEN_PATCHES>(plan, src, (int)plan.images.size(), no_bg, mean, stdv, PrePatchGeom{patch, merge, temporal_patch}, out,
                                        out_dtype, workspace, workspace_bytes, host_staging, reinterpret_cast<cudaStream_t>(stream));
}

// Host-only: the fp32 tap table of one axis of the torchvision-policy resize, exactly as vqa_qwen_video_preprocess builds it (for CPU
// replays of the kernel's arithmetic). bounds: [count][2] (first source index, taps used), taps: [count][ksize] with ksize = return value
// (call with taps = NULL to size it); *fma = 1 when the pass over this axis accumulates with fma, 0 when it rounds each product first.
extern "C" int32_t vqa_resample_table_tv(int32_t in_size, int32_t out_size, int32_t first, int32_t count, int32_t* bounds, float* taps,
                                         int32_t* fma) {
    if (in_size <= 0 || out_size <= 0 || first < 0 || count <= 0 || first + count > out_size) {
        fail(nullptr, VQA_ERR_INVALID_ARG, "bad resample table request");
        return 0;
    }
    std::vector<int> tab;
    int f = 0;
    const int ksize = pre_build_table_tv(in_size, out_size, first, count, tab, &f);
    if (bounds) memcpy(bounds, tab.data(), (size_t)count * 2 * sizeof(int));
    if (taps) memcpy(taps, tab.data() + (size_t)count * 2, (size_t)count * ksize * sizeof(float));
    if (fma) *fma = f;
    return ksize;
}
