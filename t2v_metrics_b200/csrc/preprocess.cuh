// CLIP image pre-processing on the device (SURVEY 8(f)2): expand2square + bicubic resize + centre crop + rescale + normalise.
//
// What it replaces: t2v_metrics/models/vqascore_models/mm_utils.py:128-139 (expand2square) followed by the CLIP image processor
// of the v3.0 wrapper (resize shortest edge to S with PIL BICUBIC, centre crop SxS, /255, (x - mean) / std), i.e.
// oracle/clipt5_oracle.py:clip_preprocess. The resize is Pillow's (third-party dependency of the reference, not vendored;
// installed 12.2.0, src/libImaging/Resample.c): a separable convolution with per-output-pixel windows, coefficients normalised in
// double and quantised to 22-bit fixed point, the horizontal pass first, its result ROUNDED TO uint8, then the vertical pass. The
// coefficient tables are built on the host in double exactly as Pillow builds them (so the integers are identical), the two integer
// passes run here, and the result is bit-identical to PIL for every pixel.
//
// One CTA = one image x one band of `tile_rows` output rows. The canvas rows the band needs are staged 8 at a time into shared memory
// as three byte PLANES packed four pixels to a word (padding colour filled in, so the passes need no bounds checks). Each 22-bit tap is
// split on the host into three byte digits (k = d0 + 256 d1 + 65536 d2, d2 signed) and laid out in words aligned to the same groups of
// four pixels, so one `dp4a` multiplies four pixels by four tap digits: 3 dp4a per 4 taps per channel, exact in int32
// (acc0 + (acc1 << 8) + (acc2 << 16) is the same integer Pillow accumulates). The horizontal pass writes its uint8 result four ROWS
// to a word, which is the packing the vertical pass needs; a 768-entry table does /255, -mean, /std in exact fp32. The source is read
// once from HBM (plus the band overlap, absorbed by L2), the output written once.
#pragma once
#include <cmath>
#include <cstdint>
#include <string>
#include <vector>
#include "ptx.cuh"

namespace vqa {

constexpr int PRE_PRECISION_BITS = 32 - 8 - 2;      // Resample.c PRECISION_BITS
constexpr int PRE_THREADS = 256;
constexpr int PRE_XL = 128;                         // x lanes; PRE_THREADS / PRE_XL row groups of 4 canvas rows each
constexpr int PRE_RG = PRE_THREADS / PRE_XL;
constexpr int PRE_MAX_SMEM = 200 * 1024;

struct PreImage {            // one per image, lives in the workspace (device) and is built on the host
    long long src_off;       // byte offset of the HWC uint8 RGB image inside `src`
    int h, w;                // stored image
    int paste_x, paste_y;    // where the stored image sits on the (virtual) square canvas; 0 when not padded
    int canvas_h, canvas_w;  // canvas the resize reads (= max(h, w) squared when padded, else h x w)
    int htab, vtab;          // int offsets of the packed tap tables inside the workspace (layout: see pre_pack_table)
    int hnp, vnp;            // words of 4 taps per output pixel (horizontal / vertical)
    int tile_rows;           // output rows per CTA
    int band_groups;         // groups of 4 canvas rows the band buffer holds
    int out_h, out_w;        // output window (after the crop) of this image
    long long out_off;       // element offset of this image's output inside `out`
    int x_lo4, span4;        // groups of 4 canvas columns [x_lo4, x_lo4 + span4) the horizontal tap words touch
    int chunk_groups;        // groups of 4 canvas rows staged per pass (1 or 2)
    int policy;              // PRE_PIL (22-bit fixed point, uint8 intermediate) or PRE_TORCHVISION (fp32 taps and intermediate)
    int hfma, vfma;          // PRE_TORCHVISION: the pass accumulates with fma (1) or with a rounded product then an add (0)
    int t_lo, t_hi;          // PRE_QWEN_PATCHES: the temporal slots [t_lo, t_hi) this frame is written to
};

enum PreLayout { PRE_CHW = 0, PRE_QWEN_PATCHES = 1 };
enum PrePolicy { PRE_PIL = 0, PRE_TORCHVISION = 1 };
struct PrePatchGeom { int patch, merge, temporal; };     // PRE_QWEN_PATCHES only

// ---------------------------------------------------------------------------------------------- host: Pillow's coefficient tables
inline double pre_bicubic(double x) {                 // Resample.c bicubic_filter, a = -0.5
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}

// precompute_coeffs + normalize_coeffs_8bpc for output pixels [first, first + count) of an in_size -> out_size resize over the whole
// axis (box = [0, in_size)). Appends bounds (xmin, n) pairs then count * ksize fixed-point taps to `tab`; returns ksize.
inline int pre_build_table(int in_size, int out_size, int first, int count, std::vector<int>& tab) {
    const float in0 = 0.f, in1 = (float)in_size;
    double scale = (double)(in1 - in0) / out_size;
    double filterscale = scale;
    if (filterscale < 1.0) filterscale = 1.0;
    const double support = 2.0 * filterscale;          // BICUBIC.support = 2.0
    const int ksize = (int)std::ceil(support) * 2 + 1;
    const size_t base = tab.size();
    tab.resize(base + (size_t)count * 2 + (size_t)count * ksize, 0);
    int* bounds = tab.data() + base;
    int* kk = bounds + (size_t)count * 2;
    std::vector<double> k(ksize);
    for (int i = 0; i < count; ++i) {
        const int xx = first + i;
        const double center = in0 + (xx + 0.5) * scale;
        double ww = 0.0;
        const double ss = 1.0 / filterscale;
        int xmin = (int)(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = (int)(center + support + 0.5);
        if (xmax > in_size) xmax = in_size;
        xmax -= xmin;
        for (int x = 0; x < xmax; ++x) {
            const double w = pre_bicubic((x + xmin - center + 0.5) * ss);
            k[x] = w;
            ww += w;
        }
        for (int x = 0; x < xmax; ++x)
            if (ww != 0.0) k[x] /= ww;
        for (int x = 0; x < ksize; ++x) {
            const double v = x < xmax ? k[x] : 0.0;
            kk[(size_t)i * ksize + x] = v < 0 ? (int)(-0.5 + v * (1 << PRE_PRECISION_BITS)) : (int)(0.5 + v * (1 << PRE_PRECISION_BITS));
        }
        bounds[2 * i] = xmin;
        bounds[2 * i + 1] = xmax;
    }
    return ksize;
}

// Tap words for the dp4a passes, from one axis' (bounds, kk) table of `count` outputs with `ksize` taps each. Appends to `tab`:
//   start4[count]          group (absolute position / 4) of the first tap word of each output
//   last4[count]           group of the last REAL tap
//   words[count][np][3]    byte digits d0 | d1 | d2 of the four taps of each word (zero where the window has no tap)
// and returns np = the largest number of words any output needs.
inline int pre_pack_table(const int* bounds, const int* kk, int count, int ksize, std::vector<int>& tab) {
    int np = 1;
    for (int i = 0; i < count; ++i) {
        const int x0 = bounds[2 * i], n = bounds[2 * i + 1];
        const int words = n > 0 ? (x0 + n - 1) / 4 - x0 / 4 + 1 : 1;
        if (words > np) np = words;
    }
    const size_t base = tab.size();
    tab.resize(base + (size_t)count * 2 + (size_t)count * np * 3, 0);
    int* start4 = tab.data() + base;
    int* last4 = start4 + count;
    unsigned* words = reinterpret_cast<unsigned*>(last4 + count);
    for (int i = 0; i < count; ++i) {
        const int x0 = bounds[2 * i], n = bounds[2 * i + 1];
        start4[i] = x0 / 4;
        last4[i] = n > 0 ? (x0 + n - 1) / 4 : x0 / 4;
        for (int x = 0; x < n; ++x) {
            const int a = x0 + x, w = a / 4 - start4[i], b = a % 4;
            const int k = kk[(size_t)i * ksize + x];
            unsigned* q = words + ((size_t)i * np + w) * 3;
            q[0] |= (unsigned)(k & 0xff) << (8 * b);
            q[1] |= (unsigned)((k >> 8) & 0xff) << (8 * b);
            q[2] |= (unsigned)((k >> 16) & 0xff) << (8 * b);          // arithmetic shift: the signed top digit
        }
    }
    return np;
}

// ---------------------------------------------------------------------------------------------- host: torch's antialiased bicubic taps
// What torchvision.transforms.functional.resize(uint8 tensor, BICUBIC, antialias=True) computes: a cast to fp32, then
// F.interpolate(mode="bicubic", antialias=True) (aten/src/ATen/native/cpu/UpSampleKernel.cpp, HelperInterpCubic with a = -0.5 and
// _compute_indices_min_size_weights_aa), then clamp(0, 255) and round-half-even back to uint8. The taps below reproduce torch's CPU
// build (x86-64, compiled with FMA contraction) bit for bit: the filter polynomials as fused multiply-adds, `center -/+ support` in
// fp32 before the + 0.5 in double, the argument (x - center) in fp32 then (+ 0.5) * invscale in double, weights normalised by their
// fp32 sum. The passes run width first, then height, each over an fp32 intermediate. torch accumulates `acc += px * w` sequentially
// from the first tap; its build contracts that to an fma on upscaled axes and keeps a rounded product on downscaled ones (probed on
// torch 2.11 CPU), which is what `fma` returns. Both are a compiler's choice, not part of torch's API: a build that contracts
// differently moves results by one grey level where the fp32 sum sits at a rounding tie (measured in the tests).
inline float pre_tv_cubic(float x) {
    const float a = -0.5f;
    x = std::fabs(x);
    if (x < 1.0f) return std::fmaf(std::fmaf(a + 2.0f, x, -(a + 3.0f)) * x, x, 1.0f);
    if (x < 2.0f) return std::fmaf(std::fmaf(std::fmaf(a, x, -5.0f * a), x, 8.0f * a), x, -4.0f * a);
    return 0.0f;
}

// Taps of output pixels [first, first + count) of an in_size -> out_size resize. Appends (xmin, n) bounds then count * ksize taps (fp32
// bit patterns) to `tab`; returns ksize. `fma`: whether the passes over this axis accumulate with fma.
inline int pre_build_table_tv(int in_size, int out_size, int first, int count, std::vector<int>& tab, int* fma) {
    const float scale = (float)in_size / (float)out_size;
    const float support = scale >= 1.0f ? 2.0f * scale : 2.0f;           // (interp_size * 0.5) * scale, interp_size = 4
    const float invscale = scale >= 1.0f ? 1.0f / scale : 1.0f;
    const int ksize = (int)std::ceil(support) * 2 + 1;
    const size_t base = tab.size();
    tab.resize(base + (size_t)count * 2 + (size_t)count * ksize, 0);
    int* bounds = tab.data() + base;
    float* kk = reinterpret_cast<float*>(bounds + (size_t)count * 2);
    for (int i = 0; i < count; ++i) {
        const int xx = first + i;
        const float center = (float)((double)scale * (xx + 0.5));
        int xmin = (int)((double)(center - support) + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = (int)((double)(center + support) + 0.5);
        if (xmax > in_size) xmax = in_size;
        int n = xmax - xmin;
        if (n > ksize) n = ksize;
        if (n < 0) n = 0;
        float* w = kk + (size_t)i * ksize;
        float total = 0.0f;
        for (int j = 0; j < n; ++j) {
            const float d = (float)(j + xmin) - center;
            w[j] = pre_tv_cubic((float)(((double)d + 0.5) * (double)invscale));
            total += w[j];
        }
        if (total != 0.0f)
            for (int j = 0; j < n; ++j) w[j] /= total;
        bounds[2 * i] = xmin;
        bounds[2 * i + 1] = n;
    }
    if (fma) *fma = out_size > in_size ? 1 : 0;
    return ksize;
}

// pre_pack_table for fp32 taps: start4[count], last4[count], then taps[count][np][4] (fp32, aligned to the same groups of four source
// pixels, zero where the window has no tap: a zero tap adds an exact zero under either accumulation). Returns np.
inline int pre_pack_table_tv(const int* bounds, const float* kk, int count, int ksize, std::vector<int>& tab) {
    int np = 1;
    for (int i = 0; i < count; ++i) {
        const int x0 = bounds[2 * i], n = bounds[2 * i + 1];
        const int words = n > 0 ? (x0 + n - 1) / 4 - x0 / 4 + 1 : 1;
        if (words > np) np = words;
    }
    const size_t base = tab.size();
    tab.resize(base + (size_t)count * 2 + (size_t)count * np * 4, 0);
    int* start4 = tab.data() + base;
    int* last4 = start4 + count;
    float* taps = reinterpret_cast<float*>(last4 + count);
    for (int i = 0; i < count; ++i) {
        const int x0 = bounds[2 * i], n = bounds[2 * i + 1];
        start4[i] = x0 / 4;
        last4[i] = n > 0 ? (x0 + n - 1) / 4 : x0 / 4;
        for (int x = 0; x < n; ++x) taps[((size_t)i * np) * 4 + (x0 + x) - 4 * start4[i]] = kk[(size_t)i * ksize + x];
    }
    return np;
}

// ---------------------------------------------------------------------------------------------- device
__device__ __forceinline__ int pre_clip8(int v) {     // Resample.c clip8: table lookup of (v >> PRECISION_BITS) clamped to [0, 255]
    v >>= PRE_PRECISION_BITS;
    return v < 0 ? 0 : (v > 255 ? 255 : v);
}
__device__ __forceinline__ unsigned pre_dp4a_uu(unsigned a, unsigned b, unsigned c) {      // 4 x (u8 * u8) + c
    unsigned d;
    asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int pre_dp4a_us(unsigned a, unsigned b, int c) {                // 4 x (u8 * s8) + c
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// the integer Pillow accumulates, rounded and clipped: sum(px * k) + 2^21 with k = d0 + 256 d1 + 65536 d2
__device__ __forceinline__ unsigned pre_finish(unsigned a0, unsigned a1, int a2) {
    const unsigned t = a0 + (a1 << 8) + ((unsigned)a2 << 16) + (1u << (PRE_PRECISION_BITS - 1));
    return (unsigned)pre_clip8((int)t);
}

// LAYOUT PRE_CHW: out[c][y][x] per image ([3, out_h, out_w]). PRE_QWEN_PATCHES: the Qwen2-VL processor's patch rows
// (image_processing_qwen2_vl.py:191-220): row ((by * gw/m + bx) * m + iy) * m + ix for the 14x14 patch at grid (by*m+iy, bx*m+ix),
// column (c * temporal + t) * ps*ps + py * ps + px, the frame written to temporal slots [t_lo, t_hi) (a still image: all of them).
// Per image, `policy` selects the resample: PRE_PIL (the dp4a fixed-point passes above, uint8 intermediate) or PRE_TORCHVISION (fp32
// taps, fp32 intermediate, clamp + round-half-even at the end; see pre_build_table_tv). Both share the staging, the band and the
// output stage; only the two filter passes differ.
template <typename OUT, int LAYOUT>
__global__ void __launch_bounds__(PRE_THREADS, 3)     // 3 CTAs an SM, as before the fp32 passes joined: no spills at 79 registers
image_preprocess_kernel(const uint8_t* __restrict__ src, const PreImage* __restrict__ images, const int* __restrict__ tables,
                        uchar3 background, float3 mean, float3 stdv, PrePatchGeom geom, OUT* __restrict__ out) {
    pdl_launch_dependents();
    extern __shared__ uint32_t pre_smem[];
    const PreImage im = images[blockIdx.y];
    const int y0 = blockIdx.x * im.tile_rows;
    if (y0 >= im.out_h) return;
    const int out_w = im.out_w;
    const int ny = min(im.tile_rows, im.out_h - y0);
    const int chunk_rows = im.chunk_groups * 4;
    float* lut = reinterpret_cast<float*>(pre_smem);                          // [3][256] normalised value of every grey level
    const bool tv = im.policy == PRE_TORCHVISION;
    uint32_t* band = pre_smem + 768;                                           // [3][band_groups][out_w]: 4 canvas rows per word
    float* bandf = reinterpret_cast<float*>(band);                             // PRE_TORCHVISION: [3][band_groups * 4][out_w] fp32
    uint32_t* stage = band + (size_t)3 * im.band_groups * out_w * (tv ? 4 : 1);  // [3][chunk_rows][span4]: 4 canvas columns per word
    const int* hstart = tables + im.htab;
    const uint32_t* hwords = reinterpret_cast<const uint32_t*>(hstart + 2 * out_w);
    const int* vstart = tables + im.vtab;
    const int* vlast = vstart + im.out_h;
    const uint32_t* vwords = reinterpret_cast<const uint32_t*>(vstart + 2 * im.out_h);
    // groups of 4 canvas rows this band needs: the windows are monotonic in y
    const int g0 = vstart[y0];
    const int ng = vlast[y0 + ny - 1] - g0 + 1;
    const uint8_t* img = src + im.src_off;
    const unsigned bgc[3] = {background.x, background.y, background.z};
    const int lane_x = threadIdx.x % PRE_XL, grp = threadIdx.x / PRE_XL;

    // out = ((u8 / 255) - mean[c]) / std[c] in fp32 with IEEE division and no fma, as numpy / torch compute it on the host
    for (int i = threadIdx.x; i < 768; i += PRE_THREADS) {
        const int c = i >> 8;
        const float mu = c == 0 ? mean.x : (c == 1 ? mean.y : mean.z), sd = c == 0 ? stdv.x : (c == 1 ? stdv.y : stdv.z);
        lut[i] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)(i & 255), 255.0f), mu), sd);
    }

    for (int cg = 0; cg < ng; cg += im.chunk_groups) {
        const int ngc = min(im.chunk_groups, ng - cg);
        // ---- stage canvas rows 4 (g0 + cg) ... as byte planes, 4 columns per word; outside the pasted image = padding colour
        for (int rr = 0; rr < ngc * 4; ++rr) {
            const int sy = 4 * (g0 + cg) + rr - im.paste_y;
            const bool row_in = sy >= 0 && sy < im.h;
            const uint8_t* row = img + (size_t)(row_in ? sy : 0) * im.w * 3;
            for (int gx = threadIdx.x; gx < im.span4; gx += PRE_THREADS) {
                const int sx0 = 4 * (im.x_lo4 + gx) - im.paste_x;
                uint32_t pr, pg, pb;
                if (row_in && sx0 >= 0 && sx0 + 3 < im.w) {
                    const uint8_t* p = row + (size_t)sx0 * 3;
                    if ((reinterpret_cast<uintptr_t>(p) & 3) == 0) {           // 12 aligned bytes: R0G0B0R1 G1B1R2G2 B2R3G3B3
                        const uint32_t w0 = reinterpret_cast<const uint32_t*>(p)[0], w1 = reinterpret_cast<const uint32_t*>(p)[1],
                                       w2 = reinterpret_cast<const uint32_t*>(p)[2];
                        pr = __byte_perm(__byte_perm(w0, w1, 0x0630), w2, 0x5210);
                        pg = __byte_perm(__byte_perm(w0, w1, 0x0741), w2, 0x6210);
                        pb = __byte_perm(__byte_perm(w0, w1, 0x0052), w2, 0x7410);
                    } else {
                        pr = p[0] | (p[3] << 8) | (p[6] << 16) | ((uint32_t)p[9] << 24);
                        pg = p[1] | (p[4] << 8) | (p[7] << 16) | ((uint32_t)p[10] << 24);
                        pb = p[2] | (p[5] << 8) | (p[8] << 16) | ((uint32_t)p[11] << 24);
                    }
                } else {
                    pr = pg = pb = 0;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int sx = sx0 + i;
                        const bool in = row_in && sx >= 0 && sx < im.w;
                        const uint8_t* p = row + (size_t)(in ? sx : 0) * 3;
                        pr |= (in ? (uint32_t)p[0] : bgc[0]) << (8 * i);
                        pg |= (in ? (uint32_t)p[1] : bgc[1]) << (8 * i);
                        pb |= (in ? (uint32_t)p[2] : bgc[2]) << (8 * i);
                    }
                }
                stage[(size_t)(0 * chunk_rows + rr) * im.span4 + gx] = pr;
                stage[(size_t)(1 * chunk_rows + rr) * im.span4 + gx] = pg;
                stage[(size_t)(2 * chunk_rows + rr) * im.span4 + gx] = pb;
            }
        }
        __syncthreads();
        // ---- horizontal pass, torchvision policy: fp32 taps over the staged bytes, sequential from the window's first tap
        if (tv && grp < ngc) {
            const float* htaps = reinterpret_cast<const float*>(hstart + 2 * out_w);
            for (int xx = lane_x; xx < out_w; xx += PRE_XL) {
                const int s4 = hstart[xx] - im.x_lo4;
                const float* kw = htaps + (size_t)xx * im.hnp * 4;
                float acc[4][3];
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int c = 0; c < 3; ++c) acc[q][c] = 0.0f;
                for (int pw = 0; pw < im.hnp; ++pw) {
                    float k[4];
#pragma unroll
                    for (int b = 0; b < 4; ++b) k[b] = __ldg(kw + pw * 4 + b);
#pragma unroll
                    for (int q = 0; q < 4; ++q)
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            const uint32_t px = stage[(size_t)(c * chunk_rows + grp * 4 + q) * im.span4 + s4 + pw];
#pragma unroll
                            for (int b = 0; b < 4; ++b) {
                                const float p = (float)((px >> (8 * b)) & 0xffu);
                                acc[q][c] = im.hfma ? __fmaf_rn(p, k[b], acc[q][c]) : __fadd_rn(acc[q][c], __fmul_rn(p, k[b]));
                            }
                        }
                }
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int q = 0; q < 4; ++q) bandf[((size_t)c * im.band_groups * 4 + (cg + grp) * 4 + q) * out_w + xx] = acc[q][c];
            }
        }
        // ---- horizontal pass (ImagingResampleHorizontal_8bpc): thread = one output column x one group of 4 canvas rows
        if (!tv && grp < ngc) {
            for (int xx = lane_x; xx < out_w; xx += PRE_XL) {
                const int s4 = hstart[xx] - im.x_lo4;
                const uint32_t* kw = hwords + (size_t)xx * im.hnp * 3;
                unsigned a0[4][3], a1[4][3];
                int a2[4][3];
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int c = 0; c < 3; ++c) { a0[q][c] = 0; a1[q][c] = 0; a2[q][c] = 0; }
                for (int pw = 0; pw < im.hnp; ++pw) {
                    const uint32_t d0 = __ldg(kw + pw * 3), d1 = __ldg(kw + pw * 3 + 1), d2 = __ldg(kw + pw * 3 + 2);
#pragma unroll
                    for (int q = 0; q < 4; ++q)
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            const uint32_t px = stage[(size_t)(c * chunk_rows + grp * 4 + q) * im.span4 + s4 + pw];
                            a0[q][c] = pre_dp4a_uu(px, d0, a0[q][c]);
                            a1[q][c] = pre_dp4a_uu(px, d1, a1[q][c]);
                            a2[q][c] = pre_dp4a_us(px, d2, a2[q][c]);
                        }
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    uint32_t wv = 0;
#pragma unroll
                    for (int q = 0; q < 4; ++q) wv |= pre_finish(a0[q][c], a1[q][c], a2[q][c]) << (8 * q);
                    band[((size_t)c * im.band_groups + cg + grp) * out_w + xx] = wv;
                }
            }
        }
        __syncthreads();
    }

    // ---- vertical pass (ImagingResampleVertical_8bpc) + normalisation
    OUT* dst = out + im.out_off;
    const int ps = geom.patch, mg = geom.merge, pp = geom.patch * geom.patch;
    const int gwm = LAYOUT == PRE_QWEN_PATCHES ? out_w / (ps * mg) : 0;
    for (int yy = grp; yy < ny; yy += PRE_RG) {
        const int y = y0 + yy;
        const int gs = vstart[y] - g0;
        const uint32_t* kw = vwords + (size_t)y * im.vnp * 3;
        const float* kf = reinterpret_cast<const float*>(vwords) + (size_t)y * im.vnp * 4;
        const int vn = vlast[y] - vstart[y] + 1;            // torchvision policy: only groups this CTA staged (fp32 garbage is not inert)
        for (int xx = lane_x; xx < out_w; xx += PRE_XL) {
            float v[3];
            if (tv) {
                float acc[3] = {0.0f, 0.0f, 0.0f};
                for (int pw = 0; pw < vn; ++pw) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const float k = __ldg(kf + pw * 4 + b);
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            const float p = bandf[((size_t)c * im.band_groups * 4 + (gs + pw) * 4 + b) * out_w + xx];
                            acc[c] = im.vfma ? __fmaf_rn(p, k, acc[c]) : __fadd_rn(acc[c], __fmul_rn(p, k));
                        }
                    }
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) v[c] = lut[c * 256 + (int)rintf(fminf(fmaxf(acc[c], 0.0f), 255.0f))];
            } else {
                unsigned a0[3] = {0, 0, 0}, a1[3] = {0, 0, 0};
                int a2[3] = {0, 0, 0};
                for (int pw = 0; pw < im.vnp; ++pw) {
                    const uint32_t d0 = __ldg(kw + pw * 3), d1 = __ldg(kw + pw * 3 + 1), d2 = __ldg(kw + pw * 3 + 2);
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        const uint32_t px = band[((size_t)c * im.band_groups + gs + pw) * out_w + xx];
                        a0[c] = pre_dp4a_uu(px, d0, a0[c]);
                        a1[c] = pre_dp4a_uu(px, d1, a1[c]);
                        a2[c] = pre_dp4a_us(px, d2, a2[c]);
                    }
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) v[c] = lut[c * 256 + pre_finish(a0[c], a1[c], a2[c])];
            }
            if constexpr (LAYOUT == PRE_CHW) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const size_t o = ((size_t)c * im.out_h + y) * out_w + xx;
                    if constexpr (sizeof(OUT) == 4) dst[o] = v[c];
                    else dst[o] = __float2bfloat16_rn(v[c]);
                }
            } else {
                const int gy = y / ps, py = y - gy * ps, gx = xx / ps, px_ = xx - gx * ps;
                const size_t row = (((size_t)(gy / mg) * gwm + gx / mg) * mg + gy % mg) * mg + gx % mg;
                OUT* q = dst + row * (size_t)(3 * geom.temporal * pp) + py * ps + px_;
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    for (int t = im.t_lo; t < im.t_hi; ++t) {
                        if constexpr (sizeof(OUT) == 4) q[(size_t)(c * geom.temporal + t) * pp] = v[c];
                        else q[(size_t)(c * geom.temporal + t) * pp] = __float2bfloat16_rn(v[c]);
                    }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------- host: plan + launch
struct PrePlan {
    std::vector<PreImage> images;
    std::vector<int> tables;
    int max_tiles = 0;
    size_t smem = 0;
    std::string error;
    size_t images_bytes() const { return (images.size() * sizeof(PreImage) + 15) / 16 * 16; }
    size_t bytes() const { return images_bytes() + tables.size() * sizeof(int); }
};

struct PreTableKey {
    int ch, cw, nh, nw, top, left, oh, ow, htab, vtab, hnp, vnp, tile, band_groups, x_lo4, span4, chunk_groups, policy, hfma, vfma;
};
inline size_t pre_smem_bytes(int band_groups, int out_w, int chunk_groups, int span4, int policy = PRE_PIL) {
    const size_t band_words = (size_t)3 * band_groups * out_w * (policy == PRE_TORCHVISION ? 4 : 1);   // fp32 rows vs 4 uint8 rows a word
    return 768 * sizeof(float) + (band_words + (size_t)3 * chunk_groups * 4 * span4) * sizeof(uint32_t);
}

// Tables + band geometry for "resize the ch x cw canvas to nh x nw, keep the oh x ow window at (top, left)"; shared between images
// with the same geometry. Returns nullptr (plan.error set) when the filter windows cannot fit the shared-memory budget.
inline const PreTableKey* pre_tables(PrePlan& plan, std::vector<PreTableKey>& cache, int ch, int cw, int nh, int nw, int top, int left,
                                     int oh, int ow, int policy = PRE_PIL) {
    for (const PreTableKey& k : cache)
        if (k.ch == ch && k.cw == cw && k.nh == nh && k.nw == nw && k.top == top && k.left == left && k.oh == oh && k.ow == ow &&
            k.policy == policy)
            return &k;
    PreTableKey k{ch, cw, nh, nw, top, left, oh, ow, 0, 0, 0, 0, 0, 0, 0, 0, 0, policy, 0, 0};
    std::vector<int> raw;
    const bool tv = policy == PRE_TORCHVISION;
    int ks = tv ? pre_build_table_tv(cw, nw, left, ow, raw, &k.hfma) : pre_build_table(cw, nw, left, ow, raw);
    k.htab = (int)plan.tables.size();
    k.hnp = tv ? pre_pack_table_tv(raw.data(), reinterpret_cast<const float*>(raw.data() + (size_t)ow * 2), ow, ks, plan.tables)
               : pre_pack_table(raw.data(), raw.data() + (size_t)ow * 2, ow, ks, plan.tables);
    raw.clear();
    ks = tv ? pre_build_table_tv(ch, nh, top, oh, raw, &k.vfma) : pre_build_table(ch, nh, top, oh, raw);
    k.vtab = (int)plan.tables.size();
    k.vnp = tv ? pre_pack_table_tv(raw.data(), reinterpret_cast<const float*>(raw.data() + (size_t)oh * 2), oh, ks, plan.tables)
               : pre_pack_table(raw.data(), raw.data() + (size_t)oh * 2, oh, ks, plan.tables);
    const int* hstart = plan.tables.data() + k.htab;
    const int* vstart = plan.tables.data() + k.vtab;
    k.x_lo4 = hstart[0];                           // windows are monotonic: first word of the first output .. last word of the last
    k.span4 = hstart[ow - 1] + k.hnp - k.x_lo4;
    // output rows per CTA (<= 32) and groups of 4 canvas rows staged per pass (2 or 1): the largest that fit the shared-memory budget
    int tile = 32, band = 0, chunk = PRE_RG;
    for (; tile >= 1; tile >>= 1) {
        band = 0;
        for (int y0 = 0; y0 < oh; y0 += tile) {
            const int y1 = (y0 + tile < oh ? y0 + tile : oh) - 1;
            const int groups = vstart[y1] + k.vnp - vstart[y0];
            if (groups > band) band = groups;
        }
        for (chunk = PRE_RG; chunk > 1 && pre_smem_bytes(band, ow, chunk, k.span4, policy) > (size_t)PRE_MAX_SMEM; chunk >>= 1) {}
        if (pre_smem_bytes(band, ow, chunk, k.span4, policy) <= (size_t)PRE_MAX_SMEM) break;
    }
    if (tile < 1) { plan.error = "image too large for the device resize (filter windows exceed shared memory)"; return nullptr; }
    k.tile = tile; k.band_groups = band; k.chunk_groups = chunk;
    cache.push_back(k);
    return &cache.back();
}

inline void pre_finish_image(PrePlan& plan, PreImage& im, const PreTableKey& k) {
    im.htab = k.htab; im.vtab = k.vtab; im.hnp = k.hnp; im.vnp = k.vnp;
    im.tile_rows = k.tile; im.band_groups = k.band_groups; im.out_h = k.oh; im.out_w = k.ow;
    im.x_lo4 = k.x_lo4; im.span4 = k.span4; im.chunk_groups = k.chunk_groups;
    im.policy = k.policy; im.hfma = k.hfma; im.vfma = k.vfma;
    const int tiles = (k.oh + k.tile - 1) / k.tile;
    if (tiles > plan.max_tiles) plan.max_tiles = tiles;
    const size_t sm = pre_smem_bytes(k.band_groups, k.ow, k.chunk_groups, k.span4, k.policy);
    if (sm > plan.smem) plan.smem = sm;
}

// Geometry of CLIPImageProcessor for one image (shortest edge -> S, int() truncation of the long edge, centre crop S x S), on the
// padded canvas when pad_to_square. Output [n, 3, S, S].
inline bool pre_plan(const int32_t* heights, const int32_t* widths, const int64_t* offsets, int n, int S, bool pad, PrePlan& plan) {
    std::vector<PreTableKey> cache;
    cache.reserve(n);
    plan.images.resize(n);
    for (int i = 0; i < n; ++i) {
        const int h = heights[i], w = widths[i];
        if (h <= 0 || w <= 0) { plan.error = "image with non-positive size"; return false; }
        PreImage& im = plan.images[i];
        im.src_off = offsets[i]; im.h = h; im.w = w;
        const int side = h > w ? h : w;
        im.canvas_h = pad ? side : h; im.canvas_w = pad ? side : w;
        im.paste_x = pad ? (side - w) / 2 : 0; im.paste_y = pad ? (side - h) / 2 : 0;
        const int ch = im.canvas_h, cw = im.canvas_w;
        // get_resize_output_image_size(shortest_edge = S, default_to_square = False): short -> S, long -> int(S * long / short)
        const int nw = cw <= ch ? S : (int)((double)S * cw / ch);
        const int nh = cw <= ch ? (int)((double)S * ch / cw) : S;
        const PreTableKey* k = pre_tables(plan, cache, ch, cw, nh, nw, (nh - S) / 2, (nw - S) / 2, S, S);   // centre crop
        if (!k) return false;
        pre_finish_image(plan, im, *k);
        im.out_off = (long long)i * 3 * S * S;
    }
    return true;
}

// qwen_vl_utils / Qwen2VLImageProcessor smart_resize (image_processing_qwen2_vl.py:62-87): both sides multiples of `factor`, pixel
// count within [min_pixels, max_pixels]. Python's round() is round-half-even = nearbyint in the default rounding mode.
inline bool pre_smart_resize(int height, int width, int factor, long long min_pixels, long long max_pixels, int& h_bar, int& w_bar) {
    const int mx = height > width ? height : width, mn = height > width ? width : height;
    if ((double)mx / mn > 200.0) return false;
    h_bar = (int)std::nearbyint((double)height / factor) * factor;
    w_bar = (int)std::nearbyint((double)width / factor) * factor;
    if ((long long)h_bar * w_bar > max_pixels) {
        const double beta = std::sqrt(((double)height * width) / (double)max_pixels);
        h_bar = (int)std::floor((double)height / beta / factor) * factor;
        w_bar = (int)std::floor((double)width / beta / factor) * factor;
        if (h_bar < factor) h_bar = factor;
        if (w_bar < factor) w_bar = factor;
    } else if ((long long)h_bar * w_bar < min_pixels) {
        const double beta = std::sqrt((double)min_pixels / ((double)height * width));
        h_bar = (int)std::ceil((double)height * beta / factor) * factor;
        w_bar = (int)std::ceil((double)width * beta / factor) * factor;
    }
    return true;
}

// Qwen still images: smart_resize, plain bicubic resize of the whole image (no canvas, no crop), patch-row output; image i's rows
// start at sum_{j<i} gh_j * gw_j. grid_hw[i] = (gh, gw) in patches.
inline bool pre_plan_qwen(const int32_t* heights, const int32_t* widths, const int64_t* offsets, int n, int patch, int merge, int temporal,
                          long long min_pixels, long long max_pixels, PrePlan& plan, int32_t* grid_hw, long long* total_rows) {
    std::vector<PreTableKey> cache;
    cache.reserve(n);
    plan.images.resize(n);
    long long rows = 0;
    const long long row_elems = 3LL * temporal * patch * patch;
    for (int i = 0; i < n; ++i) {
        const int h = heights[i], w = widths[i];
        if (h <= 0 || w <= 0) { plan.error = "image with non-positive size"; return false; }
        int rh, rw;
        if (!pre_smart_resize(h, w, patch * merge, min_pixels, max_pixels, rh, rw)) {
            plan.error = "absolute aspect ratio must be smaller than 200";
            return false;
        }
        PreImage& im = plan.images[i];
        im.src_off = offsets[i]; im.h = h; im.w = w;
        im.canvas_h = h; im.canvas_w = w; im.paste_x = im.paste_y = 0;
        const PreTableKey* k = pre_tables(plan, cache, h, w, rh, rw, 0, 0, rh, rw);
        if (!k) return false;
        pre_finish_image(plan, im, *k);
        im.out_off = rows * row_elems;
        im.t_lo = 0; im.t_hi = temporal;
        if (grid_hw) { grid_hw[2 * i] = rh / patch; grid_hw[2 * i + 1] = rw / patch; }
        rows += (long long)(rh / patch) * (rw / patch);
    }
    if (total_rows) *total_rows = rows;
    return true;
}

// Qwen videos: video v is frames[v] uint8 HWC frames of heights[v] x widths[v], stored back to back from offsets[v]. smart_resize with
// the video's own pixel bounds, resample policy policy[v] (PRE_PIL: frames given as images, each resized by PIL; PRE_TORCHVISION:
// decoded files, resized by torchvision), then consecutive frames form one temporal patch: frame f goes to temporal slot f % temporal
// of grid step f / temporal. A count that is not a multiple of `temporal` is completed by repeating the last frame, which is done by
// writing that frame to all the remaining slots of its step. One PreImage per frame; video v's rows start at sum_{u<v} t_u gh_u gw_u.
// grid_thw[v] = (t, gh, gw).
inline bool pre_plan_qwen_video(const int32_t* heights, const int32_t* widths, const int32_t* frames, const int32_t* policy,
                                const int64_t* offsets, int n, int patch, int merge, int temporal, const int64_t* min_pixels,
                                const int64_t* max_pixels, PrePlan& plan, int32_t* grid_thw, long long* total_rows) {
    std::vector<PreTableKey> cache;
    cache.reserve(n);
    long long rows = 0, entries = 0;
    const long long row_elems = 3LL * temporal * patch * patch;
    for (int v = 0; v < n; ++v) entries += frames[v] > 0 ? frames[v] : 0;
    if (entries > 65535) { plan.error = "too many frames in one call (at most 65535)"; return false; }
    plan.images.reserve((size_t)entries);
    for (int v = 0; v < n; ++v) {
        const int h = heights[v], w = widths[v], nf = frames[v];
        if (h <= 0 || w <= 0 || nf <= 0) { plan.error = "video with non-positive size or no frames"; return false; }
        if (policy[v] != PRE_PIL && policy[v] != PRE_TORCHVISION) { plan.error = "unknown resample policy"; return false; }
        if (min_pixels[v] <= 0 || max_pixels[v] < min_pixels[v]) { plan.error = "bad pixel bounds"; return false; }
        int rh, rw;
        if (!pre_smart_resize(h, w, patch * merge, min_pixels[v], max_pixels[v], rh, rw)) {
            plan.error = "absolute aspect ratio must be smaller than 200";
            return false;
        }
        const PreTableKey* k = pre_tables(plan, cache, h, w, rh, rw, 0, 0, rh, rw, policy[v]);
        if (!k) return false;
        const int gh = rh / patch, gw = rw / patch, gt = (nf + temporal - 1) / temporal;
        for (int f = 0; f < nf; ++f) {
            PreImage im{};
            im.src_off = offsets[v] + (long long)f * h * w * 3; im.h = h; im.w = w;
            im.canvas_h = h; im.canvas_w = w;
            pre_finish_image(plan, im, *k);
            im.out_off = (rows + (long long)(f / temporal) * gh * gw) * row_elems;
            im.t_lo = f % temporal;
            im.t_hi = f == nf - 1 ? temporal : im.t_lo + 1;
            plan.images.push_back(im);
        }
        if (grid_thw) { grid_thw[3 * v] = gt; grid_thw[3 * v + 1] = gh; grid_thw[3 * v + 2] = gw; }
        rows += (long long)gt * gh * gw;
    }
    if (total_rows) *total_rows = rows;
    return true;
}

}  // namespace vqa
