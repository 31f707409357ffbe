// nlmeans.cu -- NLMeans denoise for sm_100a behind the C-ABI of include/hbcu.h.
//
// Replaces (reference /root/reference/libhb):
//   nlmeans_alloc / nlmeans_border      templates/nlmeans_template.c:20-101   -> pad_mirror_kernel
//   build_integral_scalar / _sse2       templates/nlmeans_template.c:545-591, nlmeans_x86.c:20-149
//   nlmeans_plane                       templates/nlmeans_template.c:593-717  -> nlmeans_v3_kernel, nlmeans_v3w_kernel,
//                                                                               nlmeans_tiled_kernel, nlmeans_generic_kernel
//   taskset fork/join per frame         nlmeans.c:546-597                      -> stream/event ordering
//
// Numeric contract (SURVEY.md appendix B): patch distances are exact integers
// (the reference's u32 integral image gives the exact n x n sum of squared
// differences); weights come from the host-computed 128-entry table; the fp32
// accumulation runs in the reference's displacement order with separate
// multiply and add (no FMA); the origin term is added in double; the result is
// truncated and a zero result falls back to the source pixel.  The output is
// therefore bit-identical to the reference C code.
//
// Kernel shape.  The reference materialises a whole-plane integral image per
// displacement (33 MB at 4K) and streams it through DRAM 17 times.  Here a CTA
// owns a 128 x TH tile: TMA brings the current and the compare tile (with an
// 8 pixel halo, mirror border already real data) into shared memory once; each
// thread marches down a 4-pixel-wide column strip keeping, per displacement,
// the vertical running sum of horizontal patch-row sums in registers (the
// n-row history lives in registers too), three horizontal displacements per
// pass.  HBM traffic is the algorithmic minimum: every input tile is read once
// per output tile.  pick_kernel() chooses per plane:
//   nlmeans_v3_kernel       8-bit planes (nlmeans_v3.cuh): packed-byte patch
//                           distances, weight/pixel accumulators in tensor
//                           memory, all planes of a frame in one launch; a
//                           variant takes the distances from prefiltered planes
//   nlmeans_v3w_kernel      9/10-bit planes, fp32-exact patch distances
//   nlmeans_tiled_kernel    integer arithmetic, accumulators in shared memory:
//                           16-bit samples above 10 bit, ranges the v3 kernels
//                           are not built for (range 1)
//   nlmeans_generic_kernel  one thread per pixel: patch/range beyond the tile
//                           halo, prefilters the v3 variant does not take
#include "hbcu_common.h"
#include "hbcu_frames.h"
#include "../../include/hbcu.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>
#include <cstdio>

namespace {

using hbcu::set_error;

constexpr int kBorder    = 16;    // ((n+2)/2+15)/16*16 for every preset (nlmeans.c:529)
constexpr int kMaxFrames = 32;    // NLMEANS_FRAMES_MAX
constexpr int kMaxDevices = 64;   // peer-access flags per ordered device pair (power of two)
constexpr int kTileW     = 128;
constexpr int kHalo      = 8;     // vertical halo of the shared-memory tiles (>= n/2 + r/2)
// Horizontal halo.  Measured on B200 (tools/tma_test.cu): cp.async.bulk.tensor raises
// "illegal instruction" unless the box's first byte in global memory is 16-byte aligned,
// so the tile starts at bordered column X0 (a multiple of 128), i.e. the halo is the
// whole 16-pixel mirror border.
constexpr int kHaloX     = kBorder;
constexpr int kTilePW    = kTileW + 2 * kHaloX;  // 160 elements per tile row
constexpr int kThreads   = 256;
constexpr int kGroup     = 3;     // horizontal displacements handled per pass

// trace points per frame (HBCU_NLMEANS_TRACE)
enum { TR_H2D_BEGIN, TR_H2D_END, TR_PAD_BEGIN, TR_PAD_END, TR_KERNEL_BEGIN, TR_KERNEL_END, TR_D2H_BEGIN, TR_D2H_END, kTracePoints };
constexpr int kTraceFrames = 512;

constexpr int kMaxTiledFrames = 8; // temporal depth the tiled kernel takes (tensor maps travel as kernel parameters)

// largest sample value the fp32-exact 16-bit kernel (nlmeans_v3w_kernel) accepts (10-bit video), and the bits above it
// in a packed pair
constexpr unsigned kMax10Bit       = 1023u;
constexpr unsigned kAbove10BitBits = 0xFC00FC00u;

struct KernelParams
{
    const void *planes[kMaxFrames];   // bordered plane base pointers, frame f = current + f
    const void *pre[kMaxFrames];      // prefiltered planes the patch distances are taken from (== planes[] without prefilter)
    const void *src_pre;              // source-patch image: pre[0], or planes[0] where the reference's pointer is stale
    int   use_pre;                    // prefiltered planes in use: only the generic kernel reads them
    int   nf;
    int   w, h;                       // plane size
    int   bpitch;                     // bordered plane pitch in elements
    void *dst;
    int   dpitch;                     // output pitch in elements
    int   n_half, r_half;
    float wfact;
    int   diff_max;
    double origin_tune;
    const float *exptable;            // 128 floats in global memory
};

// ---------------------------------------------------------------------------
// pad_mirror_kernel: unbordered plane -> bordered plane with the reference's
// mirror (img[-1-x] = img[x], img[w+x] = img[w-1-x], then rows mirrored the
// same way; templates/nlmeans_template.c:20-43).
// ---------------------------------------------------------------------------
template <typename PIX>
__global__ void pad_mirror_kernel(const PIX *__restrict__ src, int spitch, int w, int h,
                                  PIX *__restrict__ dst, int bpitch, int border, unsigned *range_flag)
{
    const int bx = blockIdx.x * blockDim.x + threadIdx.x;
    const int by = blockIdx.y * blockDim.y + threadIdx.y;
    const int bw = w + 2 * border, bh = h + 2 * border;
    if (bx >= bw || by >= bh) return;
    int x = bx - border, y = by - border;
    if (x < 0) x = -1 - x; else if (x >= w) x = 2 * w - 1 - x;
    if (y < 0) y = -1 - y; else if (y >= h) y = 2 * h - 1 - y;
    x = min(max(x, 0), w - 1);   // only reachable when w < border; the reference reads out of bounds there
    y = min(max(y, 0), h - 1);
    const PIX v = src[(size_t)y * spitch + x];
    dst[(size_t)by * bpitch + bx] = v;
    if (sizeof(PIX) == 2 && range_flag != nullptr && (unsigned)v > kMax10Bit) atomicOr(range_flag, 1u);
}

// 16 bytes per thread: interior chunks are straight uint4 copies, the chunks that touch the mirror border go element by element
template <typename PIX>
__global__ void __launch_bounds__(256) pad_mirror_vec_kernel(const PIX *__restrict__ src, int spitch, int w, int h,
                                                            PIX *__restrict__ dst, int bpitch, int border, unsigned *range_flag)
{
    constexpr int EPC = 16 / (int)sizeof(PIX);
    const int cx = blockIdx.x * blockDim.x + threadIdx.x;
    const int by = blockIdx.y * blockDim.y + threadIdx.y;
    const int bw = w + 2 * border, bh = h + 2 * border;
    const int bx0 = cx * EPC;
    if (bx0 >= bw || by >= bh) return;
    int y = by - border;
    if (y < 0) y = -1 - y; else if (y >= h) y = 2 * h - 1 - y;
    y = min(max(y, 0), h - 1);
    PIX *drow = dst + (size_t)by * bpitch;
    const PIX *srow = src + (size_t)y * spitch;
    if (bx0 >= border && bx0 + EPC <= border + w)
    {
        const uint4 v = *reinterpret_cast<const uint4 *>(srow + (bx0 - border));
        *reinterpret_cast<uint4 *>(drow + bx0) = v;
        // samples above kMax10Bit in a 16-bit plane: tell the 10-bit kernel to stand down (see nlmeans_v3w_kernel)
        if (sizeof(PIX) == 2 && range_flag != nullptr && ((v.x | v.y | v.z | v.w) & kAbove10BitBits) != 0u) atomicOr(range_flag, 1u);
        return;
    }
    bool bad = false;
#pragma unroll
    for (int i = 0; i < EPC; i++)
    {
        const int bx = bx0 + i;
        if (bx >= bw) break;
        int x = bx - border;
        if (x < 0) x = -1 - x; else if (x >= w) x = 2 * w - 1 - x;
        x = min(max(x, 0), w - 1);
        const PIX v = srow[x];
        drow[bx] = v;
        bad |= sizeof(PIX) == 2 && (unsigned)v > kMax10Bit;
    }
    if (bad && range_flag != nullptr) atomicOr(range_flag, 1u);
}

template <typename PIX>
__global__ void copy_plane_kernel(const PIX *__restrict__ src, int spitch, int w, int h,
                                  PIX *__restrict__ dst, int dpitch)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x < w && y < h) dst[(size_t)y * dpitch + x] = src[(size_t)y * spitch + x];
}

// ---------------------------------------------------------------------------
// nlmeans_prefilter (templates/nlmeans_template.c:103-543): the pre-denoised image the patch distances are taken
// from.  One thread per picture sample; src/pre point at sample (0,0) of the bordered planes (the mirror border is
// real data, 16 >= 2 samples wide).  The border of `pre` is rebuilt afterwards by pad_mirror_kernel.
//   mean   : pixel_2 sum times the double 1/size^2, truncated (:115-129)
//   median : the sorting networks of :135-198 return the true median
//   csm    : min / max of the neighbours -- but the reference leaves the row loop with `goto end` after its first sample
//            and at the origin (:253-266), so column -size/2 contributes one sample and the centre column only the
//            samples above the origin; reproduced
//   reduce : (wet * pre + dry * src) / (wet + dry) (:510-526)
// edgeboost (:325-426) decides in raster order (every cleared mask sample changes the counts after it): not here.
// ---------------------------------------------------------------------------
template <typename PIX>
__global__ void __launch_bounds__(256) prefilter_kernel(const PIX *__restrict__ src, PIX *__restrict__ pre, int bpitch, int w, int h, int filter_type)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const int kind = (filter_type & (16 | 32)) ? 2 : (filter_type & (4 | 8)) ? 1 : 0;
    const int size = kind == 2 ? ((filter_type & 32) ? 5 : 3) : kind == 1 ? ((filter_type & 8) ? 5 : 3) : ((filter_type & 2) ? 5 : 3);
    const int lo = -((size - 1) / 2), hi = (size + 1) / 2;
    const PIX *c = src + (ptrdiff_t)y * bpitch + x;
    const int cv = *c;
    int out = cv;
    if (kind == 0)
    {
        unsigned sum = 0;
        for (int k = lo; k < hi; k++)
            for (int j = lo; j < hi; j++) sum += c[(ptrdiff_t)j * bpitch + k];
        out = (int)__double2uint_rz(__dmul_rn((double)sum, 1.0 / (double)(size * size)));
    }
    else if (kind == 1)
    {
        int v[25], n = 0;
        for (int k = lo; k < hi; k++)
            for (int j = lo; j < hi; j++) v[n++] = c[(ptrdiff_t)j * bpitch + k];
        // rank selection: the median is the sample with exactly n/2 samples ordered before it (ties broken by position)
        const int half = n >> 1;
        for (int i = 0; i < n; i++)
        {
            int rank = 0;
            for (int q = 0; q < n; q++) rank += (v[q] < v[i]) || (v[q] == v[i] && q < i);
            if (rank == half) out = v[i];
        }
    }
    else
    {
        int mn = c[(ptrdiff_t)lo * bpitch + lo], mx = mn;
        for (int k = lo + 1; k < hi; k++)
            for (int j = lo; j < hi; j++)
            {
                if (k == 0 && j == 0) break;
                const int pv = c[(ptrdiff_t)j * bpitch + k];
                mn = min(mn, pv);
                mx = max(mx, pv);
            }
        const int median = (mn + mx) / 2;
        const int mn2 = (mn + median) / 2, mx2 = (mx + median) / 2;
        const int mn3 = (mn2 + median) / 2, mx3 = (mx2 + median) / 2;
        if (cv < mn) out = mn; else if (cv > mx) out = mx;
        else if (cv < mn2) out = mn2; else if (cv > mx2) out = mx2;
        else if (cv < mn3) out = mn3; else if (cv > mx3) out = mx3;
    }
    int wet = 1, dry = 0;
    if ((filter_type & 512) && (filter_type & 256)) { wet = 1; dry = 3; }
    else if (filter_type & 512) { wet = 1; dry = 1; }
    else if (filter_type & 256) { wet = 3; dry = 1; }
    if (dry > 0 && !(filter_type & 1024)) out = (wet * (int)(PIX)out + dry * cv) / (wet + dry);   // with edgeboost the blend runs after it
    pre[(ptrdiff_t)y * bpitch + x] = (PIX)out;
}

// ---------------------------------------------------------------------------
// edgeboost (template :325-426).  Pass 1 classifies every sample from two 3x3 gradient kernels (pixel_2 arithmetic,
// i.e. unsigned and wrapping, a double coefficient, constants that do not scale with the bit depth): 0 = no edge,
// 1 = weak (128), 2 = strong (235).  Pass 2 visits the samples IN RASTER ORDER and clears an edge sample whose 3x3
// neighbourhood holds fewer than 3 edge samples -- counting the already cleared neighbours as cleared -- and blends the
// source back into the surviving edge samples.  The raster-order rule is a recurrence c(p) = f(c(NW), c(N), c(NE), c(W))
// with a unique solution; any fixed point of the Jacobi iteration c' = f(c) IS that solution, so the kernel below is
// iterated until nothing changes (typically 2-3 rounds; a diagonal line of isolated pairs needs one round per sample).
// ---------------------------------------------------------------------------
template <typename PIX>
__global__ void __launch_bounds__(256) edgeboost_mask_kernel(const PIX *__restrict__ src, int bpitch, int w, int h, uint8_t *__restrict__ cls, int cpitch)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    typedef typename std::conditional<sizeof(PIX) == 1, uint16_t, uint32_t>::type PIX2;
    const int kern[3][3] = { { -31, 0, 31 }, { -44, 0, 44 }, { -31, 0, 31 } };
    const PIX *c = src + (ptrdiff_t)y * bpitch + x;
    PIX2 p1 = 0, p2 = 0;
    for (int k = -1; k < 2; k++)
        for (int j = -1; j < 2; j++)
        {
            const int sv = c[(ptrdiff_t)j * bpitch + k];
            p1 = (PIX2)(p1 + kern[j + 1][k + 1] * sv);
            p2 = (PIX2)(p2 + kern[k + 1][j + 1] * sv);
        }
    // `pixelN = pixelN > 0 ? pixelN : -pixelN` is the identity on an unsigned value
    const double coef = 1.0 / 126.42;
    p1 = (PIX2)__double2uint_rz(__dadd_rn(__dmul_rn((double)p1, coef), 128.0));
    p2 = (PIX2)__double2uint_rz(__dadd_rn(__dmul_rn((double)p2, coef), 128.0));
    const int m = (int)(PIX)(p1 + p2);
    cls[(size_t)(y + 1) * cpitch + x + 1] = m > 160 ? 2 : m > 16 ? 1 : 0;        // class plane has a 1-sample zero border
}

__global__ void __launch_bounds__(256) edgeboost_clear_kernel(const uint8_t *__restrict__ cls, int cpitch, int w, int h,
                                                             const uint8_t *__restrict__ clr_old, uint8_t *__restrict__ clr_new, int *__restrict__ changed)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const size_t i = (size_t)(y + 1) * cpitch + x + 1;
    uint8_t c = 0;
    if (cls[i])
    {
        // neighbours before p in raster order (NW, N, NE, W) count only if they were not cleared; the others as classified
        int n = 1;
        n += cls[i - cpitch - 1] && !clr_old[i - cpitch - 1];
        n += cls[i - cpitch] && !clr_old[i - cpitch];
        n += cls[i - cpitch + 1] && !clr_old[i - cpitch + 1];
        n += cls[i - 1] && !clr_old[i - 1];
        n += cls[i + 1] != 0;
        n += cls[i + cpitch - 1] != 0;
        n += cls[i + cpitch] != 0;
        n += cls[i + cpitch + 1] != 0;
        c = n < 3;
    }
    clr_new[i] = c;
    if (c != clr_old[i]) *changed = 1;
}

template <typename PIX>
__global__ void __launch_bounds__(256) edgeboost_apply_kernel(const PIX *__restrict__ src, PIX *__restrict__ pre, int bpitch, int w, int h,
                                                             const uint8_t *__restrict__ cls, const uint8_t *__restrict__ clr, int cpitch, int filter_type)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const size_t i = (size_t)(y + 1) * cpitch + x + 1;
    const ptrdiff_t o = (ptrdiff_t)y * bpitch + x;
    const int sv = src[o];
    int out = pre[o];
    if (cls[i] && !clr[i]) out = cls[i] == 2 ? (3 * sv + out) / 4 : (2 * sv + 3 * out) / 5;
    int wet = 1, dry = 0;                                   // the blend the filter kernel left for us (:510-526)
    if ((filter_type & 512) && (filter_type & 256)) { wet = 1; dry = 3; }
    else if (filter_type & 512) { wet = 1; dry = 1; }
    else if (filter_type & 256) { wet = 3; dry = 1; }
    if (dry > 0) out = (wet * (int)(PIX)out + dry * sv) / (wet + dry);
    pre[o] = (PIX)out;
}

// ---------------------------------------------------------------------------
// shared numeric pieces
// ---------------------------------------------------------------------------
__device__ __forceinline__ void add_origin(float &ws, float &ps, double ot, int src)
{
    // tmp.weight_sum += origin_tune; tmp.pixel_sum += origin_tune * src   (template :649-650)
    ws = (float)__dadd_rn((double)ws, ot);
    ps = (float)__dadd_rn((double)ps, __dmul_rn(ot, (double)src));
}

__device__ __forceinline__ void add_weighted(float &ws, float &ps, int diff, int diff_max, float wfact,
                                             const float *lut, int lut_stride, int lut_off, int pix)
{
    // if (diff < diff_max) { idx = diff * wfact; w = exptable[idx]; ...}   (template :685-694)
    if (diff < diff_max)
    {
        const int idx = __float2int_rz(__fmul_rn(__int2float_rn(diff), wfact));
        const float wgt = lut[idx * lut_stride + lut_off];
        ws = __fadd_rn(ws, wgt);
        ps = __fadd_rn(ps, __fmul_rn(wgt, __int2float_rn(pix)));
    }
}

template <typename PIX>
__device__ __forceinline__ PIX finish_pixel(float ws, float ps, PIX src)
{
    // result = (pixel)(pixel_sum / weight_sum); dst = result ? result : src   (template :706-713)
    const int v = __float2int_rz(__fdiv_rn(ps, ws));
    const PIX r = (PIX)v;
    return r ? r : src;
}

// ---------------------------------------------------------------------------
// Generic kernel: one thread per output pixel, reads the bordered planes
// through L1/L2.  Any patch size / range; used when the tiled kernel's halo
// (n/2 + r/2 <= 8) does not fit, and as an independent on-device cross check.
// ---------------------------------------------------------------------------
template <typename PIX>
__global__ void nlmeans_generic_kernel(KernelParams p)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= p.w || y >= p.h) return;
    const int bp = p.bpitch;
    const size_t org = (size_t)kBorder * bp + kBorder;
    const PIX *src = (const PIX *)p.planes[0] + org;
    const PIX *src_pre = (const PIX *)p.src_pre + org;
    float ws = 0.f, ps = 0.f;
    for (int f = 0; f < p.nf; f++)
    {
        const PIX *cmp = (const PIX *)p.planes[f] + org;
        const PIX *cmp_pre = (const PIX *)p.pre[f] + org;
        for (int dy = -p.r_half; dy <= p.r_half; dy++)
        {
            for (int dx = -p.r_half; dx <= p.r_half; dx++)
            {
                if (f == 0 && dx == 0 && dy == 0)
                {
                    add_origin(ws, ps, p.origin_tune, (int)src[(size_t)y * bp + x]);
                    continue;
                }
                unsigned ssd = 0;
                for (int j = -p.n_half; j <= p.n_half; j++)
                {
                    const PIX *a = src_pre + (ptrdiff_t)(y + j) * bp + x;
                    const PIX *b = cmp_pre + (ptrdiff_t)(y + j + dy) * bp + x + dx;
                    for (int k = -p.n_half; k <= p.n_half; k++)
                    {
                        const int d = (int)a[k] - (int)b[k];
                        ssd += (unsigned)(d * d);
                    }
                }
                add_weighted(ws, ps, (int)ssd, p.diff_max, p.wfact, p.exptable, 1, 0,
                             (int)cmp[(ptrdiff_t)(y + dy) * bp + x + dx]);
            }
        }
    }
    ((PIX *)p.dst)[(size_t)y * p.dpitch + x] = finish_pixel<PIX>(ws, ps, src[(size_t)y * bp + x]);
}

// ---------------------------------------------------------------------------
// TMA / mbarrier helpers (sm_90+ PTX)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int x, int y, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------------------
// Tiled kernel.  CTA = 256 threads = 8 warps; tile = 128 x TH output pixels;
// warp w owns rows [w*TH/8, (w+1)*TH/8), lane l owns columns [4l, 4l+4).
// ---------------------------------------------------------------------------
template <typename PIX, int TH>
struct TileLayout
{
    static constexpr int kRows      = TH + 2 * kHalo;
    static constexpr int kTileBytes = kRows * kTilePW * (int)sizeof(PIX);
    static constexpr int kAccBytes  = TH * kTileW * (int)sizeof(float);
    static constexpr int kLutBytes  = HBCU_NLMEANS_EXPSIZE * 32 * (int)sizeof(float);
    static constexpr int kOffCur    = 0;
    static constexpr int kOffCmp    = kOffCur + kTileBytes;
    static constexpr int kOffWs     = kOffCmp + kTileBytes;
    static constexpr int kOffPs     = kOffWs + kAccBytes;
    static constexpr int kOffLut    = kOffPs + kAccBytes;
    static constexpr int kOffBar    = kOffLut + kLutBytes;
    static constexpr int kTotal     = kOffBar + 64;
    static_assert(kTileBytes % 128 == 0, "TMA destination must stay 128-byte aligned");
};

template <typename PIX, int NH, int TH>
__device__ __forceinline__ void nlm_group(const PIX *__restrict__ cur, const PIX *__restrict__ cmp,
                                          float *__restrict__ acc_ws, float *__restrict__ acc_ps,
                                          const float *__restrict__ lut, const KernelParams &p,
                                          int seg_y0, int x, int lane, int dy, int dx0, int ng, int origin_g)
{
    constexpr int N  = 2 * NH + 1;
    constexpr int RS = TH / 8;
    constexpr int NA = 4 + 2 * NH;            // source values a thread needs per row
    constexpr int NB = NA + kGroup - 1;       // compare values per row (all displacements of the group)

    unsigned V[kGroup][4];
    unsigned hist[N][kGroup][4];
#pragma unroll
    for (int g = 0; g < kGroup; g++)
#pragma unroll
        for (int i = 0; i < 4; i++)
        {
            V[g][i] = 0;
#pragma unroll
            for (int k = 0; k < N; k++) hist[k][g][i] = 0;
        }

#pragma unroll 1
    for (int base = -NH; base < RS + NH; base += N)
    {
#pragma unroll
        for (int k = 0; k < N; k++)
        {
            const int yy = base + k;            // row being added, relative to the segment
            if (yy < RS + NH)
            {
                const int ty = seg_y0 + yy + kHalo;
                const PIX *arow = cur + ty * kTilePW + (x + kHaloX - NH);
                const PIX *brow = cmp + (ty + dy) * kTilePW + (x + kHaloX - NH + dx0);
                int a[NA], b[NB];
#pragma unroll
                for (int j = 0; j < NA; j++) a[j] = (int)arow[j];
#pragma unroll
                for (int j = 0; j < NB; j++) b[j] = (int)brow[j];
#pragma unroll
                for (int g = 0; g < kGroup; g++)
                {
                    if (g < ng)
                    {
                        unsigned c[NA + 1];
                        c[0] = 0;
#pragma unroll
                        for (int j = 0; j < NA; j++)
                        {
                            const int d = a[j] - b[j + g];
                            c[j + 1] = c[j] + (unsigned)(d * d);
                        }
#pragma unroll
                        for (int i = 0; i < 4; i++)
                        {
                            const unsigned hsum = c[i + N] - c[i];
                            V[g][i] += hsum - hist[k][g][i];
                            hist[k][g][i] = hsum;
                        }
                    }
                }
                if (yy >= NH)
                {
                    const int oy = seg_y0 + yy - NH;                 // finished output row (tile relative)
                    float4 ws4 = *reinterpret_cast<float4 *>(acc_ws + oy * kTileW + x);
                    float4 ps4 = *reinterpret_cast<float4 *>(acc_ps + oy * kTileW + x);
                    float ws[4] = { ws4.x, ws4.y, ws4.z, ws4.w };
                    float ps[4] = { ps4.x, ps4.y, ps4.z, ps4.w };
                    const PIX *prow = cmp + (oy + kHalo + dy) * kTilePW + (x + kHaloX + dx0);
#pragma unroll
                    for (int g = 0; g < kGroup; g++)
                    {
                        if (g < ng)
                        {
                            if (g == origin_g)
                            {
#pragma unroll
                                for (int i = 0; i < 4; i++)
                                    add_origin(ws[i], ps[i], p.origin_tune, (int)cur[(oy + kHalo) * kTilePW + x + kHaloX + i]);
                            }
                            else
                            {
#pragma unroll
                                for (int i = 0; i < 4; i++)
                                    add_weighted(ws[i], ps[i], (int)V[g][i], p.diff_max, p.wfact, lut, 32, lane, (int)prow[g + i]);
                            }
                        }
                    }
                    *reinterpret_cast<float4 *>(acc_ws + oy * kTileW + x) = make_float4(ws[0], ws[1], ws[2], ws[3]);
                    *reinterpret_cast<float4 *>(acc_ps + oy * kTileW + x) = make_float4(ps[0], ps[1], ps[2], ps[3]);
                }
            }
        }
    }
}

struct TiledParams
{
    KernelParams k;
    CUtensorMap  maps[kMaxTiledFrames];   // one TMA descriptor per frame of the temporal window
    const unsigned *only_if_flag;         // when set: run only if *only_if_flag != 0 (stand-in for nlmeans_v3w_kernel)
};

// The v3 kernels take up to three planes in ONE launch (tiles of Y, U and V in one grid):
// three separate launches end in three partial waves (510 + 135 + 135 CTAs on 148 SMs = 6 rounds),
// one launch of all tiles needs 5.
struct FusedParams
{
    int nplanes;
    int first_tile[4];                    // first linear tile index of each plane, [nplanes] = total
    int tiles_x[3];
    KernelParams k[3];
    CUtensorMap  maps[3][kMaxTiledFrames];
    CUtensorMap  maps_pre[3][kMaxTiledFrames];   // the pre-denoised planes (prefilter variant of the v3 kernel only)
    const unsigned *range_flag;           // nlmeans_v3w_kernel: non-zero = some sample exceeded kMax10Bit, do nothing
};

template <typename PIX, int NH, int TH>
__global__ void __launch_bounds__(kThreads, 1) nlmeans_tiled_kernel(const __grid_constant__ TiledParams tp)
{
    const KernelParams &p = tp.k;
    if (tp.only_if_flag != nullptr && *tp.only_if_flag == 0u) return;
    using L = TileLayout<PIX, TH>;
    extern __shared__ __align__(128) uint8_t smem[];
    PIX *cur      = reinterpret_cast<PIX *>(smem + L::kOffCur);
    PIX *cmp      = reinterpret_cast<PIX *>(smem + L::kOffCmp);
    float *acc_ws = reinterpret_cast<float *>(smem + L::kOffWs);
    float *acc_ps = reinterpret_cast<float *>(smem + L::kOffPs);
    float *lut    = reinterpret_cast<float *>(smem + L::kOffLut);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + L::kOffBar);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int X0 = blockIdx.x * kTileW, Y0 = blockIdx.y * TH;
    // tile element (0,0) is bordered-plane element (X0 + border - haloX, Y0 + border - halo)
    const int gx = X0 + kBorder - kHaloX, gy = Y0 + kBorder - kHalo;

    if (tid == 0)
    {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint32_t phase = 0;
    if (tid == 0)
    {
        mbar_expect_tx(bar, L::kTileBytes);
        tma_load_2d(cur, &tp.maps[0], gx, gy, bar);
    }
    // while the tile is in flight: replicate the weight table per bank, clear the accumulators
    for (int i = tid; i < HBCU_NLMEANS_EXPSIZE * 32; i += kThreads) lut[i] = p.exptable[i >> 5];
    for (int i = tid; i < TH * kTileW; i += kThreads)
    {
        acc_ws[i] = 0.f;
        acc_ps[i] = 0.f;
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    __syncthreads();

    const int seg_y0 = warp * (TH / 8);
    const int x = lane * 4;
    for (int f = 0; f < p.nf; f++)
    {
        const PIX *B = cur;
        if (f > 0)
        {
            __syncthreads();            // every warp is done with the previous compare tile
            if (tid == 0)
            {
                fence_proxy_async();
                mbar_expect_tx(bar, L::kTileBytes);
                tma_load_2d(cmp, &tp.maps[f], gx, gy, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1;
            B = cmp;
        }
        for (int dy = -p.r_half; dy <= p.r_half; dy++)
        {
            for (int dx0 = -p.r_half; dx0 <= p.r_half; dx0 += kGroup)
            {
                const int ng = min(kGroup, p.r_half - dx0 + 1);
                const int origin_g = (f == 0 && dy == 0 && dx0 <= 0 && dx0 + ng > 0) ? -dx0 : -1;
                nlm_group<PIX, NH, TH>(cur, B, acc_ws, acc_ps, lut, p, seg_y0, x, lane, dy, dx0, ng, origin_g);
            }
        }
    }

    // each warp finishes the rows it owns
    PIX *dst = reinterpret_cast<PIX *>(p.dst);
    for (int r = 0; r < TH / 8; r++)
    {
        const int oy = seg_y0 + r;
        const int y = Y0 + oy;
        if (y >= p.h) break;
        const float4 ws4 = *reinterpret_cast<const float4 *>(acc_ws + oy * kTileW + x);
        const float4 ps4 = *reinterpret_cast<const float4 *>(acc_ps + oy * kTileW + x);
        const float ws[4] = { ws4.x, ws4.y, ws4.z, ws4.w };
        const float ps[4] = { ps4.x, ps4.y, ps4.z, ps4.w };
        PIX o[4];
#pragma unroll
        for (int i = 0; i < 4; i++)
            o[i] = finish_pixel<PIX>(ws[i], ps[i], cur[(oy + kHalo) * kTilePW + x + kHaloX + i]);
        PIX *drow = dst + (size_t)y * p.dpitch + X0 + x;
        if (X0 + x + 3 < p.w)
        {
            if (sizeof(PIX) == 1)
                *reinterpret_cast<uchar4 *>(drow) = make_uchar4(o[0], o[1], o[2], o[3]);
            else
                *reinterpret_cast<ushort4 *>(drow) = make_ushort4(o[0], o[1], o[2], o[3]);
        }
        else
        {
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (X0 + x + i < p.w) drow[i] = o[i];
        }
    }
}

// ---------------------------------------------------------------------------
// v3 kernels (nlmeans_v3.cuh).  Same tiling and the same arithmetic results as
// the kernel above, re-expressed for the B200 issue ports measured in
// profiles/r01_microbench_instruction_throughput.txt:
//   * FADD/FMUL/FFMA issue at 4 warp-instr/clk/SM, integer ALU ops (PRMT, LOP3,
//     IADD3, IMAD) at 2, F2I / I2F.U8 at 0.5, LDS at ~1.
//   * Pixels are fetched as 32-bit words (conflict-free LDS.32) and unpacked
//     with PRMT straight into the float 2^23+v (bits 0x4B0000vv): differences
//     of two such floats are exact.
//   * idx = (int)(diff*wfact) and the test diff < diff_max collapse into
//     FMUL.SAT by wfact/128 (power-of-two scaling is exact), FADD.RZ with 2^16
//     (the mantissa then holds floor(128*t)), and a 129-entry table whose
//     entries 127 and 128 are 0.  Valid while wfact < 0.99 (then diff >=
//     diff_max implies idx >= 127); pick_kernel() checks it.  No F2I.
// ---------------------------------------------------------------------------
constexpr int kLutEntries = HBCU_NLMEANS_EXPSIZE + 1;

// byte k (0..3) of word w as the float 2^23 + value
__device__ __forceinline__ float byte_as_biased_float(uint32_t w, int k)
{
    return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7650 + k));
}

// half k (0/1) of word w as the float 2^23 + value
__device__ __forceinline__ float half_as_biased_float(uint32_t w, int k)
{
    return __uint_as_float(__byte_perm(w, 0x4B000000u, k ? 0x7432 : 0x7410));
}

#include "nlmeans_v3.cuh"
// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
struct PlaneGeom
{
    int w, h;            // plane size
    int bw, bh;          // bordered size
    int bpitch;          // bordered pitch, elements
    size_t bbytes;       // bordered plane bytes
    int rpitch;          // raw staging / output pitch, elements
    size_t rbytes;
};

}  // namespace

struct hbcu_nlmeans_s
{
    hbcu_nlmeans_config_t cfg;
    int bps;
    int impl;
    PlaneGeom g[3];
    int ring, out_slots;
    std::vector<uint8_t *> ring_mem;      // [slot*3+plane] bordered planes
    std::vector<uint8_t *> pre_mem;       // [slot*3+plane] prefiltered bordered planes (planes whose prefilter mode has a filter bit)
    bool has_pre[3];
    uint8_t *eb_cls, *eb_clr[2];          // edgeboost: class plane and the two cleared-flag planes (luma size + 1-sample border)
    int *eb_changed, *eb_changed_host;    // device flag + pinned copy of the Jacobi iteration
    int eb_cpitch;
    std::vector<uint8_t *> raw_base;      // [slot] one allocation per staged frame: a frame whose planes lie back to back on
    std::vector<uint8_t *> out_base;      // [oslot] the host (hb_frame_buffer_init, fifo.c:839-881) moves as ONE copy each way
    size_t frame_cap, plane_off[3];       // capacity of such an allocation; default plane offsets inside it
    std::vector<uint8_t *> raw_mem;       // [slot*3+plane] unbordered staging (H2D target), default layout
    std::vector<uint8_t *> out_mem;       // [oslot*3+plane]
    std::vector<int64_t>   ring_index;    // frame index held by each slot
    std::vector<CUtensorMap> maps;        // [slot*3+plane] TMA descriptors of the bordered planes
    std::vector<CUtensorMap> maps3;       // same planes, box height of the v3 8-bit kernel's tile
    std::vector<CUtensorMap> maps3_pre;   // the prefiltered planes (pre_mem), same box
    float *d_exptable;                    // 3 x 128
    unsigned *d_range_flag;               // sticky: a 16-bit plane held a sample above kMax10Bit (see nlmeans_v3w_kernel)
    cudaStream_t s_h2d, s_pad, s_compute, s_d2h;   // s_compute = s_comp[frame index & 1] of the launch being queued
    cudaStream_t s_comp[2];               // consecutive frames alternate between two compute streams: the next frame's CTAs
                                          // fill the SMs the previous launch's last partial wave leaves idle
    cudaEvent_t ev_join[2];
    std::vector<cudaEvent_t> ev_h2d;      // per ring slot: raw planes have arrived (H2D done), border kernels may start
    std::vector<cudaEvent_t> ev_upload;   // per ring slot: bordered planes ready
    std::vector<cudaEvent_t> ev_readers;  // [slot*2 + compute stream]: last kernel on that stream reading the slot is done
    std::vector<cudaEvent_t> ev_kernel;   // per out slot
    std::vector<cudaEvent_t> ev_d2h;      // per out slot
    std::vector<int64_t>     out_index;
    // multi-device dealing (hbcu_nlmeans_upload_peer): a frame this handle took from a peer handle's ring / gave to one
    std::vector<cudaEvent_t> ev_peer_in;  // per ring slot, this device: the peer copy INTO the slot is done
    std::vector<cudaEvent_t> peer_wait;   // per ring slot: a peer's ev_peer_in still reading this slot (nullptr: none); the next
                                          // upload into the slot orders itself behind it
    bool mid_stream;                      // the handle's index 0 is not the stream's first frame (hbcu_nlmeans_set_stream_slice)
    cudaEvent_t ev_mark[2];
    std::vector<cudaEvent_t> ev_pool;     // event pairs around the main kernels (kernel-only timing)
    int pool_used;                        // pairs recorded since mark 0
    // HBCU_NLMEANS_TRACE=<file>: per-frame timeline of the four streams (timing events, written at destroy);
    // the tracing hook that stands in for libhb's per-filter hb_log timing (work.c:2552-2560)
    std::string trace_path;
    std::vector<cudaEvent_t> tr;          // [frame * kTracePoints + point]
    cudaEvent_t tr_base;
    int tr_frames;
    int kernel_launches;                  // main-kernel launches since mark 0
};

namespace {

// Tile heights of the tiled kernel: 128 x 144 for 8-bit planes, 128 x 96 for 16-bit planes (8 warps; the tensor maps
// `maps` are encoded for this box).
constexpr int kTH8 = 144;
constexpr int kTH16 = 96;

// v3 shapes (warps x rows per warp), measured on B200 (profiles/r02b_v3_shape_sweep.txt): 12 x 18 beat 12 x 21, 8 x 28 and
// 12 x 12 with shared-memory accumulators.  Patch 9 takes 8 warps x 27 rows: its 9-row history does not fit 168 registers.
// Both tiles are 216 rows high, so one tensor map box (`maps3`, `maps3_pre`) serves every v3 kernel.
using V3L   = V3Layout<12, 18, 2>;          // 8-bit, two compare buffers
using V3L9  = V3Layout<8, 27, 2>;           // 8-bit, patch 9
using V3LP  = V3Layout<12, 18, 1, 1, true>; // 8-bit, prefiltered planes: one compare buffer pair
using V3LW  = V3Layout<12, 18, 1, 2>;       // 16-bit: one compare buffer (two 74 KB tiles)
constexpr int kV3BoxRows = V3L::kBoxRows;
static_assert(V3L9::kBoxRows == kV3BoxRows && V3LP::kBoxRows == kV3BoxRows && V3LW::kBoxRows == kV3BoxRows &&
              V3L9::kTH == V3L::kTH, "every v3 kernel loads the same TMA box");

enum class Kern { GENERIC, TILED, V3, V3W, V3_PRE };

// One kernel instantiation: entry point, block size, dynamic shared memory, tile height.
struct Inst { const void *fn; int threads, smem, th; };

// The instantiation kernel `k` runs for a plane of `bps` bytes per sample and patch half-width nh; fn == nullptr where
// there is none.
Inst instance(Kern k, int bps, int nh)
{
    if (k == Kern::V3 && bps == 1)
        switch (nh)
        {
            case 1: return { (const void *)nlmeans_v3_kernel<1, 12, 18, 2>, 12 * 32, V3L::kTotal, V3L::kTH };
            case 2: return { (const void *)nlmeans_v3_kernel<2, 12, 18, 2>, 12 * 32, V3L::kTotal, V3L::kTH };
            case 3: return { (const void *)nlmeans_v3_kernel<3, 12, 18, 2>, 12 * 32, V3L::kTotal, V3L::kTH };
            case 4: return { (const void *)nlmeans_v3_kernel<4, 8, 27, 2>, 8 * 32, V3L9::kTotal, V3L9::kTH };
        }
    if (k == Kern::V3_PRE && bps == 1)
        switch (nh)
        {
            case 1: return { (const void *)nlmeans_v3_kernel<1, 12, 18, 1, true>, 12 * 32, V3LP::kTotal, V3LP::kTH };
            case 2: return { (const void *)nlmeans_v3_kernel<2, 12, 18, 1, true>, 12 * 32, V3LP::kTotal, V3LP::kTH };
            case 3: return { (const void *)nlmeans_v3_kernel<3, 12, 18, 1, true>, 12 * 32, V3LP::kTotal, V3LP::kTH };
        }
    if (k == Kern::V3W && bps == 2)
        switch (nh)
        {
            case 1: return { (const void *)nlmeans_v3w_kernel<1, 12, 18, 1>, 12 * 32, V3LW::kTotal, V3LW::kTH };
            case 2: return { (const void *)nlmeans_v3w_kernel<2, 12, 18, 1>, 12 * 32, V3LW::kTotal, V3LW::kTH };
            case 3: return { (const void *)nlmeans_v3w_kernel<3, 12, 18, 1>, 12 * 32, V3LW::kTotal, V3LW::kTH };
        }
    using T8 = TileLayout<uint8_t, kTH8>;
    using T16 = TileLayout<uint16_t, kTH16>;
    if (k == Kern::TILED && bps == 1)
        switch (nh)
        {
            case 1: return { (const void *)nlmeans_tiled_kernel<uint8_t, 1, kTH8>, kThreads, T8::kTotal, kTH8 };
            case 2: return { (const void *)nlmeans_tiled_kernel<uint8_t, 2, kTH8>, kThreads, T8::kTotal, kTH8 };
            case 3: return { (const void *)nlmeans_tiled_kernel<uint8_t, 3, kTH8>, kThreads, T8::kTotal, kTH8 };
            case 4: return { (const void *)nlmeans_tiled_kernel<uint8_t, 4, kTH8>, kThreads, T8::kTotal, kTH8 };
        }
    if (k == Kern::TILED && bps == 2)
        switch (nh)
        {
            case 1: return { (const void *)nlmeans_tiled_kernel<uint16_t, 1, kTH16>, kThreads, T16::kTotal, kTH16 };
            case 2: return { (const void *)nlmeans_tiled_kernel<uint16_t, 2, kTH16>, kThreads, T16::kTotal, kTH16 };
            case 3: return { (const void *)nlmeans_tiled_kernel<uint16_t, 3, kTH16>, kThreads, T16::kTotal, kTH16 };
            case 4: return { (const void *)nlmeans_tiled_kernel<uint16_t, 4, kTH16>, kThreads, T16::kTotal, kTH16 };
        }
    return { nullptr, 0, 0, 0 };
}

bool tiled_supported(const KernelParams &kp)
{
    return !kp.use_pre && kp.n_half >= 1 && kp.n_half <= 4 && kp.n_half + kp.r_half <= kHalo && kp.nf <= kMaxTiledFrames;
}

// every displacement row of the plane's range decomposes into group shapes the v3 kernels were built with (all ranges
// 3 .. 15; range 1 does not)
bool v3_groups_known(const KernelParams &kp)
{
    for (int dx0 = -kp.r_half; dx0 <= kp.r_half; dx0 += kGroup)
    {
        const int ng = std::min(kGroup, kp.r_half - dx0 + 1), ob = (12 + dx0) & 3;
        if (!v3_group_known(ng, ob, kOrgNone)) return false;
        if (dx0 <= 0 && dx0 + ng > 0 && !v3_group_known(ng, ob, -dx0)) return false;
    }
    return true;
}

// The kernel a plane runs (hbcu_nlmeans_set_impl): impl 1 the generic kernel, impl 3 the integer tiled kernel where it
// fits; impl 0 and 2 a v3 kernel where its conditions hold, else the tiled kernel, else the generic one (which impl 2
// refuses, in run_filter).
Kern pick_kernel(const hbcu_nlmeans_s *h, const KernelParams &kp)
{
    const bool tiled = tiled_supported(kp);
    if (h->impl == 1) return Kern::GENERIC;
    if (h->impl == 3) return tiled ? Kern::TILED : Kern::GENERIC;
    const bool v3 = kp.wfact < 0.99f && kp.wfact > 1e-5f && v3_groups_known(kp);    // the table trick, the group shapes
    if (v3 && kp.use_pre && h->bps == 1 && kp.n_half >= 1 && kp.n_half <= 3 && kp.n_half + kp.r_half <= kHalo &&
        kp.nf <= kMaxTiledFrames)
        return Kern::V3_PRE;
    if (v3 && tiled && h->bps == 1) return Kern::V3;
    if (v3 && tiled && h->bps == 2 && h->cfg.depth <= 10 && kp.n_half <= 3) return Kern::V3W;
    return tiled ? Kern::TILED : Kern::GENERIC;
}

// The integer tiled kernel on one plane.  only_if_flag: run only if *only_if_flag != 0 (the stand-in behind a v3w launch).
int launch_tiled(hbcu_nlmeans_s *h, const KernelParams &kp, const int *slots, int plane, const unsigned *only_if_flag)
{
    TiledParams tp;
    tp.k = kp;
    tp.only_if_flag = only_if_flag;
    for (int f = 0; f < kp.nf; f++) tp.maps[f] = h->maps[slots[f] * 3 + plane];
    const Inst in = instance(Kern::TILED, h->bps, kp.n_half);
    void *args[] = { &tp };
    HBCU_CHECK(cudaLaunchKernel(in.fn, dim3((kp.w + kTileW - 1) / kTileW, (kp.h + in.th - 1) / in.th), dim3(in.threads), args,
                                (size_t)in.smem, h->s_compute));
    hbcu::count_launch();
    return 0;
}

// Runs kernel k on the planes pl[0 .. n).  The v3 kernels take all of them in one launch (they share n_half); the tiled
// and generic kernels are called with one plane.
int launch_planes(hbcu_nlmeans_s *h, Kern k, const KernelParams *kps, const int (*slots)[kMaxFrames], const int *pl, int n)
{
    if (k == Kern::GENERIC)
    {
        const KernelParams &kp = kps[pl[0]];
        dim3 blk(32, 8), grid((kp.w + 31) / 32, (kp.h + 7) / 8);
        if (h->bps == 1) nlmeans_generic_kernel<uint8_t><<<grid, blk, 0, h->s_compute>>>(kp);
        else             nlmeans_generic_kernel<uint16_t><<<grid, blk, 0, h->s_compute>>>(kp);
        hbcu::count_launch();
        HBCU_CHECK(cudaGetLastError());
        return 0;
    }
    if (k == Kern::TILED) return launch_tiled(h, kps[pl[0]], slots[pl[0]], pl[0], nullptr);

    // one linear grid over the tiles of every plane: separate launches would end in one partial wave each
    // (510 + 135 + 135 CTAs of a 4K frame on 148 SMs)
    FusedParams fp;
    fp.nplanes = n;
    fp.range_flag = h->d_range_flag;
    const Inst in = instance(k, h->bps, kps[pl[0]].n_half);
    int total = 0;
    for (int i = 0; i < n; i++)
    {
        const KernelParams &kp = kps[pl[i]];
        fp.k[i] = kp;
        for (int f = 0; f < kp.nf; f++)
        {
            fp.maps[i][f] = h->maps3[slots[pl[i]][f] * 3 + pl[i]];
            if (k == Kern::V3_PRE) fp.maps_pre[i][f] = h->maps3_pre[slots[pl[i]][f] * 3 + pl[i]];
        }
        fp.first_tile[i] = total;
        fp.tiles_x[i] = (kp.w + kTileW - 1) / kTileW;
        total += fp.tiles_x[i] * ((kp.h + in.th - 1) / in.th);
    }
    fp.first_tile[n] = total;
    void *args[] = { &fp };
    HBCU_CHECK(cudaLaunchKernel(in.fn, dim3(total), dim3(in.threads), args, (size_t)in.smem, h->s_compute));
    hbcu::count_launch();
    // v3w computes nothing for a frame with samples above 10 bit (the border kernel raised the range flag); the integer
    // kernel behind it then does the frame, and returns at once otherwise
    if (k == Kern::V3W)
        for (int i = 0; i < n; i++)
            if (launch_tiled(h, kps[pl[i]], slots[pl[i]], pl[i], h->d_range_flag) != 0) return -1;
    return 0;
}

inline void trace(hbcu_nlmeans_s *h, int64_t index, int point, cudaStream_t st)
{
    if (h->tr.empty() || index < 0 || index >= kTraceFrames) return;
    cudaEventRecord(h->tr[(size_t)index * kTracePoints + point], st);
    if (index + 1 > h->tr_frames) h->tr_frames = (int)index + 1;
}

int pad_plane(hbcu_nlmeans_s *h, int slot, int pl, const void *src, int spitch_elems, cudaStream_t st)
{
    const PlaneGeom &g = h->g[pl];
    uint8_t *dst = h->ring_mem[slot * 3 + pl];
    const bool aligned = ((uintptr_t)src % 16 == 0) && (((size_t)spitch_elems * h->bps) % 16 == 0);
    if (aligned)
    {
        const int chunks = (g.bw * h->bps + 15) / 16;
        dim3 blk(64, 4), grid((chunks + 63) / 64, (g.bh + 3) / 4);
        if (h->bps == 1)
            pad_mirror_vec_kernel<uint8_t><<<grid, blk, 0, st>>>((const uint8_t *)src, spitch_elems, g.w, g.h, dst, g.bpitch, kBorder, nullptr);
        else
            pad_mirror_vec_kernel<uint16_t><<<grid, blk, 0, st>>>((const uint16_t *)src, spitch_elems, g.w, g.h, (uint16_t *)dst, g.bpitch, kBorder, h->d_range_flag);
    }
    else
    {
        dim3 blk(64, 4), grid((g.bw + 63) / 64, (g.bh + 3) / 4);
        if (h->bps == 1)
            pad_mirror_kernel<uint8_t><<<grid, blk, 0, st>>>((const uint8_t *)src, spitch_elems, g.w, g.h, dst, g.bpitch, kBorder, nullptr);
        else
            pad_mirror_kernel<uint16_t><<<grid, blk, 0, st>>>((const uint16_t *)src, spitch_elems, g.w, g.h, (uint16_t *)dst, g.bpitch, kBorder, h->d_range_flag);
    }
    hbcu::count_launch();
    HBCU_CHECK(cudaGetLastError());
    return 0;
}

int run_filter(hbcu_nlmeans_s *h, int64_t index, int navail, int oslot, void *const *ext_dst = nullptr, const int *ext_strides = nullptr)
{
    if (navail < 1)
    {
        set_error("nlmeans: navail must be >= 1");
        return -1;
    }
    const int cs = (int)(index & 1);
    h->s_compute = h->s_comp[cs];
    int max_nf = 1;
    for (int pl = 0; pl < 3; pl++)
    {
        const int nf = h->cfg.plane[pl].bypass ? 1 : (navail < h->cfg.plane[pl].nframes ? navail : h->cfg.plane[pl].nframes);
        if (nf > max_nf) max_nf = nf;
    }
    for (int f = 0; f < max_nf; f++)
    {
        const int slot = (int)((index + f) % h->ring);
        if (h->ring_index[slot] != index + f)
        {
            set_error("nlmeans: frame %lld is not resident (slot %d holds %lld)", (long long)(index + f), slot,
                      (long long)h->ring_index[slot]);
            return -1;
        }
        HBCU_CHECK(cudaStreamWaitEvent(h->s_compute, h->ev_upload[slot], 0));
    }
    // the output slot must have been drained by its previous download
    HBCU_CHECK(cudaStreamWaitEvent(h->s_compute, h->ev_d2h[oslot], 0));

    const int pair = h->pool_used < (int)h->ev_pool.size() / 2 ? h->pool_used : -1;
    if (pair >= 0) HBCU_CHECK(cudaEventRecord(h->ev_pool[2 * pair], h->s_compute));
    trace(h, index, TR_KERNEL_BEGIN, h->s_compute);
    KernelParams kps[3];
    int slots[3][kMaxFrames];
    bool active[3] = { false, false, false };
    for (int pl = 0; pl < 3; pl++)
    {
        const hbcu_nlmeans_plane_t &pp = h->cfg.plane[pl];
        const PlaneGeom &g = h->g[pl];
        uint8_t *dst = ext_dst ? (uint8_t *)ext_dst[pl] : h->out_mem[oslot * 3 + pl];
        const int dpitch = ext_dst ? ext_strides[pl] / h->bps : g.rpitch;
        if (ext_dst && (((uintptr_t)dst % 8) || ((size_t)ext_strides[pl] % 8)))
        {
            set_error("nlmeans: external output plane %d must be 8-byte aligned (pointer and stride)", pl);
            return -1;
        }
        const int slot0 = (int)(index % h->ring);
        const bool passthru = (pp.prefilter & 2048) != 0;
        if (pp.bypass || passthru)
        {
            // nlmeans_deborder (template :45-67): plane passes through untouched -- or, with the passthru bit, the
            // prefiltered image IS the output and NLMeans does not run (nlmeans.c:485-491; tested before strength == 0)
            dim3 blk(64, 4), grid((g.w + 63) / 64, (g.h + 3) / 4);
            const uint8_t *plane0 = (passthru && h->has_pre[pl]) ? h->pre_mem[slot0 * 3 + pl] : h->ring_mem[slot0 * 3 + pl];
            const uint8_t *src = plane0 + ((size_t)kBorder * g.bpitch + kBorder) * h->bps;
            if (h->bps == 1) copy_plane_kernel<uint8_t><<<grid, blk, 0, h->s_compute>>>(src, g.bpitch, g.w, g.h, dst, dpitch);
            else copy_plane_kernel<uint16_t><<<grid, blk, 0, h->s_compute>>>((const uint16_t *)src, g.bpitch, g.w, g.h, (uint16_t *)dst, dpitch);
            hbcu::count_launch();
            HBCU_CHECK(cudaGetLastError());
            continue;
        }
        KernelParams &kp = kps[pl];
        memset(&kp, 0, sizeof(kp));
        kp.nf    = navail < pp.nframes ? navail : pp.nframes;
        for (int f = 0; f < kp.nf; f++)
        {
            const int slot = (int)((index + f) % h->ring);
            slots[pl][f] = slot;
            kp.planes[f] = h->ring_mem[slot * 3 + pl];
            kp.pre[f]    = h->has_pre[pl] ? h->pre_mem[slot * 3 + pl] : h->ring_mem[slot * 3 + pl];
        }
        kp.use_pre = h->has_pre[pl] ? 1 : 0;
        // nlmeans_plane reads frame[0].image_pre before it prefilters frame 0 (template :612 vs :628): a frame that was
        // never a compare frame of an earlier output contributes its UNFILTERED image as the source patch
        kp.src_pre = (h->has_pre[pl] && (index >= 1 || h->mid_stream) && pp.nframes >= 2) ? kp.pre[0] : kp.planes[0];
        kp.w = g.w;
        kp.h = g.h;
        kp.bpitch = g.bpitch;
        kp.dst = dst;
        kp.dpitch = dpitch;
        kp.n_half = (pp.patch_size - 1) / 2;
        kp.r_half = (pp.range - 1) / 2;
        kp.wfact = pp.weight_fact;
        kp.diff_max = pp.diff_max;
        kp.origin_tune = pp.origin_tune;
        kp.exptable = h->d_exptable + pl * HBCU_NLMEANS_EXPSIZE;
        active[pl] = true;
    }
    Kern kern[3];
    int act[3], nact = 0;
    for (int pl = 0; pl < 3; pl++)
    {
        if (!active[pl]) continue;
        kern[pl] = pick_kernel(h, kps[pl]);
        if (h->impl == 2 && kern[pl] == Kern::GENERIC)
        {
            set_error("nlmeans: tiled kernel does not support n=%d r=%d", 2 * kps[pl].n_half + 1, 2 * kps[pl].r_half + 1);
            return -1;
        }
        act[nact++] = pl;
    }
    // one launch for all active planes when they picked the same v3 kernel and patch size, else one launch per plane
    bool fused = nact > 0 && (kern[act[0]] == Kern::V3 || kern[act[0]] == Kern::V3W);
    for (int i = 1; i < nact && fused; i++)
        fused = kern[act[i]] == kern[act[0]] && kps[act[i]].n_half == kps[act[0]].n_half;
    if (fused)
    {
        if (launch_planes(h, kern[act[0]], kps, slots, act, nact) != 0) return -1;
        h->kernel_launches++;
    }
    else
    {
        for (int i = 0; i < nact; i++)
        {
            if (launch_planes(h, kern[act[i]], kps, slots, &act[i], 1) != 0) return -1;
            h->kernel_launches++;
        }
    }
    if (pair >= 0)
    {
        HBCU_CHECK(cudaEventRecord(h->ev_pool[2 * pair + 1], h->s_compute));
        h->pool_used++;
    }
    trace(h, index, TR_KERNEL_END, h->s_compute);
    HBCU_CHECK(cudaEventRecord(h->ev_kernel[oslot], h->s_compute));
    // every slot this launch read may be overwritten once it is done (per compute stream: launches on the other
    // stream that read the same slot record their own event)
    for (int f = 0; f < max_nf; f++)
        HBCU_CHECK(cudaEventRecord(h->ev_readers[(int)((index + f) % h->ring) * 2 + cs], h->s_compute));
    h->out_index[oslot] = index;
    return 0;
}

}  // namespace

extern "C" {

int hbcu_nlmeans_create(hbcu_nlmeans_t **out, const hbcu_nlmeans_config_t *cfg)
{
    if (out == nullptr || cfg == nullptr)
    {
        set_error("nlmeans_create: null argument");
        return -1;
    }
    *out = nullptr;
    if (cfg->width < kBorder || cfg->height < kBorder || cfg->depth < 8 || cfg->depth > 16)
    {
        set_error("nlmeans_create: unsupported geometry %dx%d depth %d", cfg->width, cfg->height, cfg->depth);
        return -1;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev)
    {
        cudaGetLastError();
        set_error("nlmeans_create: CUDA device %d not available (%d devices); there is no CPU fallback", cfg->device, ndev);
        return -1;
    }
    HBCU_CHECK(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    HBCU_CHECK(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major < 10)
    {
        set_error("nlmeans_create: device %d is sm_%d%d; this library is built for sm_100a only", cfg->device, prop.major, prop.minor);
        return -1;
    }
    for (int pl = 0; pl < 3; pl++)
    {
        const hbcu_nlmeans_plane_t &pp = cfg->plane[pl];
        if (pp.bypass) continue;
        if (pp.patch_size < 1 || !(pp.patch_size & 1) || pp.range < 1 || !(pp.range & 1) ||
            pp.nframes < 1 || pp.nframes > kMaxFrames)
        {
            set_error("nlmeans_create: plane %d has invalid patch/range/frames %d/%d/%d", pl, pp.patch_size, pp.range, pp.nframes);
            return -1;
        }
        if (pp.patch_size / 2 + pp.range / 2 > kBorder)
        {
            // the reference reads outside its 16-pixel border here (undefined behaviour); refuse instead
            set_error("nlmeans_create: patch/2 + range/2 = %d exceeds the %d pixel border", pp.patch_size / 2 + pp.range / 2, kBorder);
            return -1;
        }
    }

    hbcu_nlmeans_s *h = new (std::nothrow) hbcu_nlmeans_s();
    if (h == nullptr)
    {
        set_error("nlmeans_create: out of memory");
        return -1;
    }
    h->cfg = *cfg;
    h->bps = cfg->depth > 8 ? 2 : 1;
    h->impl = 0;
    if (const char *e = getenv("HBCU_NLMEANS_IMPL")) h->impl = atoi(e) >= 0 && atoi(e) <= 3 ? atoi(e) : 0;   // test hook
    h->ring = cfg->ring_frames > 0 ? cfg->ring_frames : 8;
    h->out_slots = cfg->out_slots > 0 ? cfg->out_slots : 4;
    h->d_exptable = nullptr;
    h->d_range_flag = nullptr;
    h->pool_used = 0;
    h->kernel_launches = 0;
    for (int pl = 0; pl < 3; pl++)
    {
        PlaneGeom &g = h->g[pl];
        g.w = pl == 0 ? cfg->width : -((-cfg->width) >> cfg->chroma_shift_w);
        g.h = pl == 0 ? cfg->height : -((-cfg->height) >> cfg->chroma_shift_h);
        g.bw = g.w + 2 * kBorder;
        g.bh = g.h + 2 * kBorder;
        g.bpitch = (g.bw + 127) / 128 * 128;
        g.bbytes = (size_t)g.bpitch * g.bh * h->bps;
        g.rpitch = (g.w + 127) / 128 * 128;
        g.rbytes = (size_t)g.rpitch * g.h * h->bps;
        h->plane_off[pl] = pl == 0 ? 0 : h->plane_off[pl - 1] + h->g[pl - 1].rbytes;
        h->frame_cap = h->plane_off[pl] + g.rbytes;
    }
#define CK(expr)                                                                                          \
    do {                                                                                                  \
        cudaError_t _e = (expr);                                                                          \
        if (_e != cudaSuccess) {                                                                          \
            set_error("%s failed: %s", #expr, cudaGetErrorString(_e));                                    \
            hbcu_nlmeans_destroy(h);                                                                      \
            return -1;                                                                                    \
        }                                                                                                 \
    } while (0)
    // The NLMeans kernel fills every SM (one CTA takes the whole register file); the small border kernels
    // of the upload stream must not queue behind a whole frame of it, or the upload -> kernel chain stalls:
    // give the upload stream the highest priority so its CTAs are placed as soon as any SM frees up.
    int prio_lo = 0, prio_hi = 0;
    CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    // function attributes live in the device's context: every kernel this handle can launch opts into its dynamic shared
    // memory here, per device (a handle on a second GPU would otherwise launch with the default 48 KB limit)
    for (Kern k : { Kern::TILED, Kern::V3, Kern::V3W, Kern::V3_PRE })
        for (int nh = 1; nh <= 4; nh++)
        {
            const Inst in = instance(k, h->bps, nh);
            if (in.fn != nullptr) CK(cudaFuncSetAttribute(in.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, in.smem));
        }
    CK(cudaStreamCreateWithPriority(&h->s_h2d, cudaStreamNonBlocking, prio_hi));
    CK(cudaStreamCreateWithPriority(&h->s_pad, cudaStreamNonBlocking, prio_hi));    // border kernels: off the copy stream, so the
                                                                                   // copy engine never waits for an SM to free up
    CK(cudaStreamCreateWithPriority(&h->s_comp[0], cudaStreamNonBlocking, prio_lo));
    CK(cudaStreamCreateWithPriority(&h->s_comp[1], cudaStreamNonBlocking, prio_lo));
    h->s_compute = h->s_comp[0];
    CK(cudaEventCreateWithFlags(&h->ev_join[0], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_join[1], cudaEventDisableTiming));
    CK(cudaStreamCreateWithPriority(&h->s_d2h, cudaStreamNonBlocking, prio_hi));
    h->ring_mem.assign(h->ring * 3, nullptr);
    h->pre_mem.assign(h->ring * 3, nullptr);
    for (int pl = 0; pl < 3; pl++) h->has_pre[pl] = (cfg->plane[pl].prefilter & 63) != 0;
    h->eb_cls = h->eb_clr[0] = h->eb_clr[1] = nullptr;
    h->eb_changed = h->eb_changed_host = nullptr;
    h->eb_cpitch = cfg->width + 2;
    bool any_eb = false;
    for (int pl = 0; pl < 3; pl++) any_eb = any_eb || (h->has_pre[pl] && (cfg->plane[pl].prefilter & 1024));
    if (any_eb)
    {
        const size_t n = (size_t)h->eb_cpitch * (cfg->height + 2);
        CK(cudaMalloc(&h->eb_cls, n));
        CK(cudaMalloc(&h->eb_clr[0], n));
        CK(cudaMalloc(&h->eb_clr[1], n));
        CK(cudaMalloc(&h->eb_changed, sizeof(int)));
        CK(cudaHostAlloc(&h->eb_changed_host, sizeof(int), cudaHostAllocPortable));
    }
    h->raw_mem.assign(h->ring * 3, nullptr);
    h->out_mem.assign(h->out_slots * 3, nullptr);
    h->raw_base.assign(h->ring, nullptr);
    h->out_base.assign(h->out_slots, nullptr);
    h->ring_index.assign(h->ring, -1);
    h->out_index.assign(h->out_slots, -1);
    h->ev_upload.assign(h->ring, nullptr);
    h->ev_h2d.assign(h->ring, nullptr);
    h->ev_readers.assign(h->ring * 2, nullptr);
    h->ev_peer_in.assign(h->ring, nullptr);
    h->peer_wait.assign(h->ring, nullptr);
    h->mid_stream = false;
    h->ev_kernel.assign(h->out_slots, nullptr);
    h->ev_d2h.assign(h->out_slots, nullptr);
    h->maps.resize(h->ring * 3);
    h->maps3.resize(h->ring * 3);
    h->maps3_pre.resize(h->ring * 3);
    for (int s = 0; s < h->ring; s++)
    {
        CK(cudaEventCreateWithFlags(&h->ev_upload[s], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_h2d[s], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_readers[2 * s], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_readers[2 * s + 1], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_peer_in[s], cudaEventDisableTiming));
        CK(cudaMalloc(&h->raw_base[s], h->frame_cap));
        for (int pl = 0; pl < 3; pl++)
        {
            // cleared once: the pitch padding right of the bordered picture is never written by the border kernels but
            // travels with the plane in the multi-device halo copy (initcheck would flag every such byte)
            CK(cudaMalloc(&h->ring_mem[s * 3 + pl], h->g[pl].bbytes));
            CK(cudaMemset(h->ring_mem[s * 3 + pl], 0, h->g[pl].bbytes));
            if (h->has_pre[pl])
            {
                CK(cudaMalloc(&h->pre_mem[s * 3 + pl], h->g[pl].bbytes));
                CK(cudaMemset(h->pre_mem[s * 3 + pl], 0, h->g[pl].bbytes));
            }
            h->raw_mem[s * 3 + pl] = h->raw_base[s] + h->plane_off[pl];
            const int th = h->bps == 1 ? kTH8 : kTH16;
            if (hbcu::encode_tensor_map_2d(&h->maps[s * 3 + pl], h->bps, h->ring_mem[s * 3 + pl], (uint64_t)h->g[pl].bw,
                                           (uint64_t)h->g[pl].bh, (uint64_t)h->g[pl].bpitch * h->bps, kTilePW,
                                           th + 2 * kHalo) != 0)
            {
                hbcu_nlmeans_destroy(h);
                return -1;
            }
            if (hbcu::encode_tensor_map_2d(&h->maps3[s * 3 + pl], h->bps, h->ring_mem[s * 3 + pl], (uint64_t)h->g[pl].bw,
                                           (uint64_t)h->g[pl].bh, (uint64_t)h->g[pl].bpitch * h->bps, kTilePW,
                                           kV3BoxRows) != 0)
            {
                hbcu_nlmeans_destroy(h);
                return -1;
            }
            if (h->has_pre[pl] &&
                hbcu::encode_tensor_map_2d(&h->maps3_pre[s * 3 + pl], h->bps, h->pre_mem[s * 3 + pl], (uint64_t)h->g[pl].bw,
                                           (uint64_t)h->g[pl].bh, (uint64_t)h->g[pl].bpitch * h->bps, kTilePW,
                                           kV3BoxRows) != 0)
            {
                hbcu_nlmeans_destroy(h);
                return -1;
            }
        }
    }
    for (int s = 0; s < h->out_slots; s++)
    {
        CK(cudaEventCreateWithFlags(&h->ev_kernel[s], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_d2h[s], cudaEventDisableTiming));
        CK(cudaMalloc(&h->out_base[s], h->frame_cap));
        CK(cudaMemset(h->out_base[s], 0, h->frame_cap));       // stride padding is never written by the kernels
        for (int pl = 0; pl < 3; pl++) h->out_mem[s * 3 + pl] = h->out_base[s] + h->plane_off[pl];
    }
    CK(cudaEventCreate(&h->ev_mark[0]));
    CK(cudaEventCreate(&h->ev_mark[1]));
    h->tr_frames = 0;
    h->tr_base = nullptr;
    if (const char *e = getenv("HBCU_NLMEANS_TRACE"))
    {
        h->trace_path = e;
        h->tr.assign((size_t)kTraceFrames * kTracePoints, nullptr);
        for (auto &ev : h->tr) CK(cudaEventCreate(&ev));
        CK(cudaEventCreate(&h->tr_base));
        CK(cudaEventRecord(h->tr_base, h->s_h2d));
    }
    h->ev_pool.assign(2 * 256, nullptr);
    for (auto &e : h->ev_pool) CK(cudaEventCreate(&e));
    CK(cudaMalloc(&h->d_exptable, 3 * HBCU_NLMEANS_EXPSIZE * sizeof(float)));
    CK(cudaMalloc(&h->d_range_flag, sizeof(unsigned)));
    CK(cudaMemset(h->d_range_flag, 0, sizeof(unsigned)));
    for (int pl = 0; pl < 3; pl++)
        CK(cudaMemcpy(h->d_exptable + pl * HBCU_NLMEANS_EXPSIZE, cfg->plane[pl].exptable,
                      HBCU_NLMEANS_EXPSIZE * sizeof(float), cudaMemcpyHostToDevice));
    // the clearing memsets above ran on the legacy default stream; the handle's non-blocking streams do not wait for it
    CK(cudaDeviceSynchronize());
#undef CK
    *out = h;
    return 0;
}

void hbcu_nlmeans_destroy(hbcu_nlmeans_t *h)
{
    if (h == nullptr) return;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    if (!h->tr.empty())
    {
        if (FILE *fp = fopen(h->trace_path.c_str(), "a"))
        {
            fprintf(fp, "# frame,h2d_begin,h2d_end,pad_begin,pad_end,kernel_begin,kernel_end,d2h_begin,d2h_end (ms since create; -1 = not recorded)\n");
            for (int f = 0; f < h->tr_frames; f++)
            {
                fprintf(fp, "%d", f);
                for (int k = 0; k < kTracePoints; k++)
                {
                    float ms = -1.f;
                    if (cudaEventElapsedTime(&ms, h->tr_base, h->tr[(size_t)f * kTracePoints + k]) != cudaSuccess) { ms = -1.f; cudaGetLastError(); }
                    fprintf(fp, ",%.4f", ms);
                }
                fprintf(fp, "\n");
            }
            fclose(fp);
        }
        for (auto ev : h->tr) if (ev) cudaEventDestroy(ev);
        if (h->tr_base) cudaEventDestroy(h->tr_base);
    }
    for (auto p : h->ring_mem) if (p) cudaFree(p);
    for (auto p : h->pre_mem) if (p) cudaFree(p);
    if (h->eb_cls) cudaFree(h->eb_cls);
    if (h->eb_clr[0]) cudaFree(h->eb_clr[0]);
    if (h->eb_clr[1]) cudaFree(h->eb_clr[1]);
    if (h->eb_changed) cudaFree(h->eb_changed);
    if (h->eb_changed_host) cudaFreeHost(h->eb_changed_host);
    for (auto p : h->raw_base) if (p) cudaFree(p);
    for (auto p : h->out_base) if (p) cudaFree(p);
    for (auto e : h->ev_upload) if (e) cudaEventDestroy(e);
    for (auto e : h->ev_readers) if (e) cudaEventDestroy(e);
    for (auto e : h->ev_peer_in) if (e) cudaEventDestroy(e);
    for (auto e : h->ev_kernel) if (e) cudaEventDestroy(e);
    for (auto e : h->ev_d2h) if (e) cudaEventDestroy(e);
    if (h->ev_mark[0]) cudaEventDestroy(h->ev_mark[0]);
    if (h->ev_mark[1]) cudaEventDestroy(h->ev_mark[1]);
    for (auto e : h->ev_pool) if (e) cudaEventDestroy(e);
    if (h->d_exptable) cudaFree(h->d_exptable);
    if (h->d_range_flag) cudaFree(h->d_range_flag);
    if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
    if (h->s_pad) cudaStreamDestroy(h->s_pad);
    for (auto e : h->ev_h2d) if (e) cudaEventDestroy(e);
    for (int i = 0; i < 2; i++)
    {
        if (h->s_comp[i]) cudaStreamDestroy(h->s_comp[i]);
        if (h->ev_join[i]) cudaEventDestroy(h->ev_join[i]);
    }
    if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
    delete h;
}

// Planes laid out back to back (plane p+1 starts where plane p's stride x height ends), the way hb_frame_buffer_init
// builds a STANDARD hb_buffer_t: such a frame crosses PCIe as one copy instead of three (measured with
// tools/copy_bench.cu, both directions busy: 0.278 vs 0.307 ms per 4K frame).
static bool frame_is_contiguous(const hbcu_nlmeans_t *h, const void *const planes[3], const int strides[3], size_t off[3], size_t *total)
{
    size_t o = 0;
    for (int pl = 0; pl < 3; pl++)
    {
        const PlaneGeom &g = h->g[pl];
        if ((const uint8_t *)planes[pl] != (const uint8_t *)planes[0] + o) return false;
        if (strides[pl] < g.w * h->bps || (strides[pl] % 16) != 0) return false;
        off[pl] = o;
        o += (size_t)strides[pl] * g.h;
    }
    *total = o;
    return o <= h->frame_cap;
}

static int upload_common(hbcu_nlmeans_t *h, int64_t index, const void *const planes[3], const int strides[3], bool from_device)
{
    if (h == nullptr || planes == nullptr || strides == nullptr || index < 0)
    {
        set_error("nlmeans_upload: bad argument");
        return -1;
    }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    const int slot = (int)(index % h->ring);
    // do not overwrite a slot a queued kernel still reads
    // raw staging of this slot is free once its previous border kernels ran; the bordered planes once their readers are done
    HBCU_CHECK(cudaStreamWaitEvent(h->s_h2d, h->ev_upload[slot], 0));
    HBCU_CHECK(cudaStreamWaitEvent(h->s_pad, h->ev_readers[2 * slot], 0));
    HBCU_CHECK(cudaStreamWaitEvent(h->s_pad, h->ev_readers[2 * slot + 1], 0));
    if (h->peer_wait[slot] != nullptr)
    {
        HBCU_CHECK(cudaStreamWaitEvent(h->s_pad, h->peer_wait[slot], 0));     // a peer device still copies the slot's planes
        h->peer_wait[slot] = nullptr;
    }
    size_t off[3] = { 0, 0, 0 }, total = 0;
    const bool whole = !from_device && frame_is_contiguous(h, planes, strides, off, &total);
    if (!from_device)
    {
        trace(h, index, TR_H2D_BEGIN, h->s_h2d);
        if (whole)
        {
            HBCU_CHECK(cudaMemcpyAsync(h->raw_base[slot], planes[0], total, cudaMemcpyHostToDevice, h->s_h2d));
        }
        else
        {
            for (int pl = 0; pl < 3; pl++)
            {
                const PlaneGeom &g = h->g[pl];
                HBCU_CHECK(cudaMemcpy2DAsync(h->raw_mem[slot * 3 + pl], (size_t)g.rpitch * h->bps, planes[pl], (size_t)strides[pl],
                                             (size_t)g.w * h->bps, (size_t)g.h, cudaMemcpyHostToDevice, h->s_h2d));
            }
        }
        trace(h, index, TR_H2D_END, h->s_h2d);
        HBCU_CHECK(cudaEventRecord(h->ev_h2d[slot], h->s_h2d));
        HBCU_CHECK(cudaStreamWaitEvent(h->s_pad, h->ev_h2d[slot], 0));
    }
    trace(h, index, TR_PAD_BEGIN, h->s_pad);
    for (int pl = 0; pl < 3; pl++)
    {
        const PlaneGeom &g = h->g[pl];
        if (from_device)
        {
            if (pad_plane(h, slot, pl, planes[pl], strides[pl] / h->bps, h->s_pad) != 0) return -1;
        }
        else if (whole)
        {
            if (pad_plane(h, slot, pl, h->raw_base[slot] + off[pl], strides[pl] / h->bps, h->s_pad) != 0) return -1;
        }
        else
        {
            if (pad_plane(h, slot, pl, h->raw_mem[slot * 3 + pl], g.rpitch, h->s_pad) != 0) return -1;
        }
    }
    for (int pl = 0; pl < 3; pl++)
    {
        if (!h->has_pre[pl]) continue;
        // nlmeans_prefilter (template :428-543): filtered copy of the picture, then its own mirror border
        const PlaneGeom &g = h->g[pl];
        const size_t org = ((size_t)kBorder * g.bpitch + kBorder) * h->bps;
        const uint8_t *srcb = h->ring_mem[slot * 3 + pl] + org;
        uint8_t *preb = h->pre_mem[slot * 3 + pl];
        dim3 blk(64, 4), grid((g.w + 63) / 64, (g.h + 3) / 4), bgrid((g.bw + 63) / 64, (g.bh + 3) / 4);
        const int ft = h->cfg.plane[pl].prefilter;
        if (h->bps == 1) prefilter_kernel<uint8_t><<<grid, blk, 0, h->s_pad>>>(srcb, preb + org, g.bpitch, g.w, g.h, ft);
        else             prefilter_kernel<uint16_t><<<grid, blk, 0, h->s_pad>>>((const uint16_t *)srcb, (uint16_t *)(preb + org), g.bpitch, g.w, g.h, ft);
        hbcu::count_launch();
        if (ft & 1024)
        {
            // edgeboost: classify, iterate the raster-order clearing rule to its fixed point (host reads a flag per
            // round: this rarely used mode makes the upload synchronous), blend
            const int cp = h->eb_cpitch;
            const size_t n = (size_t)cp * (g.h + 2);
            HBCU_CHECK(cudaMemsetAsync(h->eb_cls, 0, n, h->s_pad));
            HBCU_CHECK(cudaMemsetAsync(h->eb_clr[0], 0, n, h->s_pad));
            HBCU_CHECK(cudaMemsetAsync(h->eb_clr[1], 0, n, h->s_pad));
            if (h->bps == 1) edgeboost_mask_kernel<uint8_t><<<grid, blk, 0, h->s_pad>>>(srcb, g.bpitch, g.w, g.h, h->eb_cls, cp);
            else             edgeboost_mask_kernel<uint16_t><<<grid, blk, 0, h->s_pad>>>((const uint16_t *)srcb, g.bpitch, g.w, g.h, h->eb_cls, cp);
            hbcu::count_launch();
            // rounds are queued in batches and the host looks at the flag of a batch's LAST round only: once a round changes
            // nothing the state is the fixed point and every later round leaves it alone, so extra rounds are harmless and
            // the host waits once per batch instead of once per round (ADVICE r1)
            constexpr int kRoundsPerWait = 8;
            int cur = 0;
            for (int round = 0; round < g.w + g.h + 2; round += kRoundsPerWait)
            {
                for (int k = 0; k < kRoundsPerWait; k++)
                {
                    HBCU_CHECK(cudaMemsetAsync(h->eb_changed, 0, sizeof(int), h->s_pad));
                    edgeboost_clear_kernel<<<grid, blk, 0, h->s_pad>>>(h->eb_cls, cp, g.w, g.h, h->eb_clr[cur], h->eb_clr[cur ^ 1], h->eb_changed);
                    hbcu::count_launch();
                    cur ^= 1;
                }
                HBCU_CHECK(cudaMemcpyAsync(h->eb_changed_host, h->eb_changed, sizeof(int), cudaMemcpyDeviceToHost, h->s_pad));
                HBCU_CHECK(cudaStreamSynchronize(h->s_pad));
                if (*h->eb_changed_host == 0) break;
            }
            if (h->bps == 1) edgeboost_apply_kernel<uint8_t><<<grid, blk, 0, h->s_pad>>>(srcb, preb + org, g.bpitch, g.w, g.h, h->eb_cls, h->eb_clr[cur], cp, ft);
            else             edgeboost_apply_kernel<uint16_t><<<grid, blk, 0, h->s_pad>>>((const uint16_t *)srcb, (uint16_t *)(preb + org), g.bpitch, g.w, g.h, h->eb_cls, h->eb_clr[cur], cp, ft);
            hbcu::count_launch();
        }
        if (h->bps == 1) pad_mirror_kernel<uint8_t><<<bgrid, blk, 0, h->s_pad>>>(preb + org, g.bpitch, g.w, g.h, preb, g.bpitch, kBorder, nullptr);
        else             pad_mirror_kernel<uint16_t><<<bgrid, blk, 0, h->s_pad>>>((const uint16_t *)(preb + org), g.bpitch, g.w, g.h, (uint16_t *)preb, g.bpitch, kBorder, nullptr);
        hbcu::count_launch();
        HBCU_CHECK(cudaGetLastError());
    }
    trace(h, index, TR_PAD_END, h->s_pad);
    HBCU_CHECK(cudaEventRecord(h->ev_upload[slot], h->s_pad));
    h->ring_index[slot] = index;
    return 0;
}

int hbcu_nlmeans_upload(hbcu_nlmeans_t *h, int64_t index, const void *const planes[3], const int strides[3])
{
    return upload_common(h, index, planes, strides, false);
}

int hbcu_nlmeans_upload_device(hbcu_nlmeans_t *h, int64_t index, const void *const dplanes[3], const int strides[3])
{
    return upload_common(h, index, dplanes, strides, true);
}

int hbcu_nlmeans_set_stream_slice(hbcu_nlmeans_t *h, int mid_stream)
{
    if (h == nullptr) { set_error("nlmeans_set_stream_slice: bad argument"); return -1; }
    h->mid_stream = mid_stream != 0;
    return 0;
}

// Frame `src_index` of `src` (already uploaded there: bordered, prefiltered) becomes frame `dst_index` of `dst`, copied
// device to device (NVLink peer copy between two GPUs, a plain device copy when both handles share one).  This is the
// temporal halo of block-cyclic dealing: the first nframes-1 frames of a block are also the look-ahead window of the
// previous block, which lives on another device -- one H2D per frame, the halo travels GPU to GPU.
int hbcu_nlmeans_upload_peer(hbcu_nlmeans_t *dst, int64_t dst_index, hbcu_nlmeans_t *src, int64_t src_index)
{
    if (dst == nullptr || src == nullptr || dst == src || dst_index < 0 || src_index < 0)
    {
        set_error("nlmeans_upload_peer: bad argument");
        return -1;
    }
    if (dst->bps != src->bps || dst->cfg.width != src->cfg.width || dst->cfg.height != src->cfg.height)
    {
        set_error("nlmeans_upload_peer: the two handles differ in geometry");
        return -1;
    }
    for (int pl = 0; pl < 3; pl++)
        if (dst->g[pl].bbytes != src->g[pl].bbytes || dst->has_pre[pl] != src->has_pre[pl])
        {
            set_error("nlmeans_upload_peer: the two handles differ in plane %d (layout or prefilter)", pl);
            return -1;
        }
    const int dslot = (int)(dst_index % dst->ring), sslot = (int)(src_index % src->ring);
    if (src->ring_index[sslot] != src_index)
    {
        set_error("nlmeans_upload_peer: frame %lld is not resident on the source handle", (long long)src_index);
        return -1;
    }
    const int ddev = dst->cfg.device, sdev = src->cfg.device;
    HBCU_CHECK(cudaSetDevice(ddev));
    if (ddev != sdev)
    {
        // direct NVLink path, asked for once per ordered pair of devices; without peer access the copy is staged by the
        // driver (still correct)
        static bool asked[kMaxDevices][kMaxDevices] = {};
        bool &done = asked[ddev & (kMaxDevices - 1)][sdev & (kMaxDevices - 1)];
        if (!done)
        {
            if (cudaDeviceEnablePeerAccess(sdev, 0) != cudaSuccess) cudaGetLastError();   // already enabled, or not supported
            done = true;
        }
    }
    // the destination slot is free once the kernels reading its previous frame are done (and no peer reads it)
    HBCU_CHECK(cudaStreamWaitEvent(dst->s_pad, dst->ev_readers[2 * dslot], 0));
    HBCU_CHECK(cudaStreamWaitEvent(dst->s_pad, dst->ev_readers[2 * dslot + 1], 0));
    if (dst->peer_wait[dslot] != nullptr)
    {
        HBCU_CHECK(cudaStreamWaitEvent(dst->s_pad, dst->peer_wait[dslot], 0));
        dst->peer_wait[dslot] = nullptr;
    }
    HBCU_CHECK(cudaStreamWaitEvent(dst->s_pad, src->ev_upload[sslot], 0));          // source planes complete
    for (int pl = 0; pl < 3; pl++)
    {
        // two handles on ONE device (tests, or a deliberate 2-handle setup): an ordinary stream-ordered device copy --
        // cudaMemcpyPeerAsync(dev, dev) was seen to run ahead of the stream's event waits on one box (frames computed
        // from a halo that had not landed); between two devices it is the NVLink peer copy
        if (ddev == sdev)
        {
            HBCU_CHECK(cudaMemcpyAsync(dst->ring_mem[dslot * 3 + pl], src->ring_mem[sslot * 3 + pl], src->g[pl].bbytes, cudaMemcpyDeviceToDevice, dst->s_pad));
            if (dst->has_pre[pl])
                HBCU_CHECK(cudaMemcpyAsync(dst->pre_mem[dslot * 3 + pl], src->pre_mem[sslot * 3 + pl], src->g[pl].bbytes, cudaMemcpyDeviceToDevice, dst->s_pad));
        }
        else
        {
            HBCU_CHECK(cudaMemcpyPeerAsync(dst->ring_mem[dslot * 3 + pl], ddev, src->ring_mem[sslot * 3 + pl], sdev, src->g[pl].bbytes, dst->s_pad));
            if (dst->has_pre[pl])
                HBCU_CHECK(cudaMemcpyPeerAsync(dst->pre_mem[dslot * 3 + pl], ddev, src->pre_mem[sslot * 3 + pl], sdev, src->g[pl].bbytes, dst->s_pad));
        }
    }
    HBCU_CHECK(cudaEventRecord(dst->ev_upload[dslot], dst->s_pad));
    HBCU_CHECK(cudaEventRecord(dst->ev_peer_in[dslot], dst->s_pad));
    src->peer_wait[sslot] = dst->ev_peer_in[dslot];
    dst->ring_index[dslot] = dst_index;
    return 0;
}

int hbcu_nlmeans_wait_upload(hbcu_nlmeans_t *h, int64_t index)
{
    if (h == nullptr || index < 0) { set_error("nlmeans_wait_upload: bad argument"); return -1; }
    const int slot = (int)(index % h->ring);
    if (h->ring_index[slot] != index) { set_error("nlmeans_wait_upload: frame %lld not resident", (long long)index); return -1; }
    HBCU_CHECK(cudaEventSynchronize(h->ev_upload[slot]));
    return 0;
}

int hbcu_nlmeans_filter(hbcu_nlmeans_t *h, int64_t index, int navail, void *const planes[3], const int strides[3])
{
    if (h == nullptr || planes == nullptr || strides == nullptr || index < 0)
    {
        set_error("nlmeans_filter: bad argument");
        return -1;
    }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    const int oslot = (int)(index % h->out_slots);
    size_t off[3] = { 0, 0, 0 }, total = 0;
    const bool whole = frame_is_contiguous(h, planes, strides, off, &total);
    if (whole)
    {
        // the kernels write the output slot in the host buffer's own layout: one copy brings the frame back
        void *dst[3] = { h->out_base[oslot] + off[0], h->out_base[oslot] + off[1], h->out_base[oslot] + off[2] };
        if (run_filter(h, index, navail, oslot, dst, strides) != 0) return -1;
    }
    else if (run_filter(h, index, navail, oslot) != 0) return -1;
    HBCU_CHECK(cudaStreamWaitEvent(h->s_d2h, h->ev_kernel[oslot], 0));
    trace(h, index, TR_D2H_BEGIN, h->s_d2h);
    if (whole)
    {
        HBCU_CHECK(cudaMemcpyAsync(planes[0], h->out_base[oslot], total, cudaMemcpyDeviceToHost, h->s_d2h));
    }
    else
    {
        for (int pl = 0; pl < 3; pl++)
        {
            const PlaneGeom &g = h->g[pl];
            HBCU_CHECK(cudaMemcpy2DAsync(planes[pl], (size_t)strides[pl], h->out_mem[oslot * 3 + pl], (size_t)g.rpitch * h->bps,
                                         (size_t)g.w * h->bps, (size_t)g.h, cudaMemcpyDeviceToHost, h->s_d2h));
        }
    }
    trace(h, index, TR_D2H_END, h->s_d2h);
    HBCU_CHECK(cudaEventRecord(h->ev_d2h[oslot], h->s_d2h));
    return 0;
}

int hbcu_nlmeans_wait(hbcu_nlmeans_t *h, int64_t index)
{
    if (h == nullptr || index < 0) { set_error("nlmeans_wait: bad argument"); return -1; }
    const int oslot = (int)(index % h->out_slots);
    if (h->out_index[oslot] != index) { set_error("nlmeans_wait: frame %lld is not in flight", (long long)index); return -1; }
    HBCU_CHECK(cudaEventSynchronize(h->ev_d2h[oslot]));
    return 0;
}

int hbcu_nlmeans_poll(hbcu_nlmeans_t *h, int64_t index)
{
    if (h == nullptr || index < 0) { set_error("nlmeans_poll: bad argument"); return -1; }
    const int oslot = (int)(index % h->out_slots);
    if (h->out_index[oslot] != index) { set_error("nlmeans_poll: frame %lld is not in flight", (long long)index); return -1; }
    cudaError_t e = cudaEventQuery(h->ev_d2h[oslot]);
    if (e == cudaSuccess) return 1;
    if (e == cudaErrorNotReady) return 0;
    set_error("nlmeans_poll: %s", cudaGetErrorString(e));
    return -1;
}

int hbcu_nlmeans_filter_device(hbcu_nlmeans_t *h, int64_t index, int navail, void *out_planes[3], int out_strides[3])
{
    if (h == nullptr || index < 0) { set_error("nlmeans_filter_device: bad argument"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    const int oslot = (int)(index % h->out_slots);
    if (run_filter(h, index, navail, oslot) != 0) return -1;
    // no download: the slot is free again as soon as the kernel is done
    HBCU_CHECK(cudaEventRecord(h->ev_d2h[oslot], h->s_compute));
    for (int pl = 0; pl < 3; pl++)
    {
        if (out_planes) out_planes[pl] = h->out_mem[oslot * 3 + pl];
        if (out_strides) out_strides[pl] = h->g[pl].rpitch * h->bps;
    }
    return 0;
}

int hbcu_nlmeans_filter_into(hbcu_nlmeans_t *h, int64_t index, int navail, void *const dplanes[3], const int strides[3])
{
    if (h == nullptr || index < 0 || dplanes == nullptr || strides == nullptr) { set_error("nlmeans_filter_into: bad argument"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    const int oslot = (int)(index % h->out_slots);
    if (run_filter(h, index, navail, oslot, dplanes, strides) != 0) return -1;
    HBCU_CHECK(cudaEventRecord(h->ev_d2h[oslot], h->s_compute));
    return 0;
}

static bool frame_fits(const hbcu_nlmeans_t *h, const hbcu_frame_t *f)
{
    if (f == nullptr || f->device != h->cfg.device) return false;
    for (int pl = 0; pl < 3; pl++)
        if (f->row_bytes[pl] != h->g[pl].w * h->bps || f->rows[pl] != h->g[pl].h) return false;
    return true;
}

int hbcu_nlmeans_upload_frame(hbcu_nlmeans_t *h, int64_t index, hbcu_frame_t *in)
{
    if (h == nullptr || index < 0 || !frame_fits(h, in)) { set_error("nlmeans_upload_frame: bad argument or frame geometry"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    // the border kernels are the only readers: they run on s_pad
    if (hbcu::frame_begin_read(in, h->s_pad) != 0) return -1;
    const void *planes[3] = { in->plane[0], in->plane[1], in->plane[2] };
    if (upload_common(h, index, planes, in->stride, true) != 0) return -1;
    return hbcu::frame_end_read(in, h->s_pad);
}

int hbcu_nlmeans_filter_frame(hbcu_nlmeans_t *h, int64_t index, int navail, hbcu_frame_t *out)
{
    if (h == nullptr || index < 0 || !frame_fits(h, out)) { set_error("nlmeans_filter_frame: bad argument or frame geometry"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    const int oslot = (int)(index % h->out_slots);
    cudaStream_t st = h->s_comp[index & 1];          // the stream run_filter() will launch on
    if (hbcu::frame_begin_write(out, st) != 0) return -1;
    void *planes[3] = { out->plane[0], out->plane[1], out->plane[2] };
    if (run_filter(h, index, navail, oslot, planes, out->stride) != 0) return -1;
    HBCU_CHECK(cudaEventRecord(h->ev_d2h[oslot], h->s_compute));  // no download: the slot is free once the kernel is done
    return hbcu::frame_end_write(out, h->s_compute);
}

int hbcu_nlmeans_stream_wait(hbcu_nlmeans_t *h, void *cuda_stream)
{
    // makes a caller-owned stream (e.g. the one NCCL runs on) wait for everything queued on the compute stream
    if (h == nullptr) { set_error("nlmeans_stream_wait: null handle"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    for (int i = 0; i < 2; i++)
    {
        HBCU_CHECK(cudaEventRecord(h->ev_join[i], h->s_comp[i]));
        HBCU_CHECK(cudaStreamWaitEvent((cudaStream_t)cuda_stream, h->ev_join[i], 0));
    }
    return 0;
}

int hbcu_nlmeans_sync(hbcu_nlmeans_t *h)
{
    if (h == nullptr) { set_error("nlmeans_sync: null handle"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    HBCU_CHECK(cudaStreamSynchronize(h->s_h2d));
    HBCU_CHECK(cudaStreamSynchronize(h->s_pad));
    HBCU_CHECK(cudaStreamSynchronize(h->s_comp[0]));
    HBCU_CHECK(cudaStreamSynchronize(h->s_comp[1]));
    HBCU_CHECK(cudaStreamSynchronize(h->s_d2h));
    return 0;
}

int hbcu_nlmeans_set_impl(hbcu_nlmeans_t *h, int impl)
{
    if (h == nullptr || impl < 0 || impl > 3) { set_error("nlmeans_set_impl: bad argument"); return -1; }
    h->impl = impl;
    return 0;
}

int hbcu_nlmeans_mark(hbcu_nlmeans_t *h, int which)
{
    if (h == nullptr || which < 0 || which > 1) { set_error("nlmeans_mark: bad argument"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    if (which == 0)
    {
        h->pool_used = 0;
        h->kernel_launches = 0;
    }
    // the mark sits behind everything queued on both compute streams; work queued after it starts after it
    HBCU_CHECK(cudaEventRecord(h->ev_join[1], h->s_comp[1]));
    HBCU_CHECK(cudaStreamWaitEvent(h->s_comp[0], h->ev_join[1], 0));
    HBCU_CHECK(cudaEventRecord(h->ev_mark[which], h->s_comp[0]));
    HBCU_CHECK(cudaStreamWaitEvent(h->s_comp[1], h->ev_mark[which], 0));
    return 0;
}

int hbcu_nlmeans_elapsed_ms(hbcu_nlmeans_t *h, float *ms)
{
    if (h == nullptr || ms == nullptr) { set_error("nlmeans_elapsed_ms: bad argument"); return -1; }
    HBCU_CHECK(cudaEventSynchronize(h->ev_mark[1]));
    HBCU_CHECK(cudaEventElapsedTime(ms, h->ev_mark[0], h->ev_mark[1]));
    return 0;
}

int hbcu_nlmeans_kernel_ms(hbcu_nlmeans_t *h, float *ms, int *launches)
{
    if (h == nullptr) { set_error("nlmeans_kernel_ms: null handle"); return -1; }
    // sums the event pairs recorded around the main kernels since mark 0 (at most 256 filter calls)
    float total = 0.f;
    for (int i = 0; i < h->pool_used; i++)
    {
        float t = 0.f;
        HBCU_CHECK(cudaEventSynchronize(h->ev_pool[2 * i + 1]));
        HBCU_CHECK(cudaEventElapsedTime(&t, h->ev_pool[2 * i], h->ev_pool[2 * i + 1]));
        total += t;
    }
    if (ms) *ms = total;
    if (launches) *launches = h->pool_used;   // filter calls timed (3 plane launches each)
    return 0;
}

}  // extern "C"
