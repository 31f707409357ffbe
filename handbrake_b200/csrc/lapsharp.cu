// lapsharp.cu -- Laplacian sharpen for sm_100a behind the C-ABI of include/hbcu.h.
//
// Replaces DEF_LAPSHARP_FUNC (reference libhb/lapsharp.c:125-182) and the frame batching of
// mt_frame_filter.c:169-237: frames are independent, so each one is upload -> kernel -> download
// on the handle's streams with `slots` frames in flight.
//
// Numeric contract kept bit for bit: the convolution accumulates in int16 (8-bit) / int32 (16-bit),
// the sharpening term is evaluated in double exactly as written in the reference
// ((acc*coef - src)*strength, truncated toward zero), then clamped.  Border rule as in the
// reference, including its dependence on the stride: pixels with x < (stride-width)/2 + offset_max
// are copied, and the last columns read the stride region to the right of the picture.
#include "hbcu_common.h"
#include "hbcu_frames.h"
#include "../../include/hbcu.h"

#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

namespace {

using hbcu::set_error;

// the four convolution kernels (lapsharp.c:36-93) as compile-time tables: the kernel id is a template parameter, so every
// coefficient is an immediate and the zero taps (4 of 9 for lap, 12 of 25 for log) cost nothing
struct LapTaps { int v[25]; };
__host__ __device__ constexpr LapTaps lap_taps(int kid)
{
    return kid == 0 ? LapTaps{ { 0, -1, 0, -1, 5, -1, 0, -1, 0 } }                                                    // lap
         : kid == 1 ? LapTaps{ { -1, -4, -1, -4, 25, -4, -1, -4, -1 } }                                               // isolap
         : kid == 2 ? LapTaps{ { 0, 0, -1, 0, 0, 0, -1, -2, -1, 0, -1, -2, 21, -2, -1, 0, -1, -2, -1, 0, 0, 0, -1, 0, 0 } }       // log
                    : LapTaps{ { 0, -1, -1, -1, 0, -1, -3, -4, -3, -1, -1, -4, 55, -4, -1, -1, -3, -4, -3, -1, 0, -1, -1, -1, 0 } }; // isolog
}

struct LapPlane
{
    const void *src;
    void *dst;
    int width, height, spitch, dpitch, kid, vec;      // vec: rows can be read as aligned 32-bit words
    double coef, strength;
};
struct LapFrame
{
    LapPlane pl[3];
    int max_value;
};

template <typename PIX, typename ACC>
__device__ __forceinline__ int lap_finish(int acc, int s0, double coef, double strength, int max_value)
{
    // the sharpening term exactly as the reference writes it (lapsharp.c:160-176): ACC wrap, double arithmetic,
    // truncation toward zero, ACC wrap again, clamp
    ACC pixel = (ACC)acc;
    const double dp = (double)pixel, ds = (double)s0;
    const double t = __dmul_rn(__dsub_rn(__dmul_rn(dp, coef), ds), strength);
    pixel = (ACC)((int)(ACC)(int)t + s0);
    int v = pixel;
    v = v < 0 ? 0 : v;
    return v > max_value ? max_value : v;
}

// one thread = 4 adjacent pixels of one row.  Interior groups read each of their SIZE input rows as three (8-bit) or four
// (16-bit) aligned 32-bit words through the read-only path and pick the SIZE+3 samples out of them.
template <typename PIX, typename ACC, int KID, bool VEC>
__device__ __forceinline__ void lap_px4(const LapPlane &p, int max_value, int x0, int y)
{
    constexpr int SIZE = KID < 2 ? 3 : 5;
    constexpr int offset_min = -((SIZE - 1) / 2), offset_max = (SIZE + 1) / 2;
    constexpr LapTaps K = lap_taps(KID);
    const PIX *src = (const PIX *)p.src;
    const int width = p.width, height = p.height, spitch = p.spitch;
    const int stride_border = (spitch - width) / 2;
    const PIX *row = src + (size_t)y * spitch;
    int out[4];
    const bool row_copy = (y < offset_max) || (y > height - offset_max);
    // the whole group of 4 is interior when its first and last pixel are (the x conditions are monotone)
    const bool all_interior = !row_copy && !(x0 < stride_border + offset_max) && !(x0 + 3 > width + stride_border - offset_max) && (x0 + 3 < width);
    if (all_interior)
    {
        int acc[4] = { 0, 0, 0, 0 };
        int s0[4];
#pragma unroll
        for (int j = offset_min; j < offset_max; j++)
        {
            const PIX *r = src + (size_t)(y + j) * spitch + x0;
            int v[SIZE + 3];                                   // samples x0 + offset_min .. x0 + offset_max + 2
            if (VEC)
            {
                if (sizeof(PIX) == 1)
                {
                    const uint32_t *rw = reinterpret_cast<const uint32_t *>(r - 4);     // x0 is a multiple of 4 and >= 4 here
                    const uint32_t w0 = __ldg(rw), w1 = __ldg(rw + 1), w2 = __ldg(rw + 2);
#pragma unroll
                    for (int t = 0; t < SIZE + 3; t++)
                    {
                        const int b = offset_min + t + 4;
                        const uint32_t w = b < 4 ? w0 : b < 8 ? w1 : w2;
                        v[t] = (int)((w >> (8 * (b & 3))) & 0xffu);
                    }
                }
                else
                {
                    const uint32_t *rw = reinterpret_cast<const uint32_t *>(r - 2);
                    const uint32_t w0 = __ldg(rw), w1 = __ldg(rw + 1), w2 = __ldg(rw + 2), w3 = __ldg(rw + 3);
#pragma unroll
                    for (int t = 0; t < SIZE + 3; t++)
                    {
                        const int b = offset_min + t + 2;      // sample index among the eight loaded
                        const uint32_t w = b < 2 ? w0 : b < 4 ? w1 : b < 6 ? w2 : w3;
                        v[t] = (int)((b & 1) ? (w >> 16) : (w & 0xffffu));
                    }
                }
            }
            else
            {
#pragma unroll
                for (int t = 0; t < SIZE + 3; t++) v[t] = r[offset_min + t];
            }
            if (j == 0)
            {
#pragma unroll
                for (int i = 0; i < 4; i++) s0[i] = v[i - offset_min];
            }
#pragma unroll
            for (int k = 0; k < SIZE; k++)
            {
                const int c = K.v[(j - offset_min) * SIZE + k];
                if (c == 0) continue;
#pragma unroll
                for (int i = 0; i < 4; i++) acc[i] += c * v[i + k];
            }
        }
#pragma unroll
        for (int i = 0; i < 4; i++) out[i] = lap_finish<PIX, ACC>(acc[i], s0[i], p.coef, p.strength, max_value);
    }
    else
    {
#pragma unroll
        for (int i = 0; i < 4; i++)
        {
            const int x = x0 + i;
            if (x >= width) { out[i] = 0; continue; }
            const int s0 = row[x];
            if (row_copy || (x < stride_border + offset_max) || (x > width + stride_border - offset_max))
            {
                out[i] = s0;
                continue;
            }
            int acc = 0;
#pragma unroll
            for (int k = offset_min; k < offset_max; k++)
#pragma unroll
                for (int j = offset_min; j < offset_max; j++)
                {
                    const int c = K.v[(j - offset_min) * SIZE + k - offset_min];
                    if (c != 0) acc += c * (int)src[(size_t)(y + j) * spitch + (x + k)];
                }
            out[i] = lap_finish<PIX, ACC>(acc, s0, p.coef, p.strength, max_value);
        }
    }
    PIX *drow = (PIX *)p.dst + (size_t)y * p.dpitch;
    if (x0 + 3 < width)
    {
        if (sizeof(PIX) == 1) *reinterpret_cast<uchar4 *>(drow + x0) = make_uchar4(out[0], out[1], out[2], out[3]);
        else                  *reinterpret_cast<ushort4 *>(drow + x0) = make_ushort4(out[0], out[1], out[2], out[3]);
    }
    else
    {
        for (int i = 0; i < 4; i++)
            if (x0 + i < width) drow[x0 + i] = (PIX)out[i];
    }
}

__device__ __forceinline__ int dp4a_us(uint32_t a, int b, int c)        // 4 unsigned bytes . 4 signed bytes + c
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// taps k .. k+3 of kernel row j as four signed bytes (every coefficient of the four kernels fits: |c| <= 55)
template <int KID>
__host__ __device__ constexpr int lap_tap_word(int j, int k)
{
    constexpr int SIZE = KID < 2 ? 3 : 5;
    constexpr LapTaps K = lap_taps(KID);
    unsigned w = 0;
    for (int t = 0; t < 4; t++)
        if (k + t < SIZE) w |= (unsigned)(K.v[j * SIZE + k + t] & 0xff) << (8 * t);
    return (int)w;
}

// Round 2: one thread = 4 adjacent pixels of R consecutive rows.  A thread-tile that lies wholly inside the filtered
// region reads each of its R + SIZE - 1 input rows ONCE as aligned 32-bit words (round 1 read SIZE rows per output row)
// and, at 8 bit, feeds them to the byte dot product: the 4-byte window of an output pixel in one input row is a funnel
// shift of two loaded words and `dp4a` applies that kernel row's taps in one instruction (9 / 25 multiply-adds per pixel
// become 3 / 5+).  Accumulating in 32 bits and wrapping to ACC once equals the reference's wrap after every tap
// (lapsharp.c:150-158: modular arithmetic).  Every other tile goes row by row through lap_px4.
template <typename PIX, typename ACC, int KID, bool VEC, int R>
__device__ __forceinline__ void lap_tile(const LapPlane &p, int max_value, int x0, int y0)
{
    constexpr int SIZE = KID < 2 ? 3 : 5;
    constexpr int offset_min = -((SIZE - 1) / 2), offset_max = (SIZE + 1) / 2;
    constexpr int NR = R + SIZE - 1;
    constexpr LapTaps K = lap_taps(KID);
    const int width = p.width, height = p.height, spitch = p.spitch;
    const int stride_border = (spitch - width) / 2;
    const bool interior = VEC && y0 >= offset_max && y0 + R - 1 <= height - offset_max
                       && !(x0 < stride_border + offset_max) && !(x0 + 3 > width + stride_border - offset_max) && (x0 + 3 < width);
    if (!interior)
    {
#pragma unroll 1
        for (int r = 0; r < R; r++)
            if (y0 + r < height) lap_px4<PIX, ACC, KID, VEC>(p, max_value, x0, y0 + r);
        return;
    }
    const PIX *src = (const PIX *)p.src + (size_t)(y0 + offset_min) * spitch + x0;
    int acc[R][4];
#pragma unroll
    for (int r = 0; r < R; r++)
#pragma unroll
        for (int i = 0; i < 4; i++) acc[r][i] = 0;
    if (sizeof(PIX) == 1)
    {
        uint32_t centre[R];
#pragma unroll
        for (int q = 0; q < NR; q++)                           // input row y0 + offset_min + q
        {
            const uint32_t *rw = reinterpret_cast<const uint32_t *>(src + (size_t)q * spitch - 4);
            const uint32_t w0 = __ldg(rw), w1 = __ldg(rw + 1), w2 = __ldg(rw + 2);
            uint32_t win[4], fifth[4];
#pragma unroll
            for (int i = 0; i < 4; i++)
            {
                const int b = 4 + i + offset_min;              // byte index of the window's first sample in (w0, w1, w2)
                win[i] = b < 4 ? __funnelshift_r(w0, w1, 8 * b) : b == 4 ? w1 : __funnelshift_r(w1, w2, 8 * (b - 4));
                const int b5 = b + 4;                          // fifth sample of a 5-tap row
                fifth[i] = b5 < 8 ? (w1 >> (8 * (b5 - 4))) & 0xffu : (w2 >> (8 * (b5 - 8))) & 0xffu;
            }
#pragma unroll
            for (int r = 0; r < R; r++)
            {
                const int j = q - r;                           // kernel row this input row is for output row r
                if (j < 0 || j >= SIZE) continue;
                const int tw = j == 0 ? lap_tap_word<KID>(0, 0) : j == 1 ? lap_tap_word<KID>(1, 0) : j == 2 ? lap_tap_word<KID>(2, 0)
                             : j == 3 ? lap_tap_word<KID>(SIZE > 3 ? 3 : 0, 0) : lap_tap_word<KID>(SIZE > 4 ? 4 : 0, 0);
                const int c5 = SIZE == 5 ? K.v[j * SIZE + SIZE - 1] : 0;
#pragma unroll
                for (int i = 0; i < 4; i++)
                {
                    if (tw != 0) acc[r][i] = dp4a_us(win[i], tw, acc[r][i]);
                    if (c5 != 0) acc[r][i] += c5 * (int)fifth[i];
                }
                if (j == -offset_min) centre[r] = w1;
            }
        }
        uint8_t *drow = (uint8_t *)p.dst + (size_t)y0 * p.dpitch + x0;
#pragma unroll
        for (int r = 0; r < R; r++)
        {
            int o[4];
#pragma unroll
            for (int i = 0; i < 4; i++)
                o[i] = lap_finish<PIX, ACC>(acc[r][i], (int)((centre[r] >> (8 * i)) & 0xffu), p.coef, p.strength, max_value);
            *reinterpret_cast<uchar4 *>(drow + (size_t)r * p.dpitch) = make_uchar4(o[0], o[1], o[2], o[3]);
        }
    }
    else
    {
        uint32_t centre[R][2];
#pragma unroll
        for (int q = 0; q < NR; q++)
        {
            const uint32_t *rw = reinterpret_cast<const uint32_t *>(src + (size_t)q * spitch - 2);
            const uint32_t w0 = __ldg(rw), w1 = __ldg(rw + 1), w2 = __ldg(rw + 2), w3 = __ldg(rw + 3);
            int v[SIZE + 3];                                   // samples x0 + offset_min .. x0 + offset_max + 2
#pragma unroll
            for (int t = 0; t < SIZE + 3; t++)
            {
                const int b = offset_min + t + 2;
                const uint32_t w = b < 2 ? w0 : b < 4 ? w1 : b < 6 ? w2 : w3;
                v[t] = (int)((b & 1) ? (w >> 16) : (w & 0xffffu));
            }
#pragma unroll
            for (int r = 0; r < R; r++)
            {
                const int j = q - r;
                if (j < 0 || j >= SIZE) continue;
#pragma unroll
                for (int k = 0; k < SIZE; k++)
                {
                    const int c = K.v[j * SIZE + k];
                    if (c == 0) continue;
#pragma unroll
                    for (int i = 0; i < 4; i++) acc[r][i] += c * v[i + k];
                }
                if (j == -offset_min) { centre[r][0] = w1; centre[r][1] = w2; }
            }
        }
        uint16_t *drow = (uint16_t *)p.dst + (size_t)y0 * p.dpitch + x0;
#pragma unroll
        for (int r = 0; r < R; r++)
        {
            int o[4];
#pragma unroll
            for (int i = 0; i < 4; i++)
            {
                const uint32_t w = centre[r][i >> 1];
                o[i] = lap_finish<PIX, ACC>(acc[r][i], (int)((i & 1) ? (w >> 16) : (w & 0xffffu)), p.coef, p.strength, max_value);
            }
            *reinterpret_cast<ushort4 *>(drow + (size_t)r * p.dpitch) = make_ushort4(o[0], o[1], o[2], o[3]);
        }
    }
}

// all three planes of a frame in ONE launch (blockIdx.z = plane; the grid is sized for luma, chroma CTAs beyond their plane
// leave at once): three launches per frame ended in three partial waves
template <typename PIX, typename ACC, bool VEC, int R, int MINB>
__global__ void __launch_bounds__(256, MINB) lapsharp_kernel(const __grid_constant__ LapFrame f)
{
    const LapPlane &p = f.pl[blockIdx.z];
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4, y0 = (blockIdx.y * blockDim.y + threadIdx.y) * R;
    if (x0 >= p.width || y0 >= p.height) return;
    switch (p.kid)                                   // uniform per CTA
    {
        case 0:  lap_tile<PIX, ACC, 0, VEC, R>(p, f.max_value, x0, y0); break;
        case 1:  lap_tile<PIX, ACC, 1, VEC, R>(p, f.max_value, x0, y0); break;
        case 2:  lap_tile<PIX, ACC, 2, VEC, R>(p, f.max_value, x0, y0); break;
        default: lap_tile<PIX, ACC, 3, VEC, R>(p, f.max_value, x0, y0); break;
    }
}

struct Geom { int w, h, pitch; size_t bytes; };

}  // namespace

struct hbcu_lapsharp_s
{
    hbcu_lapsharp_config_t cfg;
    int bps, maxv, slots, next;
    Geom g[3];
    std::vector<uint8_t *> in_base, out_base;    // one allocation per frame, planes back to back at the reference stride
    size_t frame_bytes, plane_off[3];             // = the layout of a STANDARD hb_buffer_t: a frame moves as one copy
    std::vector<uint8_t *> in_mem, out_mem;
    std::vector<int64_t> ticket;
    std::vector<cudaEvent_t> ev_up, ev_k, ev_down;
    cudaStream_t s_h2d, s_compute, s_d2h;
    cudaEvent_t ev_mark[2];
};

namespace {

const double kCoef[4] = { 1.0, 1.0 / 5, 1.0 / 5, 1.0 / 15 };     // lapsharp.c:95-101

// hb_frame_buffer_mirror_stride (fifo.c:906-959) for a frame that never visits the host.  The reference runs its 16-bit
// variant for every format with `width` in samples as the word index: for 8-bit frames the margin comes out negative
// and nothing is written, so only 16-bit planes with a padded stride need this.
__global__ void mirror_stride16_kernel(uint16_t *d, int width, int height, int stride)
{
    const int yy = blockIdx.x * blockDim.y + threadIdx.y;
    if (yy >= height) return;
    const int margin = stride - width, margin_front = margin / 2, margin_back = margin - margin_front;
    const size_t row = (size_t)yy * stride;
    for (int ii = threadIdx.x; ii < margin_back; ii += blockDim.x) d[row + width + ii] = d[row + width - ii - 1];
    for (int ii = threadIdx.x; ii < margin_front; ii += blockDim.x) d[row + stride - 1 - ii] = d[row + stride + ii];
}

int launch_frame(hbcu_lapsharp_s *h, const void *const src[3], const int spitch_elems[3], void *const dst[3])
{
    LapFrame f;
    f.max_value = h->maxv;
    for (int pl = 0; pl < 3; pl++)
    {
        const Geom &g = h->g[pl];
        LapPlane &p = f.pl[pl];
        p.src = src[pl];
        p.dst = dst[pl];
        p.width = g.w; p.height = g.h; p.spitch = spitch_elems[pl]; p.dpitch = g.pitch;
        p.kid = h->cfg.kernel[pl];
        p.coef = kCoef[p.kid];
        p.strength = h->cfg.strength[pl];
        p.vec = ((uintptr_t)src[pl] % 4 == 0) && (((size_t)spitch_elems[pl] * h->bps) % 4 == 0);
    }
    const Geom &g0 = h->g[0];
    const bool vec = f.pl[0].vec && f.pl[1].vec && f.pl[2].vec;
    // 4 rows per thread at 4 CTAs per SM (64 registers) measured best of {2, 4, 8 rows} x {2..6 CTAs}: 47.7k frames/s against
    // 42.7k at 2 CTAs per SM (profiles/r02_lapsharp_variants.txt).  The int -> double conversions stay instructions: building
    // the double from its bit pattern (2^52 + v, then subtract the bias) measured slower, 43.9k against 46.8k on the same box
    // (the two extra DADD and the xor cost more issue slots than the quarter-rate I2F.F64 costs pipe time).
    constexpr int R = 4;
    dim3 blk(32, 8), grid(((g0.w + 3) / 4 + 31) / 32, (g0.h + 8 * R - 1) / (8 * R), 3);
#define LAP(PIX, ACC, MB)                                                                                          \
    do {                                                                                                           \
        if (!vec) lapsharp_kernel<PIX, ACC, false, R, 2><<<grid, blk, 0, h->s_compute>>>(f);                         \
        else      lapsharp_kernel<PIX, ACC, true, R, MB><<<grid, blk, 0, h->s_compute>>>(f);                          \
    } while (0)
    if (h->bps == 1) LAP(uint8_t, int16_t, 4);
    else             LAP(uint16_t, int32_t, 3);          // 85 registers: the 16-bit tile spills at 64
#undef LAP
    hbcu::count_launch();
    HBCU_CHECK(cudaGetLastError());
    return 0;
}

int find_ticket(hbcu_lapsharp_s *h, int64_t t)
{
    for (int s = 0; s < h->slots; s++) if (h->ticket[s] == t) return s;
    return -1;
}

}  // namespace

extern "C" {

int hbcu_lapsharp_create(hbcu_lapsharp_t **out, const hbcu_lapsharp_config_t *cfg)
{
    if (out == nullptr || cfg == nullptr) { set_error("lapsharp_create: null argument"); return -1; }
    *out = nullptr;
    if (cfg->width < 8 || cfg->height < 8 || cfg->depth < 8 || cfg->depth > 16)
    {
        set_error("lapsharp_create: unsupported geometry %dx%d depth %d", cfg->width, cfg->height, cfg->depth);
        return -1;
    }
    for (int c = 0; c < 3; c++)
        if (cfg->kernel[c] < 0 || cfg->kernel[c] > 3) { set_error("lapsharp_create: bad kernel id %d", cfg->kernel[c]); return -1; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev)
    {
        cudaGetLastError();
        set_error("lapsharp_create: CUDA device %d not available (%d devices); there is no CPU fallback", cfg->device, ndev);
        return -1;
    }
    HBCU_CHECK(cudaSetDevice(cfg->device));
    hbcu_lapsharp_s *h = new (std::nothrow) hbcu_lapsharp_s();
    if (h == nullptr) { set_error("lapsharp_create: out of memory"); return -1; }
    h->cfg = *cfg;
    h->bps = cfg->depth > 8 ? 2 : 1;
    h->maxv = (1 << cfg->depth) - 1;
    h->slots = cfg->slots >= 2 ? cfg->slots : 4;
    h->next = 0;
    h->s_h2d = h->s_compute = h->s_d2h = nullptr;
    h->ev_mark[0] = h->ev_mark[1] = nullptr;
    for (int pl = 0; pl < 3; pl++)
    {
        Geom &g = h->g[pl];
        g.w = pl == 0 ? cfg->width : -((-cfg->width) >> cfg->chroma_shift_w);
        g.h = pl == 0 ? cfg->height : -((-cfg->height) >> cfg->chroma_shift_h);
        g.pitch = ((g.w * h->bps + 63) / 64 * 64) / h->bps;          // hb_image_stride
        g.bytes = (size_t)g.pitch * g.h * h->bps;
        h->plane_off[pl] = pl == 0 ? 0 : h->plane_off[pl - 1] + h->g[pl - 1].bytes;
        h->frame_bytes = h->plane_off[pl] + g.bytes;
    }
#define CK(expr)                                                                  \
    do {                                                                          \
        cudaError_t _e = (expr);                                                  \
        if (_e != cudaSuccess) {                                                  \
            set_error("%s failed: %s", #expr, cudaGetErrorString(_e));            \
            hbcu_lapsharp_destroy(h);                                             \
            return -1;                                                            \
        }                                                                         \
    } while (0)
    CK(cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->s_compute, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking));
    h->in_mem.assign(h->slots * 3, nullptr);
    h->out_mem.assign(h->slots * 3, nullptr);
    h->in_base.assign(h->slots, nullptr);
    h->out_base.assign(h->slots, nullptr);
    h->ticket.assign(h->slots, -1);
    h->ev_up.assign(h->slots, nullptr);
    h->ev_k.assign(h->slots, nullptr);
    h->ev_down.assign(h->slots, nullptr);
    for (int s = 0; s < h->slots; s++)
    {
        CK(cudaEventCreateWithFlags(&h->ev_up[s], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_k[s], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_down[s], cudaEventDisableTiming));
        CK(cudaMalloc(&h->in_base[s], h->frame_bytes + 256));
        CK(cudaMemset(h->in_base[s], 0, h->frame_bytes + 256));
        CK(cudaMalloc(&h->out_base[s], h->frame_bytes));
        CK(cudaMemset(h->out_base[s], 0, h->frame_bytes));
        for (int pl = 0; pl < 3; pl++)
        {
            h->in_mem[s * 3 + pl] = h->in_base[s] + h->plane_off[pl];
            h->out_mem[s * 3 + pl] = h->out_base[s] + h->plane_off[pl];
        }
    }
    CK(cudaEventCreate(&h->ev_mark[0]));
    CK(cudaEventCreate(&h->ev_mark[1]));
    // the clearing memsets above ran on the legacy default stream; the handle's non-blocking streams do not wait for it
    CK(cudaDeviceSynchronize());
#undef CK
    *out = h;
    return 0;
}

void hbcu_lapsharp_destroy(hbcu_lapsharp_t *h)
{
    if (h == nullptr) return;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    for (auto p : h->in_base) if (p) cudaFree(p);
    for (auto p : h->out_base) if (p) cudaFree(p);
    for (auto e : h->ev_up) if (e) cudaEventDestroy(e);
    for (auto e : h->ev_k) if (e) cudaEventDestroy(e);
    for (auto e : h->ev_down) if (e) cudaEventDestroy(e);
    if (h->ev_mark[0]) cudaEventDestroy(h->ev_mark[0]);
    if (h->ev_mark[1]) cudaEventDestroy(h->ev_mark[1]);
    if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
    if (h->s_compute) cudaStreamDestroy(h->s_compute);
    if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
    delete h;
}

// the caller's planes have exactly the device layout (back to back, reference stride): the frame is one copy
static bool same_layout(const hbcu_lapsharp_t *h, const void *const planes[3], const int strides[3])
{
    for (int pl = 0; pl < 3; pl++)
    {
        if ((size_t)strides[pl] != (size_t)h->g[pl].pitch * h->bps) return false;
        if ((const uint8_t *)planes[pl] != (const uint8_t *)planes[0] + h->plane_off[pl]) return false;
    }
    return true;
}

int hbcu_lapsharp_filter(hbcu_lapsharp_t *h, int64_t ticket, const void *const in_planes[3], const int in_strides[3],
                         void *const out_planes[3], const int out_strides[3])
{
    if (h == nullptr || in_planes == nullptr || out_planes == nullptr) { set_error("lapsharp_filter: bad argument"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    const int s = h->next;
    h->next = (h->next + 1) % h->slots;
    // the slot's previous frame must have left it (kernel read the input, download read the output)
    HBCU_CHECK(cudaStreamWaitEvent(h->s_h2d, h->ev_k[s], 0));
    const bool whole_in = same_layout(h, in_planes, in_strides);
    if (whole_in) HBCU_CHECK(cudaMemcpyAsync(h->in_base[s], in_planes[0], h->frame_bytes, cudaMemcpyHostToDevice, h->s_h2d));
    for (int pl = 0; pl < 3 && !whole_in; pl++)
    {
        const Geom &g = h->g[pl];
        const bool same = (size_t)in_strides[pl] == (size_t)g.pitch * h->bps;
        HBCU_CHECK(cudaMemcpy2DAsync(h->in_mem[s * 3 + pl], (size_t)g.pitch * h->bps, in_planes[pl], (size_t)in_strides[pl],
                                     same ? (size_t)g.pitch * h->bps : (size_t)g.w * h->bps, (size_t)g.h, cudaMemcpyHostToDevice, h->s_h2d));
    }
    HBCU_CHECK(cudaEventRecord(h->ev_up[s], h->s_h2d));
    HBCU_CHECK(cudaStreamWaitEvent(h->s_compute, h->ev_up[s], 0));
    HBCU_CHECK(cudaStreamWaitEvent(h->s_compute, h->ev_down[s], 0));
    {
        const void *srcs[3] = { h->in_mem[s * 3 + 0], h->in_mem[s * 3 + 1], h->in_mem[s * 3 + 2] };
        void *dsts[3] = { h->out_mem[s * 3 + 0], h->out_mem[s * 3 + 1], h->out_mem[s * 3 + 2] };
        const int sp[3] = { h->g[0].pitch, h->g[1].pitch, h->g[2].pitch };
        if (launch_frame(h, srcs, sp, dsts) != 0) return -1;
    }
    HBCU_CHECK(cudaEventRecord(h->ev_k[s], h->s_compute));
    HBCU_CHECK(cudaStreamWaitEvent(h->s_d2h, h->ev_k[s], 0));
    const bool whole_out = same_layout(h, out_planes, out_strides);
    if (whole_out) HBCU_CHECK(cudaMemcpyAsync(out_planes[0], h->out_base[s], h->frame_bytes, cudaMemcpyDeviceToHost, h->s_d2h));
    for (int pl = 0; pl < 3 && !whole_out; pl++)
    {
        const Geom &g = h->g[pl];
        HBCU_CHECK(cudaMemcpy2DAsync(out_planes[pl], (size_t)out_strides[pl], h->out_mem[s * 3 + pl], (size_t)g.pitch * h->bps,
                                     (size_t)g.w * h->bps, (size_t)g.h, cudaMemcpyDeviceToHost, h->s_d2h));
    }
    HBCU_CHECK(cudaEventRecord(h->ev_down[s], h->s_d2h));
    h->ticket[s] = ticket;
    return 0;
}

static bool frame_fits(const hbcu_lapsharp_t *h, const hbcu_frame_t *f)
{
    if (f->device != h->cfg.device) return false;
    for (int pl = 0; pl < 3; pl++)
        if (f->row_bytes[pl] != h->g[pl].w * h->bps || f->rows[pl] != h->g[pl].h || f->stride[pl] != h->g[pl].pitch * h->bps) return false;
    return true;
}

int hbcu_lapsharp_filter_frames(hbcu_lapsharp_t *h, int64_t ticket,
                                hbcu_frame_t *in_frame, const void *const in_planes[3], const int in_strides[3],
                                hbcu_frame_t *out_frame, void *const out_planes[3], const int out_strides[3])
{
    if (h == nullptr || (in_frame == nullptr && (in_planes == nullptr || in_strides == nullptr)) ||
        (out_frame == nullptr && (out_planes == nullptr || out_strides == nullptr)) ||
        (in_frame && !frame_fits(h, in_frame)) || (out_frame && !frame_fits(h, out_frame)))
    {
        set_error("lapsharp_filter_frames: bad argument or frame geometry");
        return -1;
    }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    const int s = h->next;
    h->next = (h->next + 1) % h->slots;
    if (in_frame == nullptr)
    {
        HBCU_CHECK(cudaStreamWaitEvent(h->s_h2d, h->ev_k[s], 0));
        const bool whole_in = same_layout(h, in_planes, in_strides);
        if (whole_in) HBCU_CHECK(cudaMemcpyAsync(h->in_base[s], in_planes[0], h->frame_bytes, cudaMemcpyHostToDevice, h->s_h2d));
        for (int pl = 0; pl < 3 && !whole_in; pl++)
        {
            const Geom &g = h->g[pl];
            const bool same = (size_t)in_strides[pl] == (size_t)g.pitch * h->bps;
            HBCU_CHECK(cudaMemcpy2DAsync(h->in_mem[s * 3 + pl], (size_t)g.pitch * h->bps, in_planes[pl], (size_t)in_strides[pl],
                                         same ? (size_t)g.pitch * h->bps : (size_t)g.w * h->bps, (size_t)g.h, cudaMemcpyHostToDevice, h->s_h2d));
        }
        HBCU_CHECK(cudaEventRecord(h->ev_up[s], h->s_h2d));
        HBCU_CHECK(cudaStreamWaitEvent(h->s_compute, h->ev_up[s], 0));
    }
    else if (hbcu::frame_begin_read(in_frame, h->s_compute) != 0) return -1;
    // lapsharp.c:333 mirrors the picture into the stride padding first; a device frame gets that in a private copy
    bool staged = false;
    if (in_frame != nullptr && h->bps == 2)
        for (int pl = 0; pl < 3; pl++) staged = staged || h->g[pl].pitch != h->g[pl].w;
    if (staged)
    {
        HBCU_CHECK(cudaStreamWaitEvent(h->s_compute, h->ev_k[s], 0));
        HBCU_CHECK(cudaMemcpyAsync(h->in_base[s], in_frame->base, h->frame_bytes, cudaMemcpyDeviceToDevice, h->s_compute));
        for (int pl = 0; pl < 3; pl++)
        {
            const Geom &g = h->g[pl];
            if (g.pitch == g.w) continue;
            mirror_stride16_kernel<<<(g.h + 7) / 8, dim3(32, 8), 0, h->s_compute>>>((uint16_t *)h->in_mem[s * 3 + pl], g.w, g.h, g.pitch);
            hbcu::count_launch();
        }
        HBCU_CHECK(cudaGetLastError());
    }
    HBCU_CHECK(cudaStreamWaitEvent(h->s_compute, h->ev_down[s], 0));
    if (out_frame && hbcu::frame_begin_write(out_frame, h->s_compute) != 0) return -1;
    {
        const void *srcs[3];
        void *dsts[3];
        int sp[3];
        for (int pl = 0; pl < 3; pl++)
        {
            srcs[pl] = (in_frame && !staged) ? (const void *)in_frame->plane[pl] : (const void *)h->in_mem[s * 3 + pl];
            dsts[pl] = out_frame ? (void *)out_frame->plane[pl] : (void *)h->out_mem[s * 3 + pl];
            sp[pl] = h->g[pl].pitch;
        }
        if (launch_frame(h, srcs, sp, dsts) != 0) return -1;
    }
    HBCU_CHECK(cudaEventRecord(h->ev_k[s], h->s_compute));
    if (in_frame && hbcu::frame_end_read(in_frame, h->s_compute) != 0) return -1;
    if (out_frame)
    {
        if (hbcu::frame_end_write(out_frame, h->s_compute) != 0) return -1;
        HBCU_CHECK(cudaEventRecord(h->ev_down[s], h->s_compute));
    }
    else
    {
        HBCU_CHECK(cudaStreamWaitEvent(h->s_d2h, h->ev_k[s], 0));
        const bool whole_out = same_layout(h, out_planes, out_strides);
        if (whole_out) HBCU_CHECK(cudaMemcpyAsync(out_planes[0], h->out_base[s], h->frame_bytes, cudaMemcpyDeviceToHost, h->s_d2h));
        for (int pl = 0; pl < 3 && !whole_out; pl++)
        {
            const Geom &g = h->g[pl];
            HBCU_CHECK(cudaMemcpy2DAsync(out_planes[pl], (size_t)out_strides[pl], h->out_mem[s * 3 + pl], (size_t)g.pitch * h->bps,
                                         (size_t)g.w * h->bps, (size_t)g.h, cudaMemcpyDeviceToHost, h->s_d2h));
        }
        HBCU_CHECK(cudaEventRecord(h->ev_down[s], h->s_d2h));
    }
    h->ticket[s] = ticket;
    return 0;
}

int hbcu_lapsharp_filter_device(hbcu_lapsharp_t *h, int64_t ticket, const void *const dplanes[3], const int strides[3],
                                void *out_planes[3], int out_strides[3])
{
    if (h == nullptr || dplanes == nullptr || strides == nullptr) { set_error("lapsharp_filter_device: bad argument"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    const int s = h->next;
    h->next = (h->next + 1) % h->slots;
    {
        void *dsts[3] = { h->out_mem[s * 3 + 0], h->out_mem[s * 3 + 1], h->out_mem[s * 3 + 2] };
        const int sp[3] = { strides[0] / h->bps, strides[1] / h->bps, strides[2] / h->bps };
        if (launch_frame(h, dplanes, sp, dsts) != 0) return -1;
    }
    HBCU_CHECK(cudaEventRecord(h->ev_k[s], h->s_compute));
    HBCU_CHECK(cudaEventRecord(h->ev_down[s], h->s_compute));
    h->ticket[s] = ticket;
    for (int pl = 0; pl < 3; pl++)
    {
        if (out_planes) out_planes[pl] = h->out_mem[s * 3 + pl];
        if (out_strides) out_strides[pl] = h->g[pl].pitch * h->bps;
    }
    return 0;
}

int hbcu_lapsharp_wait(hbcu_lapsharp_t *h, int64_t ticket)
{
    if (h == nullptr) { set_error("lapsharp_wait: null handle"); return -1; }
    const int s = find_ticket(h, ticket);
    if (s < 0) { set_error("lapsharp_wait: ticket %lld is not in flight", (long long)ticket); return -1; }
    HBCU_CHECK(cudaEventSynchronize(h->ev_down[s]));
    return 0;
}

int hbcu_lapsharp_poll(hbcu_lapsharp_t *h, int64_t ticket)
{
    if (h == nullptr) { set_error("lapsharp_poll: null handle"); return -1; }
    const int s = find_ticket(h, ticket);
    if (s < 0) { set_error("lapsharp_poll: ticket %lld is not in flight", (long long)ticket); return -1; }
    cudaError_t e = cudaEventQuery(h->ev_down[s]);
    if (e == cudaSuccess) return 1;
    if (e == cudaErrorNotReady) return 0;
    set_error("lapsharp_poll: %s", cudaGetErrorString(e));
    return -1;
}

int hbcu_lapsharp_sync(hbcu_lapsharp_t *h)
{
    if (h == nullptr) { set_error("lapsharp_sync: null handle"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    HBCU_CHECK(cudaStreamSynchronize(h->s_h2d));
    HBCU_CHECK(cudaStreamSynchronize(h->s_compute));
    HBCU_CHECK(cudaStreamSynchronize(h->s_d2h));
    return 0;
}

int hbcu_lapsharp_mark(hbcu_lapsharp_t *h, int which)
{
    if (h == nullptr || which < 0 || which > 1) { set_error("lapsharp_mark: bad argument"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    HBCU_CHECK(cudaEventRecord(h->ev_mark[which], h->s_compute));
    return 0;
}

int hbcu_lapsharp_elapsed_ms(hbcu_lapsharp_t *h, float *ms)
{
    if (h == nullptr || ms == nullptr) { set_error("lapsharp_elapsed_ms: bad argument"); return -1; }
    HBCU_CHECK(cudaEventSynchronize(h->ev_mark[1]));
    HBCU_CHECK(cudaEventElapsedTime(ms, h->ev_mark[0], h->ev_mark[1]));
    return 0;
}

}  // extern "C"
