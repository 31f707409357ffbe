// comb_detect.cu -- comb detection for sm_100a behind the C-ABI of include/hbcu.h.
//
// Replaces (reference /root/reference/libhb):
//   detect_gamma_combed_segment / detect_combed_segment   templates/comb_detect_template.c:288-402, 789-933
//   mask_filter_work / mask_erode_work / mask_dilate_work comb_detect.c:901-966, 726-792, 556-622
//   check_filtered_combing_mask / check_combing_mask      comb_detect.c:221-276, 384-454
//   check_combing_results                                 comb_detect.c:1029-1049
// The reference runs five fork/join tasksets over row segments; here one frame is
// three kernels on one stream, all on a one-bit-per-pixel mask:
//   comb_mask_bits2_kernel   raw mask from the prev/cur/next luma planes (gamma values come from the
//                            host-built table staged in shared memory, so the float results are the
//                            reference's bit for bit; no FMA contraction: -fmad=false + explicit rn ops)
//   comb_filter_bits_kernel  filter -> erode -> dilate -> erode fused in shared memory,
//                            intermediate masks never touch HBM
//   comb_score_bits_kernel   block sums -> LIGHT/HEAVY flags (atomicOr), verdict read back through
//                            pinned memory
// Integer work is bit-exact by construction; the segment decomposition of the reference does
// not influence its result (block grid is globally aligned, SURVEY.md 8a/a14).
#include "hbcu_common.h"
#include "hbcu_frames.h"
#include "../../include/hbcu.h"

#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

namespace {

using hbcu::set_error;

struct CombParams
{
    int w, h, pitch;              // luma plane, pitch in elements
    int mode, spatial_metric, filter_mode;
    int mthresh, athresh, athresh_sq, athresh6;
    int c32min, c32max;
    float g_mthresh, g_athresh, g_athresh6;
    int force;
    int lut_size;
    const float *gamma_lut;
    int block_threshold, block_width, block_height;
};

// ---------------------------------------------------------------------------
// The combing mask is one bit per pixel: a warp evaluates 32 neighbouring pixels and
// __ballot_sync() delivers their mask word; the whole filter chain (filter -> erode -> dilate -> erode, comb_detect.c:
// 556-966) then runs on 32 pixels per integer instruction -- neighbours are shifted words, the "n of 8 neighbours"
// rules a bit-sliced adder tree -- and block scores are popcounts.  Mask traffic drops from 8 bytes to 4 bits per pixel
// and the three mask passes from ~165 us to a few us per 4K frame.
//   bit plane layout: row y, word wx at  bits[(y + kGuard) * wpitch + 1 + wx];  kGuard zero rows above and below and one
//   zero word left and right of every row are never written, so neighbours need no bounds checks.
// ---------------------------------------------------------------------------
constexpr int kGuard = 4;
constexpr int kMaskRows = 16;                  // rows a thread marches down in the mask kernel

enum { OP_CLASSIC = 0, OP_HV = 1, OP_ERODE = 2, OP_DILATE = 3 };

// the first gate of the decision (comb_detect_template.c:300-312): both vertical neighbours differ from the sample in the
// same direction by more than the threshold.  Only samples that pass need the previous / next frame at all.
template <bool GAMMA>
__device__ __forceinline__ bool comb_spatial(const CombParams &p, int pu1, int pc, int pd1, float gu1, float gc, float gd1)
{
    if (GAMMA)
    {
        const float up = __fsub_rn(gc, gu1), down = __fsub_rn(gc, gd1);
        return (up > p.g_athresh && down > p.g_athresh) || (up < -p.g_athresh && down < -p.g_athresh);
    }
    const int up = pc - pu1, down = pc - pd1;
    return (up > p.athresh && down > p.athresh) || (up < -p.athresh && down < -p.athresh);
}

// the rest for a sample that passed comb_spatial: motion against the previous / next frame (q* / n*: rows y-1, y, y+1
// of those frames, as samples or as gamma values), then the spatial metric
template <bool GAMMA>
__device__ __forceinline__ int comb_rest(const CombParams &p, int pu2, int pu1, int pc, int pd1, int pd2,
                                         float gu2, float gu1, float gc, float gd1, float gd2,
                                         int qu1, int qc, int qd1, int nu1, int nc, int nd1,
                                         float qgu1, float qgc, float qgd1, float ngu1, float ngc, float ngd1)
{
    if (GAMMA)
    {
        int motion = 0;
        if (p.g_mthresh > 0)
        {
            if (fabsf(__fsub_rn(qgc, gc)) > p.g_mthresh && fabsf(__fsub_rn(gu1, ngu1)) > p.g_mthresh &&
                fabsf(__fsub_rn(gd1, ngd1)) > p.g_mthresh)
                motion++;
            if (fabsf(__fsub_rn(ngc, gc)) > p.g_mthresh && fabsf(__fsub_rn(qgu1, gu1)) > p.g_mthresh &&
                fabsf(__fsub_rn(qgd1, gd1)) > p.g_mthresh)
                motion++;
        }
        else
            motion = 1;
        if (!(motion || p.force)) return 0;
        const float lhs = __fadd_rn(__fadd_rn(gu2, __fmul_rn(4.0f, gc)), gd2);     // left to right, no contraction
        const float rhs = __fmul_rn(3.0f, __fadd_rn(gu1, gd1));
        return fabsf(__fsub_rn(lhs, rhs)) > p.g_athresh6;
    }
    int motion = 0;
    if (p.mthresh > 0)
    {
        if (abs(qc - pc) > p.mthresh && abs(pu1 - nu1) > p.mthresh && abs(pd1 - nd1) > p.mthresh) motion++;
        if (abs(nc - pc) > p.mthresh && abs(qu1 - pu1) > p.mthresh && abs(qd1 - pd1) > p.mthresh) motion++;
    }
    else
        motion = 1;
    if (!(motion || p.force)) return 0;
    if (p.spatial_metric == 0) return (abs(pc - pd2) < p.c32min) && (abs(pc - pd1) > p.c32max);
    if (p.spatial_metric == 1) return (pu1 - pc) * (pd1 - pc) > p.athresh_sq;
    if (p.spatial_metric == 2) return abs(pu2 + 4 * pc + pd2 - 3 * (pu1 + pd1)) > p.athresh6;
    return 0;
}

// The mask kernel, in three phases rather than a row loop that stalls on its own loads: (1) the spatial gate of all kMaskRows
// rows from the column segment in registers; (2) every previous / next-frame sample some gated row of this lane needs (rows
// y-1, y, y+1: consecutive output rows share two of three) issued back to back as predicated loads, then their gamma
// lookups; (3) the motion tests and the metric, ballots and stores.  A row loop in which each gated row fetches its own six
// samples has up to 16 exposed DRAM round trips per lane (8.3 long-scoreboard stalls per issue,
// profiles/r02_comb_mask_ncu.json) and fetches every sample up to three times: 49.2 us against 37.8 us for the 4K 10-bit
// luma plane (profiles/r02_comb_mask2_ncu.json).
template <typename PIX, bool GAMMA>
__global__ void __launch_bounds__(256) comb_mask_bits2_kernel(const PIX *__restrict__ prev, const PIX *__restrict__ cur,
                                                             const PIX *__restrict__ next, uint32_t *__restrict__ bits,
                                                             int wpitch, CombParams p)
{
    extern __shared__ float s_lut[];
    if (GAMMA)
    {
        for (int i = threadIdx.x; i < p.lut_size; i += blockDim.x) s_lut[i] = p.gamma_lut[i];
        __syncthreads();
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wx = blockIdx.x * 8 + warp;
    if (wx * 32 >= p.w) return;                               // whole warp
    const int x = wx * 32 + lane;
    const bool colok = x < p.w;
    const int xc = colok ? x : p.w - 1;
    const int y0 = blockIdx.y * kMaskRows;
    int c[kMaskRows + 4];
    float g[kMaskRows + 4];
#pragma unroll
    for (int k = 0; k < kMaskRows + 4; k++)
        c[k] = cur[(size_t)min(max(y0 - 2 + k, 0), p.h - 1) * p.pitch + xc];
#pragma unroll
    for (int k = 0; k < kMaskRows + 4; k++)
        g[k] = GAMMA ? s_lut[c[k]] : 0.f;
    unsigned gate = 0;
#pragma unroll
    for (int r = 0; r < kMaskRows; r++)
    {
        const int y = y0 + r;
        if (colok && y >= 2 && y < p.h - 2 && comb_spatial<GAMMA>(p, c[r + 1], c[r + 2], c[r + 3], g[r + 1], g[r + 2], g[r + 3])) gate |= 1u << r;
    }
    // window row k <-> picture row y0 - 1 + k; output row r reads k = r, r + 1, r + 2 (inside the picture: 2 <= y < h - 2)
    const bool motion_test = GAMMA ? p.g_mthresh > 0 : p.mthresh > 0;
    const unsigned need = motion_test ? (gate | (gate << 1) | (gate << 2)) : 0u;
    int q[kMaskRows + 2], n[kMaskRows + 2];
    float qg[kMaskRows + 2], ng[kMaskRows + 2];
    const PIX *pcol = prev + (size_t)(y0 - 1) * p.pitch + xc, *ncol = next + (size_t)(y0 - 1) * p.pitch + xc;
#pragma unroll
    for (int k = 0; k < kMaskRows + 2; k++)
    {
        q[k] = n[k] = 0;
        if ((need >> k) & 1u)
        {
            q[k] = pcol[(size_t)k * p.pitch];
            n[k] = ncol[(size_t)k * p.pitch];
        }
    }
#pragma unroll
    for (int k = 0; k < kMaskRows + 2; k++)
    {
        qg[k] = ng[k] = 0.f;
        if (GAMMA && ((need >> k) & 1u)) { qg[k] = s_lut[q[k]]; ng[k] = s_lut[n[k]]; }
    }
#pragma unroll
    for (int r = 0; r < kMaskRows; r++)
    {
        const int y = y0 + r;
        if (y >= p.h) break;                                  // warp uniform
        int m = 0;
        if ((gate >> r) & 1u)
            m = comb_rest<GAMMA>(p, c[r], c[r + 1], c[r + 2], c[r + 3], c[r + 4], g[r], g[r + 1], g[r + 2], g[r + 3], g[r + 4],
                                 q[r], q[r + 1], q[r + 2], n[r], n[r + 1], n[r + 2],
                                 qg[r], qg[r + 1], qg[r + 2], ng[r], ng[r + 1], ng[r + 2]);
        const uint32_t word = __ballot_sync(0xffffffffu, m != 0);
        if (lane == 0) bits[(size_t)(y + kGuard) * wpitch + 1 + wx] = word;
    }
}

struct Nb { uint32_t l, c, r; };      // the words of the left / same / right pixel of every bit position
__device__ __forceinline__ Nb neighbours(const uint32_t *row, int ci, int ncols)
{
    const uint32_t w = row[ci], wl = ci > 0 ? row[ci - 1] : 0u, wr = ci + 1 < ncols ? row[ci + 1] : 0u;
    return Nb{ (w << 1) | (wl >> 31), w, (w >> 1) | (wr << 31) };
}
__device__ __forceinline__ void full_add(uint32_t a, uint32_t b, uint32_t c, uint32_t &s, uint32_t &cy)
{
    const uint32_t t = a ^ b;
    s = t ^ c;
    cy = (a & b) | (c & t);
}

constexpr int BT_W = 8, BT_R = 32;                           // tile: 8 words (256 pixels) x 32 rows, halo kGuard rows / one word
constexpr int BS_W = BT_W + 2, BS_R = BT_R + 2 * kGuard;

__device__ __forceinline__ void bits_stage(const uint32_t *src, uint32_t *dst, int op, int shrink, int wx0, int gy0, int w, int h)
{
    const int rows = BS_R - 2 * shrink;
    for (int i = threadIdx.x; i < rows * BS_W; i += blockDim.x)
    {
        const int r = shrink + i / BS_W, ci = i % BS_W;
        const int gy = gy0 + r, wx = wx0 + ci;
        uint32_t v = 0;
        if (gy >= 1 && gy <= h - 2)
        {
            const Nb c = neighbours(src + r * BS_W, ci, BS_W);
            if (op == OP_CLASSIC || op == OP_HV)
            {
                v = c.l & c.c & c.r;
                if (op == OP_HV) v &= src[(r - 1) * BS_W + ci] & src[(r + 1) * BS_W + ci];
            }
            else
            {
                const Nb u = neighbours(src + (r - 1) * BS_W, ci, BS_W), d = neighbours(src + (r + 1) * BS_W, ci, BS_W);
                // bit-sliced count of the 8 neighbours
                uint32_t s1, c1, s2, c2, b0, c4, t, c5;
                full_add(u.l, u.c, u.r, s1, c1);
                full_add(d.l, d.c, d.r, s2, c2);
                const uint32_t s3 = c.l ^ c.r, c3 = c.l & c.r;
                full_add(s1, s2, s3, b0, c4);
                full_add(c1, c2, c3, t, c5);
                const uint32_t b1 = t ^ c4, c6 = t & c4;
                const uint32_t b2 = c5 ^ c6, b3 = c5 & c6;
                (void)b0;
                if (op == OP_ERODE) v = c.c & (b1 | b2 | b3);            // keep a set pixel with >= 2 set neighbours
                else                v = c.c | b2 | b3;                   // set a pixel with >= 4 set neighbours
            }
            // columns 1 .. w-2 only
            const int gx0 = wx * 32;
            uint32_t vm = 0xffffffffu;
            if (gx0 < 1) vm &= ~1u;
            if (gx0 + 31 > w - 2) vm = (w - 2 - gx0 >= 0) ? (vm & (0xffffffffu >> (31 - (w - 2 - gx0)))) : 0u;
            if (wx < 0) vm = 0u;
            v &= vm;
        }
        dst[r * BS_W + ci] = v;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(256) comb_filter_bits_kernel(const uint32_t *__restrict__ raw, uint32_t *__restrict__ out,
                                                              int wpitch, int nwords, int w, int h, int filter_mode)
{
    __shared__ uint32_t a[BS_R * BS_W], b[BS_R * BS_W];
    const int wx0 = blockIdx.x * BT_W - 1, gy0 = blockIdx.y * BT_R - kGuard;
    for (int i = threadIdx.x; i < BS_R * BS_W; i += blockDim.x)
    {
        const int gy = gy0 + i / BS_W, wx = wx0 + i % BS_W;
        a[i] = (gy >= -kGuard && gy < h + kGuard && wx >= -1 && wx <= nwords) ? raw[(size_t)(gy + kGuard) * wpitch + 1 + wx] : 0u;
        b[i] = 0;
    }
    __syncthreads();
    const uint32_t *res;
    if (filter_mode == 1)
    {
        bits_stage(a, b, OP_CLASSIC, 1, wx0, gy0, w, h);
        res = b;
    }
    else
    {
        bits_stage(a, b, OP_HV, 1, wx0, gy0, w, h);              // mask -> temp
        if (filter_mode == 2)
        {
            bits_stage(b, a, OP_ERODE, 2, wx0, gy0, w, h);       // temp -> filtered
            bits_stage(a, b, OP_DILATE, 3, wx0, gy0, w, h);      // filtered -> temp
            bits_stage(b, a, OP_ERODE, 4, wx0, gy0, w, h);       // temp -> filtered
            res = a;
        }
        else
            res = nullptr;                                        // nothing ever writes mask_filtered: stays 0
    }
    for (int i = threadIdx.x; i < BT_R * BT_W; i += blockDim.x)
    {
        const int r = kGuard + i / BT_W, ci = 1 + i % BT_W;
        const int gy = gy0 + r, wx = wx0 + ci;
        if (gy < h && wx < nwords) out[(size_t)(gy + kGuard) * wpitch + 1 + wx] = res ? res[r * BS_W + ci] : 0u;
    }
}

// block scores on a bit plane: one warp per block, a lane per row
__global__ void __launch_bounds__(128) comb_score_bits_kernel(const uint32_t *__restrict__ bits, int wpitch, int w, int h,
                                                             int bw, int bh, int nbx, int nby, int threshold, int filtered,
                                                             int *__restrict__ flags)
{
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= nbx * nby) return;
    const int x0 = (warp % nbx) * bw, y0 = (warp / nbx) * bh;
    int score = 0;
    for (int r = lane; r < bh; r += 32)
    {
        const uint32_t *row = bits + (size_t)(y0 + r + kGuard) * wpitch + 1;
        for (int wx = x0 >> 5; wx <= (x0 + bw - 1) >> 5; wx++)
        {
            uint32_t v = row[wx];
            if (!filtered)
            {
                // check_combing_mask (:384-454): score counts p[x-1] & p[x] & p[x+1]; at x == 0 / x == w-1 the missing side is dropped
                uint32_t l = (v << 1) | (row[wx - 1] >> 31), rr = (v >> 1) | (row[wx + 1] << 31);
                if (wx == 0) l |= 1u;
                if (wx == (w - 1) >> 5) rr |= 1u << ((w - 1) & 31);
                v &= l & rr;
            }
            const int lo = max(x0 - wx * 32, 0), hi = min(x0 + bw - 1 - wx * 32, 31);
            const uint32_t m = (0xffffffffu >> (31 - hi)) & (0xffffffffu << lo);
            score += __popc(v & m);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) score += __shfl_xor_sync(0xffffffffu, score, o);
    if (lane == 0)
    {
        int f = 0;
        if (score >= threshold / 2) f |= 1;
        if (score > threshold) f |= 2;
        if (f) atomicOr(flags, f);
    }
}

// test hook: bit plane -> byte mask
__global__ void __launch_bounds__(256) comb_unpack_bits_kernel(const uint32_t *__restrict__ bits, int wpitch, uint8_t *__restrict__ mask, int mpitch, int w, int h)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x < w && y < h) mask[(size_t)y * mpitch + x] = (bits[(size_t)(y + kGuard) * wpitch + 1 + (x >> 5)] >> (x & 31)) & 1u;
}

}  // namespace

struct hbcu_comb_detect_s
{
    hbcu_comb_detect_config_t cfg;
    int bps, pitch, mpitch;
    size_t plane_bytes;
    int slots;
    std::vector<uint8_t *> luma;
    std::vector<int64_t> index;
    std::vector<cudaEvent_t> ev_upload, ev_readers;
    uint8_t *d_mask, *d_scored;      // byte masks unpacked from the bit planes for hbcu_comb_detect_masks
    uint32_t *d_bits, *d_fbits;      // raw / filtered bit planes
    int wpitch, nwords;
    float *d_lut;
    int nres;
    int *d_flags;            // nres ints
    int *h_flags;            // pinned
    std::vector<int64_t> res_index;
    std::vector<cudaEvent_t> ev_result;
    int next_res;
    cudaStream_t s_h2d, s_compute;
    cudaEvent_t ev_mark[2];
};

extern "C" {

int hbcu_comb_detect_create(hbcu_comb_detect_t **out, const hbcu_comb_detect_config_t *cfg)
{
    if (out == nullptr || cfg == nullptr || cfg->gamma_lut == nullptr)
    {
        set_error("comb_detect_create: null argument");
        return -1;
    }
    *out = nullptr;
    if (cfg->width < 4 || cfg->height < 5 || cfg->depth < 8 || cfg->depth > 16 || cfg->block_width < 1 || cfg->block_height < 1)
    {
        set_error("comb_detect_create: unsupported geometry %dx%d depth %d", cfg->width, cfg->height, cfg->depth);
        return -1;
    }
    if ((cfg->mode & 1) != 0 && ((size_t)sizeof(float) << cfg->depth) > 48 * 1024)
    {
        // refused here, where the job can still continue without the filter (work.c:1861-1868), not per frame
        set_error("comb_detect_create: the gamma table of mode %d at depth %d does not fit shared memory (depths up to 13)", cfg->mode, cfg->depth);
        return -1;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev)
    {
        cudaGetLastError();
        set_error("comb_detect_create: CUDA device %d not available (%d devices); there is no CPU fallback", cfg->device, ndev);
        return -1;
    }
    HBCU_CHECK(cudaSetDevice(cfg->device));
    hbcu_comb_detect_s *h = new (std::nothrow) hbcu_comb_detect_s();
    if (h == nullptr) { set_error("comb_detect_create: out of memory"); return -1; }
    h->cfg = *cfg;
    h->bps = cfg->depth > 8 ? 2 : 1;
    h->pitch = (cfg->width + 127) / 128 * 128;
    h->mpitch = h->pitch;
    h->plane_bytes = (size_t)h->pitch * cfg->height * h->bps;
    h->slots = cfg->slots >= 4 ? cfg->slots : 4;
    h->nres = 16;
    h->next_res = 0;
    h->d_mask = h->d_scored = nullptr;
    h->d_bits = h->d_fbits = nullptr;
    h->nwords = (cfg->width + 31) / 32;
    h->wpitch = h->nwords + 2;
    h->d_lut = nullptr;
    h->d_flags = nullptr;
    h->h_flags = nullptr;
    h->s_h2d = h->s_compute = nullptr;
    h->ev_mark[0] = h->ev_mark[1] = nullptr;
#define CK(expr)                                                                  \
    do {                                                                          \
        cudaError_t _e = (expr);                                                  \
        if (_e != cudaSuccess) {                                                  \
            set_error("%s failed: %s", #expr, cudaGetErrorString(_e));            \
            hbcu_comb_detect_destroy(h);                                          \
            return -1;                                                            \
        }                                                                         \
    } while (0)
    CK(cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->s_compute, cudaStreamNonBlocking));
    h->luma.assign(h->slots, nullptr);
    h->index.assign(h->slots, -1);
    h->ev_upload.assign(h->slots, nullptr);
    h->ev_readers.assign(h->slots, nullptr);
    for (int s = 0; s < h->slots; s++)
    {
        CK(cudaMalloc(&h->luma[s], h->plane_bytes));
        CK(cudaEventCreateWithFlags(&h->ev_upload[s], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_readers[s], cudaEventDisableTiming));
    }
    const size_t mbytes = (size_t)h->mpitch * cfg->height;
    CK(cudaMalloc(&h->d_mask, mbytes));
    CK(cudaMalloc(&h->d_scored, mbytes));
    CK(cudaMemset(h->d_mask, 0, mbytes));
    CK(cudaMemset(h->d_scored, 0, mbytes));
    const size_t bbytes = (size_t)h->wpitch * (cfg->height + 2 * kGuard) * sizeof(uint32_t);
    CK(cudaMalloc(&h->d_bits, bbytes));
    CK(cudaMalloc(&h->d_fbits, bbytes));
    CK(cudaMemset(h->d_bits, 0, bbytes));
    CK(cudaMemset(h->d_fbits, 0, bbytes));
    const int lut_size = 1 << cfg->depth;
    CK(cudaMalloc(&h->d_lut, lut_size * sizeof(float)));
    CK(cudaMemcpy(h->d_lut, cfg->gamma_lut, lut_size * sizeof(float), cudaMemcpyHostToDevice));
    h->cfg.gamma_lut = nullptr;   // the caller's table is not kept
    CK(cudaMalloc(&h->d_flags, h->nres * sizeof(int)));
    CK(cudaHostAlloc(&h->h_flags, h->nres * sizeof(int), cudaHostAllocPortable));
    h->res_index.assign(h->nres, -1);
    h->ev_result.assign(h->nres, nullptr);
    for (int r = 0; r < h->nres; r++) CK(cudaEventCreateWithFlags(&h->ev_result[r], cudaEventDisableTiming));
    CK(cudaEventCreate(&h->ev_mark[0]));
    CK(cudaEventCreate(&h->ev_mark[1]));
    // the clearing memsets above ran on the legacy default stream; the handle's non-blocking streams do not wait for it
    CK(cudaDeviceSynchronize());
#undef CK
    *out = h;
    return 0;
}

void hbcu_comb_detect_destroy(hbcu_comb_detect_t *h)
{
    if (h == nullptr) return;
    cudaSetDevice(h->cfg.device);
    cudaDeviceSynchronize();
    for (auto p : h->luma) if (p) cudaFree(p);
    for (auto e : h->ev_upload) if (e) cudaEventDestroy(e);
    for (auto e : h->ev_readers) if (e) cudaEventDestroy(e);
    for (auto e : h->ev_result) if (e) cudaEventDestroy(e);
    if (h->d_mask) cudaFree(h->d_mask);
    if (h->d_scored) cudaFree(h->d_scored);
    if (h->d_bits) cudaFree(h->d_bits);
    if (h->d_fbits) cudaFree(h->d_fbits);
    if (h->d_lut) cudaFree(h->d_lut);
    if (h->d_flags) cudaFree(h->d_flags);
    if (h->h_flags) cudaFreeHost(h->h_flags);
    if (h->ev_mark[0]) cudaEventDestroy(h->ev_mark[0]);
    if (h->ev_mark[1]) cudaEventDestroy(h->ev_mark[1]);
    if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
    if (h->s_compute) cudaStreamDestroy(h->s_compute);
    delete h;
}

static int comb_upload(hbcu_comb_detect_t *h, int64_t index, const void *luma, int stride, cudaMemcpyKind kind)
{
    if (h == nullptr || luma == nullptr || index < 0) { set_error("comb_detect_upload: bad argument"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    const int slot = (int)(index % h->slots);
    HBCU_CHECK(cudaStreamWaitEvent(h->s_h2d, h->ev_readers[slot], 0));
    HBCU_CHECK(cudaMemcpy2DAsync(h->luma[slot], (size_t)h->pitch * h->bps, luma, (size_t)stride,
                                 (size_t)h->cfg.width * h->bps, (size_t)h->cfg.height, kind, h->s_h2d));
    HBCU_CHECK(cudaEventRecord(h->ev_upload[slot], h->s_h2d));
    h->index[slot] = index;
    return 0;
}

int hbcu_comb_detect_upload(hbcu_comb_detect_t *h, int64_t index, const void *luma, int stride)
{
    return comb_upload(h, index, luma, stride, cudaMemcpyHostToDevice);
}

int hbcu_comb_detect_upload_device(hbcu_comb_detect_t *h, int64_t index, const void *dluma, int stride)
{
    return comb_upload(h, index, dluma, stride, cudaMemcpyDeviceToDevice);
}

int hbcu_comb_detect_upload_frame(hbcu_comb_detect_t *h, int64_t index, hbcu_frame_t *in)
{
    if (h == nullptr || in == nullptr || in->device != h->cfg.device || in->row_bytes[0] != h->cfg.width * h->bps || in->rows[0] != h->cfg.height)
    {
        set_error("comb_detect_upload_frame: bad argument or frame geometry");
        return -1;
    }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    if (hbcu::frame_begin_read(in, h->s_h2d) != 0) return -1;
    if (comb_upload(h, index, in->plane[0], in->stride[0], cudaMemcpyDeviceToDevice) != 0) return -1;
    return hbcu::frame_end_read(in, h->s_h2d);
}

int hbcu_comb_detect_run(hbcu_comb_detect_t *h, int64_t prev, int64_t cur, int64_t next, int force)
{
    if (h == nullptr || prev < 0 || cur < 0 || next < 0) { set_error("comb_detect_run: bad argument"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    const int64_t idx[3] = { prev, cur, next };
    const uint8_t *pl[3];
    for (int k = 0; k < 3; k++)
    {
        const int slot = (int)(idx[k] % h->slots);
        if (h->index[slot] != idx[k])
        {
            set_error("comb_detect_run: frame %lld is not resident", (long long)idx[k]);
            return -1;
        }
        HBCU_CHECK(cudaStreamWaitEvent(h->s_compute, h->ev_upload[slot], 0));
        pl[k] = h->luma[slot];
    }
    const int r = h->next_res;
    h->next_res = (h->next_res + 1) % h->nres;
    // the result slot is reused only after its previous verdict has been copied out (stream order)
    const hbcu_comb_detect_config_t &c = h->cfg;
    CombParams p;
    p.w = c.width; p.h = c.height; p.pitch = h->pitch;
    p.mode = c.mode; p.spatial_metric = c.spatial_metric; p.filter_mode = c.filter_mode;
    p.mthresh = c.motion_threshold; p.athresh = c.spatial_threshold;
    p.athresh_sq = c.spatial_threshold * c.spatial_threshold; p.athresh6 = 6 * c.spatial_threshold;
    p.c32min = c.comb32detect_min; p.c32max = c.comb32detect_max;
    p.g_mthresh = c.gamma_motion_threshold; p.g_athresh = c.gamma_spatial_threshold; p.g_athresh6 = c.gamma_spatial_threshold6;
    p.force = force;
    p.lut_size = 1 << c.depth;
    p.gamma_lut = h->d_lut;
    p.block_threshold = c.block_threshold; p.block_width = c.block_width; p.block_height = c.block_height;

    HBCU_CHECK(cudaMemsetAsync(h->d_flags + r, 0, sizeof(int), h->s_compute));
    // block grid: y = k*bh while y + bh <= height; x = j*bw while x < width - bw   (comb_detect.c:238-240)
    const int bw = c.block_width < c.width ? c.block_width : c.width;
    const int bh = c.block_height < c.height ? c.block_height : c.height;
    const int nby = c.height / bh;
    const int nbx = (c.width - bw + bw - 1) / bw;       // number of j with j*bw < width - bw
    const bool gamma = (c.mode & 1) != 0;
    const size_t lut_bytes = gamma ? (size_t)p.lut_size * sizeof(float) : 0;
    if (lut_bytes > 48 * 1024)
    {
        set_error("comb_detect: gamma table for depth %d does not fit shared memory", c.depth);
        return -1;
    }
    dim3 mgrid((h->nwords + 7) / 8, (c.height + kMaskRows - 1) / kMaskRows);
#define MASK(PIX, A, B, D)                                                                                                  \
    do {                                                                                                                    \
        if (gamma) comb_mask_bits2_kernel<PIX, true><<<mgrid, 256, lut_bytes, h->s_compute>>>(A, B, D, h->d_bits, h->wpitch, p); \
        else       comb_mask_bits2_kernel<PIX, false><<<mgrid, 256, 0, h->s_compute>>>(A, B, D, h->d_bits, h->wpitch, p);        \
    } while (0)
    if (h->bps == 1) MASK(uint8_t, pl[0], pl[1], pl[2]);
    else             MASK(uint16_t, (const uint16_t *)pl[0], (const uint16_t *)pl[1], (const uint16_t *)pl[2]);
#undef MASK
    hbcu::count_launch();
    HBCU_CHECK(cudaGetLastError());
    const bool filtered = (c.mode & 2) != 0;
    const uint32_t *scored = h->d_bits;
    if (filtered)
    {
        dim3 fgrid((h->nwords + BT_W - 1) / BT_W, (c.height + BT_R - 1) / BT_R);
        comb_filter_bits_kernel<<<fgrid, 256, 0, h->s_compute>>>(h->d_bits, h->d_fbits, h->wpitch, h->nwords, c.width, c.height, c.filter_mode);
        hbcu::count_launch();
        HBCU_CHECK(cudaGetLastError());
        scored = h->d_fbits;
    }
    if (nbx > 0 && nby > 0)
    {
        const int warps = nbx * nby;
        comb_score_bits_kernel<<<(warps * 32 + 127) / 128, 128, 0, h->s_compute>>>(scored, h->wpitch, c.width, c.height, bw, bh, nbx, nby,
                                                                                    c.block_threshold, filtered ? 1 : 0, h->d_flags + r);
        hbcu::count_launch();
        HBCU_CHECK(cudaGetLastError());
    }
    HBCU_CHECK(cudaMemcpyAsync(h->h_flags + r, h->d_flags + r, sizeof(int), cudaMemcpyDeviceToHost, h->s_compute));
    HBCU_CHECK(cudaEventRecord(h->ev_result[r], h->s_compute));
    h->res_index[r] = cur;
    // prev is never needed again once this run is done (the window moves forward)
    HBCU_CHECK(cudaEventRecord(h->ev_readers[(int)(prev % h->slots)], h->s_compute));
    return 0;
}

int hbcu_comb_detect_result(hbcu_comb_detect_t *h, int64_t cur, int *combed)
{
    if (h == nullptr || combed == nullptr) { set_error("comb_detect_result: bad argument"); return -1; }
    for (int r = 0; r < h->nres; r++)
    {
        if (h->res_index[r] == cur)
        {
            HBCU_CHECK(cudaEventSynchronize(h->ev_result[r]));
            const int f = h->h_flags[r];
            *combed = (f & 2) ? 2 : (f & 1) ? 1 : 0;     // check_combing_results, comb_detect.c:1029-1049
            return 0;
        }
    }
    set_error("comb_detect_result: no run pending for frame %lld", (long long)cur);
    return -1;
}

int hbcu_comb_detect_masks(hbcu_comb_detect_t *h, uint8_t *raw, uint8_t *scored)
{
    if (h == nullptr) { set_error("comb_detect_masks: null handle"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    HBCU_CHECK(cudaStreamSynchronize(h->s_compute));
    const size_t w = h->cfg.width, hh = h->cfg.height;
    dim3 blk(64, 4), grid(((int)w + 63) / 64, ((int)hh + 3) / 4);
    comb_unpack_bits_kernel<<<grid, blk, 0, h->s_compute>>>(h->d_bits, h->wpitch, h->d_mask, h->mpitch, (int)w, (int)hh);
    comb_unpack_bits_kernel<<<grid, blk, 0, h->s_compute>>>((h->cfg.mode & 2) ? h->d_fbits : h->d_bits, h->wpitch, h->d_scored, h->mpitch, (int)w, (int)hh);
    HBCU_CHECK(cudaStreamSynchronize(h->s_compute));
    if (raw) HBCU_CHECK(cudaMemcpy2D(raw, w, h->d_mask, h->mpitch, w, hh, cudaMemcpyDeviceToHost));
    if (scored) HBCU_CHECK(cudaMemcpy2D(scored, w, h->d_scored, h->mpitch, w, hh, cudaMemcpyDeviceToHost));
    return 0;
}

int hbcu_comb_detect_sync(hbcu_comb_detect_t *h)
{
    if (h == nullptr) { set_error("comb_detect_sync: null handle"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    HBCU_CHECK(cudaStreamSynchronize(h->s_h2d));
    HBCU_CHECK(cudaStreamSynchronize(h->s_compute));
    return 0;
}

int hbcu_comb_detect_mark(hbcu_comb_detect_t *h, int which)
{
    if (h == nullptr || which < 0 || which > 1) { set_error("comb_detect_mark: bad argument"); return -1; }
    HBCU_CHECK(cudaSetDevice(h->cfg.device));
    HBCU_CHECK(cudaEventRecord(h->ev_mark[which], h->s_compute));
    return 0;
}

int hbcu_comb_detect_elapsed_ms(hbcu_comb_detect_t *h, float *ms)
{
    if (h == nullptr || ms == nullptr) { set_error("comb_detect_elapsed_ms: bad argument"); return -1; }
    HBCU_CHECK(cudaEventSynchronize(h->ev_mark[1]));
    HBCU_CHECK(cudaEventElapsedTime(ms, h->ev_mark[0], h->ev_mark[1]));
    return 0;
}

}  // extern "C"
