// nlmeans_v3.cuh -- third generation of the fused 8-bit NLMeans tile kernel (included by nlmeans.cu).
//
// Same arithmetic contract as nlmeans_tiled_kernel (bit-identical to templates/nlmeans_template.c:593-717), same
// tiling idea (TMA tile in shared memory, a lane marches down a 4-pixel-wide column strip keeping the vertical running
// sum of horizontal patch-row sums and its N-row history in registers).  What changed, each item from the r01 ncu
// capture (profiles/r01g_nlmeans_fused_ncu.json: 29 thread-instructions per pixel x displacement, 68 % issue,
// ALU pipe 57 %, 35 % of the shared-memory wavefront budget):
//   * group shape (NG displacements), byte offset of the compare window and the origin slot are template parameters:
//     no per-row predicate/branch chains, and for the range-3 presets the three compare windows come straight out of
//     the raw words with 6 funnel shifts per row instead of 13 (the source window is never re-aligned: only the
//     relative alignment of source and compare matters to VABSDIFF4);
//   * the running sum V is kept as the integer 0x4B000000 + V: as a float that is 2^23 + V, so
//     fma.rn.sat(2^23 + V, wfact/128, -2^23 * wfact/128) = rn(V * wfact/128) exactly -- I2F and FMUL.SAT collapse into
//     one FFMA on the idle FMA pipe;
//   * the three-row delay line of compare words is indexed by the unrolled row slot instead of being shifted: no MOVs;
//   * warm-up rows are peeled: the steady-state loop has no "row >= NH" test;
//   * the compare tile of frame 1 is in flight while frame 0 is compared with itself (second mbarrier);
//   * accumulators (weight sum, pixel sum; 8 bytes per pixel) live in TENSOR MEMORY (tcgen05.ld/st, 32x32b.x8:
//     a lane's 4 x 2 floats are 8 columns of its own TMEM lane).  That takes their 16 wavefronts per row off the
//     shared-memory pipe and -- shared memory no longer bounds the tile -- lets a warp march 18-20 rows instead of 12:
//     the 2*NH warm-up rows drop from 50 % to 30-33 % of the patch-row-sum work.
#pragma once

template <int NW, int RS, int NBUF, int BPS = 1, bool PRE = false>
struct V3Layout
{
    static constexpr int kTH        = NW * RS;
    static constexpr int kLoads     = kTH + 2 * kHalo > 256 ? 2 : 1;                     // a TMA box has at most 256 rows
    static constexpr int kBoxRows   = ((kTH + 2 * kHalo + kLoads - 1) / kLoads + 3) / 4 * 4;   // 4 rows x 160 B keep every box 128-byte aligned
    static constexpr int kRows      = kBoxRows * kLoads;                                 // >= kTH + 2 * kHalo; surplus rows are loaded, never used
    static constexpr int kRowBytes  = kTilePW * BPS;
    static constexpr int kTileBytes = kRows * kRowBytes;
    static constexpr int kLutBytes  = kLutEntries * 32 * (int)sizeof(float);
    static constexpr int kOffCur    = 0;
    static constexpr int kOffCmp    = kOffCur + kTileBytes;
    // prefilter variant: the pre-denoised current tile and ONE pre-denoised compare tile (patch distances are taken from
    // these, pixel values from the plain tiles)
    static constexpr int kOffPre0   = kOffCmp + NBUF * kTileBytes;
    static constexpr int kOffCmpPre = kOffPre0 + (PRE ? kTileBytes : 0);
    static constexpr int kOffLut    = kOffCmpPre + (PRE ? kTileBytes : 0);
    static_assert(!PRE || NBUF == 1, "the prefilter variant keeps one compare buffer pair");
    static constexpr int kOffBar    = kOffLut + kLutBytes;                               // 1 + NBUF mbarriers, TMEM base word
    static constexpr int kUsed      = kOffBar + 64;
    // one CTA per SM by construction (the kernel allocates all 512 TMEM columns; a second resident CTA would spin)
    static constexpr int kTotal     = kUsed < 117 * 1024 ? 117 * 1024 : kUsed;
    static_assert(kBoxRows <= 256, "TMA box rows");
    static_assert((kBoxRows * kRowBytes) % 128 == 0, "TMA destination must stay 128-byte aligned");
    static_assert((NW + 3) / 4 * RS * 8 <= 512, "accumulators must fit 512 TMEM columns per lane quarter");
    static_assert(kTotal <= 227 * 1024, "shared memory");
};

// accumulator rows of one warp in tensor memory (8 columns per lane)
struct V3Acc
{
    uint32_t taddr;     // lane quarter of this warp (bits 31..16) + first column of its strip
    __device__ __forceinline__ void load(int r, uint32_t (&v)[8]) const
    {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                     : "r"(taddr + (uint32_t)r * 8u));
    }
    // the registers are tied to the wait so that no consumer is scheduled above it
    __device__ __forceinline__ void wait_load(uint32_t (&v)[8]) const
    {
        asm volatile("tcgen05.wait::ld.sync.aligned;"
                     : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]) :: "memory");
    }
    __device__ __forceinline__ void store(int r, const uint32_t (&v)[8]) const
    {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                     :: "r"(taddr + (uint32_t)r * 8u), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                     : "memory");
    }
    __device__ __forceinline__ void wait_store() const { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
};

// packed fp32 pairs (sm_100 add/mul.f32x2): each half is an IEEE round-to-nearest (or toward-zero) fp32 operation
__device__ __forceinline__ uint64_t v3_pack2(float a, float b)
{
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void v3_unpack2(uint64_t v, float &a, float &b)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ uint64_t v3_add2(uint64_t a, uint64_t b)
{
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t v3_add2_rz(uint64_t a, uint64_t b)
{
    uint64_t r;
    asm("add.rz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// product of two pairs of NON-NEGATIVE floats.  Written as fma(a, b, +0): ptxas contracts mul.rn.f32x2 + add.rn.f32x2
// into one FFMA2 even under -fmad=false (seen in the SASS; the reference rounds the product before it adds), and it
// cannot fold an explicit fma.  a * b + (+0) == rn(a * b) whenever the product is not -0, which weights and pixels never are.
__device__ __forceinline__ uint64_t v3_mul2(uint64_t a, uint64_t b)
{
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(0ull));
    return r;
}
// position of pixel i of a lane's four in the accumulator words (pairs (0, 2) and (1, 3))
__device__ __forceinline__ constexpr int v3_acc_slot(int i) { return (i & 1) * 2 + (i >> 1); }

constexpr int kOrgNone = -1;
constexpr uint32_t kVBias = 0x4B000000u;     // bits of 2^23

// One group of NG horizontally adjacent displacements (dy, dx0 .. dx0+NG-1) over `rows` output rows of this warp's strip.
//   OBS  : (12 + dx0) & 3, the byte offset of the compare window inside its first word
//   ORG  : slot of the origin displacement inside the group, or kOrgNone
// A struct so that the row step can be a function template of its unrolled slot K (every index into hist / P is a
// compile-time constant; everything is force-inlined and the arrays live in registers).
template <int NH, int NG, int OBS, int ORG, bool PRE, class ACC>
struct V3Group
{
    static constexpr int N      = 2 * NH + 1;
    static constexpr int PW     = kTilePW / 4;       // tile pitch in words
    static constexpr int FIRSTB = 4 - NH;            // the source stream starts 4 pixels left of the lane's first pixel:
    static constexpr int LASTB  = 7 + NH;            // the four windows cover its bytes FIRSTB .. LASTB
    static constexpr int NWA    = LASTB / 4 + 1;     // source words (3 for every patch size <= 9)
    static constexpr int LASTC  = LASTB + NG - 1;    // last compare-stream byte any displacement of the group touches
    static constexpr int NAL    = LASTC / 4 + 1;     // compare-stream words
    static constexpr int NRAW   = NAL + 1;           // raw words that cover them at any byte offset
    static_assert(NWA == 3, "patch size");

    uint32_t V[NG][4];
    uint32_t hist[N][NG][4];
    uint32_t P[PRE ? 1 : N][2];                      // compare-stream words 1 and 2 of the last rows: the averaged pixels
    const uint32_t *arow, *brow, *orow, *prow;       // (prefilter variant: re-read from the PLAIN compare tile instead)
    const ACC &acc;
    uint32_t lut_lane_addr;
    float wscale, wbias;
    double origin_tune;

    // srcp / cmpd: the tiles the patch distances are taken from (source, compare); cmpv: the compare tile whose pixels are
    // averaged; cur: the plain current tile (origin term).  Without a prefilter srcp == cur and cmpd == cmpv.
    __device__ __forceinline__ V3Group(const uint32_t *srcp, const uint32_t *cmpd, const uint32_t *cmpv, const uint32_t *cur, const ACC &acc_,
                                       uint32_t lut_lane_addr_, float wscale_, float wbias_, double origin_tune_, int seg_y0, int lane, int dy, int dx0)
        : acc(acc_), lut_lane_addr(lut_lane_addr_), wscale(wscale_), wbias(wbias_), origin_tune(origin_tune_)
    {
        const int s   = 12 + dx0;                    // tile byte (relative to 4 * lane) of compare-stream byte 0
        const int wb0 = s >> 2;
#pragma unroll
        for (int g = 0; g < NG; g++)
#pragma unroll
            for (int i = 0; i < 4; i++)
            {
                V[g][i] = kVBias;
#pragma unroll
                for (int k = 0; k < N; k++) hist[k][g][i] = 0;
            }
#pragma unroll
        for (int k = 0; k < (PRE ? 1 : N); k++) P[k][0] = P[k][1] = 0;
        arow = srcp + (seg_y0 - NH + kHalo) * PW + lane + 3;
        brow = cmpd + (seg_y0 - NH + kHalo + dy) * PW + lane + wb0;
        orow = cur + (seg_y0 + kHalo) * PW + lane + kHaloX / 4;
        prow = cmpv + (seg_y0 + kHalo + dy) * PW + lane + wb0 + 1;
    }

    static __device__ __forceinline__ bool is_origin(int g) { return ORG >= 0 && g == ORG; }

    // one row step in unrolled slot K; OUT: the row NH above completes and is averaged into accumulator row r
    template <int K, bool OUT>
    __device__ __forceinline__ void step(int r)
    {
        uint32_t a[NWA], raw[NRAW], bg0[NAL];
#pragma unroll
        for (int j = 0; j < NWA; j++) a[j] = arow[j];
#pragma unroll
        for (int j = 0; j < NRAW; j++) raw[j] = brow[j];
        arow += PW;
        brow += PW;
        uint32_t accv[8];
        if (OUT) acc.load(r, accv);
        // compare stream aligned for displacement 0 of the group
#pragma unroll
        for (int j = 0; j < NAL; j++) bg0[j] = OBS == 0 ? raw[j] : __funnelshift_r(raw[j], raw[j + 1], 8 * OBS);
#pragma unroll
        for (int g = 0; g < NG; g++)
        {
            if (ORG != kOrgNone && is_origin(g)) continue;
            uint32_t D[NWA];
#pragma unroll
            for (int w = 0; w < NWA; w++)
            {
                uint32_t bw;
                if (g == 0) bw = bg0[w];
                else
                {
                    const int sh = (OBS + g) & 3, q = (OBS + g) >> 2;       // compile-time after unrolling
                    const int j1 = w + q + 1 < NRAW ? w + q + 1 : NRAW - 1;
                    bw = sh ? __funnelshift_r(raw[w + q], raw[j1], 8 * sh) : raw[w + q];
                }
                D[w] = __vabsdiffu4(a[w], bw);
            }
            if constexpr (NH == 3)
            {
                // patch 7: the windows are bytes 1+i .. 7+i of the D stream = word 1 (bytes 4..7, shared) plus exactly
                // three more bytes.  Byte 0 of the stream belongs to no window: cleared, it is the zero that pads those
                // three bytes (gathered by PRMT from words 0 and 2) to a word, so every window is IDP4A(X, X, T1).
                const uint32_t T1 = __dp4a(D[1], D[1], 0u);
                const uint32_t Z  = D[0] & 0xFFFFFF00u;
                uint32_t X[4];
                X[0] = Z;                                   // bytes 1, 2, 3
                X[1] = __byte_perm(Z, D[2], 0x0432);        // bytes 2, 3, 8
                X[2] = __byte_perm(Z, D[2], 0x0543);        // bytes 3, 8, 9
                X[3] = __byte_perm(Z, D[2], 0x0654);        // bytes 8, 9, 10
#pragma unroll
                for (int i = 0; i < 4; i++)
                {
                    const uint32_t hs = __dp4a(X[i], X[i], T1);
                    V[g][i] = V[g][i] + hs - hist[K][g][i];
                    hist[K][g][i] = hs;
                }
            }
            else
            {
            // patch-row sums over bytes FIRSTB+i .. FIRSTB+i+N-1 of the D stream: whole words by IDP4A(D, D), partial
            // words by IDP4A(D & mask, D); the first whole word is shared by the four windows
            uint32_t T[NWA];
#pragma unroll
            for (int w = 0; w < NWA; w++) T[w] = __dp4a(D[w], D[w], 0u);
#pragma unroll
            for (int i = 0; i < 4; i++)
            {
                const int b0 = FIRSTB + i, b1 = FIRSTB + i + N - 1;
                uint32_t hs = 0;
                bool started = false;
#pragma unroll
                for (int w = 0; w < NWA; w++)
                {
                    const int lo = b0 > 4 * w ? b0 : 4 * w, hi = b1 < 4 * w + 3 ? b1 : 4 * w + 3;
                    if (lo == 4 * w && hi == 4 * w + 3 && !started) { hs = T[w]; started = true; }
                }
                bool used_full = false;
#pragma unroll
                for (int w = 0; w < NWA; w++)
                {
                    const int lo = b0 > 4 * w ? b0 : 4 * w, hi = b1 < 4 * w + 3 ? b1 : 4 * w + 3;
                    if (lo > hi) continue;
                    if (lo == 4 * w && hi == 4 * w + 3)
                    {
                        if (started && !used_full) { used_full = true; continue; }   // already in hs
                        hs = __dp4a(D[w], D[w], hs);
                    }
                    else
                    {
                        uint32_t m = 0;
#pragma unroll
                        for (int bb = 0; bb < 4; bb++)
                            if (4 * w + bb >= lo && 4 * w + bb <= hi) m |= 0xFFu << (8 * bb);
                        hs = __dp4a(D[w] & m, D[w], hs);
                    }
                }
                V[g][i] = V[g][i] + hs - hist[K][g][i];
                hist[K][g][i] = hs;
            }
            }
        }
        if (OUT)
        {
            constexpr int KP = PRE ? 0 : (K + N - NH) % N;   // the compare row of the output row was loaded NH steps ago
            uint32_t p0, p1;
            if constexpr (PRE)
            {
                const uint32_t q0 = prow[r * PW], q1 = prow[r * PW + 1], q2 = prow[r * PW + 2];
                p0 = OBS == 0 ? q0 : __funnelshift_r(q0, q1, 8 * OBS);
                p1 = OBS == 0 ? q1 : __funnelshift_r(q1, q2, 8 * OBS);
            }
            else
            {
                p0 = P[KP][0];
                p1 = P[KP][1];
            }
            // pixels 0/2 and 1/3 of the lane's four travel as packed pairs (add/mul.rn.f32x2: two IEEE fp32 operations per
            // issue slot, same rounding as the scalar instructions); accumulator words are stored in that order:
            // {ws0, ws2, ws1, ws3, ps0, ps2, ps1, ps3}
            uint64_t pix2[NG + 1];                        // (compare pixel j, compare pixel j + 2) as floats
#pragma unroll
            for (int j = 0; j < NG + 1; j++)
                pix2[j] = v3_add2(v3_pack2(byte_as_biased_float(j < 4 ? p0 : p1, j & 3), byte_as_biased_float(j + 2 < 4 ? p0 : p1, (j + 2) & 3)),
                                  v3_pack2(-8388608.0f, -8388608.0f));
            acc.wait_load(accv);                          // issued at the top of the step: the patch-row sums covered its latency
            uint64_t W[NG][2];                            // weights of pixels (0, 2) and (1, 3)
#pragma unroll
            for (int g = 0; g < NG; g++)
            {
                if (ORG != kOrgNone && is_origin(g)) continue;
                float t[4];
#pragma unroll
                for (int i = 0; i < 4; i++)
                    asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(t[i]) : "f"(__uint_as_float(V[g][i])), "f"(wscale), "f"(wbias));
#pragma unroll
                for (int h = 0; h < 2; h++)
                {
                    float u0, u1, w0, w1;
                    v3_unpack2(v3_add2_rz(v3_pack2(t[h], t[h + 2]), v3_pack2(65536.0f, 65536.0f)), u0, u1);   // 65536 + floor(128 t)
                    asm("ld.shared.f32 %0, [%1];" : "=f"(w0) : "r"((__float_as_uint(u0) << 7) + lut_lane_addr));
                    asm("ld.shared.f32 %0, [%1];" : "=f"(w1) : "r"((__float_as_uint(u1) << 7) + lut_lane_addr));
                    W[g][h] = v3_pack2(w0, w1);
                }
            }
            uint64_t ws2[2], ps2[2];
#pragma unroll
            for (int h = 0; h < 2; h++)
            {
                ws2[h] = v3_pack2(__uint_as_float(accv[2 * h]), __uint_as_float(accv[2 * h + 1]));
                ps2[h] = v3_pack2(__uint_as_float(accv[4 + 2 * h]), __uint_as_float(accv[4 + 2 * h + 1]));
            }
#pragma unroll
            for (int g = 0; g < NG; g++)
            {
                if (ORG != kOrgNone && is_origin(g))
                {
                    const uint32_t cw = orow[r * PW];
#pragma unroll
                    for (int h = 0; h < 2; h++)
                    {
                        float wa, wb, pa, pb;
                        v3_unpack2(ws2[h], wa, wb);
                        v3_unpack2(ps2[h], pa, pb);
                        add_origin(wa, pa, origin_tune, (int)((cw >> (8 * h)) & 0xffu));
                        add_origin(wb, pb, origin_tune, (int)((cw >> (8 * (h + 2))) & 0xffu));
                        ws2[h] = v3_pack2(wa, wb);
                        ps2[h] = v3_pack2(pa, pb);
                    }
                }
                else
                {
#pragma unroll
                    for (int h = 0; h < 2; h++)
                    {
                        ws2[h] = v3_add2(ws2[h], W[g][h]);
                        ps2[h] = v3_add2(ps2[h], v3_mul2(W[g][h], pix2[g + h]));
                    }
                }
            }
#pragma unroll
            for (int h = 0; h < 2; h++)
            {
                float a, b;
                v3_unpack2(ws2[h], a, b);
                accv[2 * h] = __float_as_uint(a); accv[2 * h + 1] = __float_as_uint(b);
                v3_unpack2(ps2[h], a, b);
                accv[4 + 2 * h] = __float_as_uint(a); accv[4 + 2 * h + 1] = __float_as_uint(b);
            }
            acc.store(r, accv);
        }
        if constexpr (!PRE)
        {
            P[K][0] = bg0[1];
            P[K][1] = bg0[2];
        }
    }

    template <int... Ks>
    __device__ __forceinline__ void warm_up(std::integer_sequence<int, Ks...>)
    {
        (step<Ks, false>(0), ...);
    }
    template <int... Ms>
    __device__ __forceinline__ void rows_from(int r0, int rows, std::integer_sequence<int, Ms...>)
    {
        ((r0 + Ms < rows ? step<(2 * NH + Ms) % N, true>(r0 + Ms) : (void)0), ...);
    }
    template <int... Ms>
    __device__ __forceinline__ void batch(int r0, std::integer_sequence<int, Ms...>)
    {
        (step<(2 * NH + Ms) % N, true>(r0 + Ms), ...);
    }

    // EXACT: `rows` is a multiple of N -- batches of N rows without a per-row test (and without the register moves the
    // merge points of those tests cost)
    template <bool EXACT>
    __device__ __forceinline__ void run(int rows)
    {
        // warm-up: the first 2*NH rows only build patch-row sums (slots 0 .. 2NH-1);
        // steady state: output row r completes at row step r + 2NH, slot (r + 2NH) % N
        warm_up(std::make_integer_sequence<int, 2 * NH>{});
        if (EXACT)
        {
#pragma unroll 1
            for (int r0 = 0; r0 < rows; r0 += N) batch(r0, std::make_integer_sequence<int, N>{});
        }
        else
        {
#pragma unroll 1
            for (int r0 = 0; r0 < rows; r0 += N) rows_from(r0, rows, std::make_integer_sequence<int, N>{});
        }
        acc.wait_store();
    }
};

template <int NH, int NG, int OBS, int ORG, bool EXACT, bool PRE, class ACC>
__device__ __forceinline__ void v3_group(const uint32_t *__restrict__ srcp, const uint32_t *__restrict__ cmpd, const uint32_t *__restrict__ cmpv,
                                         const uint32_t *__restrict__ cur, const ACC &acc,
                                         uint32_t lut_lane_addr, float wscale, float wbias, double origin_tune,
                                         int seg_y0, int rows, int lane, int dy, int dx0)
{
    V3Group<NH, NG, OBS, ORG, PRE, ACC> g(srcp, cmpd, cmpv, cur, acc, lut_lane_addr, wscale, wbias, origin_tune, seg_y0, lane, dy, dx0);
    g.template run<EXACT>(rows);
}

// Group shapes a displacement row can be cut into (three displacements per group, the remainder last), keyed by
// {displacements, (12 + dx0) & 3, origin slot}.  Every range 3 .. 15 decomposes into these eleven (v3_group_known()).
#define V3_GROUP_SHAPES(X) \
    X(3, 0, kOrgNone) X(3, 1, kOrgNone) X(3, 2, kOrgNone) X(3, 3, kOrgNone) \
    X(3, 3, 1) X(3, 2, 2) X(3, 0, 0) \
    X(2, 1, kOrgNone) X(2, 0, kOrgNone) X(1, 3, kOrgNone) X(1, 2, kOrgNone)

__host__ __device__ inline bool v3_group_known(int ng, int ob, int org)
{
#define X(NG_, OB_, ORG_) if (ng == NG_ && ob == OB_ && org == ORG_) return true;
    V3_GROUP_SHAPES(X)
#undef X
    return false;
}

template <int NH, int NW, int RS, int NBUF, bool PRE = false>
__global__ void __launch_bounds__(NW * 32, 1) nlmeans_v3_kernel(const __grid_constant__ FusedParams fp)
{
    constexpr int kThreads = NW * 32;
    using L = V3Layout<NW, RS, NBUF, 1, PRE>;
    int pl = 0;
    while (pl + 1 < fp.nplanes && (int)blockIdx.x >= fp.first_tile[pl + 1]) pl++;
    const KernelParams &p = fp.k[pl];
    const CUtensorMap *maps = fp.maps[pl];
    const CUtensorMap *maps_pre = fp.maps_pre[pl];       // prefilter variant only
    const int tile = (int)blockIdx.x - fp.first_tile[pl];
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *cur  = smem + L::kOffCur;
    float *lut    = reinterpret_cast<float *>(smem + L::kOffLut);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + L::kOffBar);           // [0] current tile, [1 + b] compare buffer b
    uint32_t *tmem_base_slot = reinterpret_cast<uint32_t *>(smem + L::kOffBar + 8 * (1 + NBUF));

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int X0 = (tile % fp.tiles_x[pl]) * kTileW, Y0 = (tile / fp.tiles_x[pl]) * L::kTH;
    const int gx = X0 + kBorder - kHaloX, gy = Y0 + kBorder - kHalo;

    if (tid == 0)
    {
        for (int b = 0; b < 1 + NBUF; b++) mbar_init(bar + b, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    if (warp == 0)
    {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" :: "r"(smem_u32(tmem_base_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (tid == 0)
    {
        mbar_expect_tx(bar, L::kTileBytes * (PRE ? 2 : 1));
        for (int l = 0; l < L::kLoads; l++) tma_load_2d(cur + l * L::kBoxRows * kTilePW, &maps[0], gx, gy + l * L::kBoxRows, bar);
        if (PRE)
            for (int l = 0; l < L::kLoads; l++) tma_load_2d(smem + L::kOffPre0 + l * L::kBoxRows * kTilePW, &maps_pre[0], gx, gy + l * L::kBoxRows, bar);
        // frame 0 is compared with itself: the compare buffers are free, fill them with the following frames now
        for (int b = 0; b < NBUF && 1 + b < p.nf; b++)
        {
            mbar_expect_tx(bar + 1 + b, L::kTileBytes * (PRE ? 2 : 1));
            for (int l = 0; l < L::kLoads; l++)
                tma_load_2d(smem + L::kOffCmp + b * L::kTileBytes + l * L::kBoxRows * kTilePW, &maps[1 + b], gx, gy + l * L::kBoxRows, bar + 1 + b);
            if (PRE)
                for (int l = 0; l < L::kLoads; l++)
                    tma_load_2d(smem + L::kOffCmpPre + l * L::kBoxRows * kTilePW, &maps_pre[1 + b], gx, gy + l * L::kBoxRows, bar + 1 + b);
        }
    }
    for (int i = tid; i < kLutEntries * 32; i += kThreads)
    {
        const int e = i >> 5;
        lut[i] = e < HBCU_NLMEANS_EXPSIZE ? p.exptable[e] : 0.f;
    }

    const int seg_y0 = warp * RS;
    int rows = p.h - (Y0 + seg_y0);                                     // rows of this warp's strip inside the plane
    rows = rows < 0 ? 0 : (rows > RS ? RS : rows);
    V3Acc acc;
    acc.taddr = *tmem_base_slot + ((uint32_t)(warp & 3) << 21) + (uint32_t)((warp >> 2) * RS * 8);   // lane 32 * (warp % 4) in bits 31..16
    uint32_t z[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
    for (int r = 0; r < RS; r++) acc.store(r, z);
    acc.wait_store();
    mbar_wait(bar, 0);
    __syncthreads();

    const float wscale = p.wfact * 0.0078125f;                         // wfact / 128, exact
    const float wbias  = -8388608.0f * wscale;                         // exact (power-of-two scaling)
    // shared address of this lane's copy of table entry 0, pre-biased by -(0x47800000 << 7)
    const uint32_t lut_lane_addr = smem_u32(lut) + (uint32_t)lane * 4u - (0x47800000u << 7);
    const uint32_t *cw = reinterpret_cast<const uint32_t *>(cur);
    const uint32_t *pre0w = reinterpret_cast<const uint32_t *>(smem + L::kOffPre0);
    // the source patches: the pre-denoised current tile -- or the plain one where the reference's pointer is stale
    // (KernelParams::src_pre, the first frame of a stream)
    const uint32_t *srcw = (PRE && p.src_pre != p.planes[0]) ? pre0w : cw;
    for (int f = 0; f < p.nf; f++)
    {
        const uint32_t *bw = cw;
        const int buf = (f - 1) % NBUF;
        if (f > 0)
        {
            mbar_wait(bar + 1 + buf, (uint32_t)(((f - 1) / NBUF) & 1));
            bw = reinterpret_cast<const uint32_t *>(smem + L::kOffCmp + buf * L::kTileBytes);
        }
        // the tile the patch distances compare against: the pre-denoised twin of `bw` in the prefilter variant
        const uint32_t *bd = !PRE ? bw : (f == 0 ? pre0w : reinterpret_cast<const uint32_t *>(smem + L::kOffCmpPre));
        if (rows > 0)
        {
            constexpr bool kExact = RS % (2 * NH + 1) == 0;             // then partial strips run to their end (rows beyond the plane are never stored)
            const int nrows = kExact ? RS : rows;
            for (int dy = -p.r_half; dy <= p.r_half; dy++)
            {
                for (int dx0 = -p.r_half; dx0 <= p.r_half; dx0 += kGroup)
                {
                    const int ng  = min(kGroup, p.r_half - dx0 + 1);
                    const int org = (f == 0 && dy == 0 && dx0 <= 0 && dx0 + ng > 0) ? -dx0 : kOrgNone;
                    const int ob  = (12 + dx0) & 3;
#define X(NG_, OB_, ORG_)                                                                                                   \
                    if (ng == NG_ && ob == OB_ && org == ORG_)                                                              \
                        v3_group<NH, NG_, OB_, ORG_, kExact, PRE>(srcw, bd, bw, cw, acc, lut_lane_addr, wscale, wbias, p.origin_tune, seg_y0, nrows, lane, dy, dx0); \
                    else
                    V3_GROUP_SHAPES(X)
#undef X
                    { /* unreachable: the launcher checked v3_group_known() for every group of this range */ }
                }
            }
        }
        // the buffer just read takes frame f + NBUF (uniform condition: every warp reaches the barrier)
        if (f > 0 && f + NBUF < p.nf)
        {
            __syncthreads();
            if (tid == 0)
            {
                fence_proxy_async();
                mbar_expect_tx(bar + 1 + buf, L::kTileBytes * (PRE ? 2 : 1));
                for (int l = 0; l < L::kLoads; l++)
                    tma_load_2d(smem + L::kOffCmp + buf * L::kTileBytes + l * L::kBoxRows * kTilePW, &maps[f + NBUF], gx, gy + l * L::kBoxRows, bar + 1 + buf);
                if (PRE)
                    for (int l = 0; l < L::kLoads; l++)
                        tma_load_2d(smem + L::kOffCmpPre + l * L::kBoxRows * kTilePW, &maps_pre[f + NBUF], gx, gy + l * L::kBoxRows, bar + 1 + buf);
            }
        }
    }

    const int x = lane * 4;
    uint8_t *dst = reinterpret_cast<uint8_t *>(p.dst);
    for (int r = 0; r < rows; r++)
    {
        const int oy = seg_y0 + r;
        const int y = Y0 + oy;
        uint32_t accv[8];
        acc.load(r, accv);
        acc.wait_load(accv);
        const uint32_t cwd = cw[(oy + kHalo) * (kTilePW / 4) + lane + kHaloX / 4];
        uint8_t o[4];
#pragma unroll
        for (int i = 0; i < 4; i++)
            o[i] = finish_pixel<uint8_t>(__uint_as_float(accv[v3_acc_slot(i)]), __uint_as_float(accv[4 + v3_acc_slot(i)]), (uint8_t)((cwd >> (8 * i)) & 0xffu));
        uint8_t *drow = dst + (size_t)y * p.dpitch + X0 + x;
        if (X0 + x + 3 < p.w)
            *reinterpret_cast<uchar4 *>(drow) = make_uchar4(o[0], o[1], o[2], o[3]);
        else
        {
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (X0 + x + i < p.w) drow[i] = o[i];
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
    {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" :: "r"(*tmem_base_slot) : "memory");
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// 16-bit samples (yuv420p10 planes; every sample <= kMax10Bit = 1023).  A 16-bit container can hold samples above
// 1023.  The border kernel raises a sticky flag when it sees one; this kernel then returns at once and the integer
// kernel launched right behind it (which returns at once when the flag is clear) does the frame: same output either
// way, no host round trip.
//
// Same march as the 8-bit group: a lane owns 4 adjacent pixels and walks down its strip with the vertical running sum V
// of horizontal patch-row sums in registers.  The squared differences have no packed-integer instruction at this width;
// they are fp32 integers instead -- every value stays below 2^24, so every add/fma is exact in ANY order, which frees the
// grouping: the four windows of a row share their middle (27 fp32 operations per displacement and row instead of a
// 10-long prefix chain plus window differences; packing two displacements into f32x2 pairs was costed and dropped -- the
// operand pairs cost as many PRMTs as the packed arithmetic saves).  V is a plain integer here
// (49 x 1023^2 does not fit the 2^23-biased-float trick of the 8-bit kernel): I2FP + FMUL.SAT.
// The compare pixels of the output row are re-read from shared memory (no 7-row delay line of words in registers).
template <int NH, int NG, int OB, int ORG, class ACC>
struct V3Group16
{
    static constexpr int N    = 2 * NH + 1;
    static constexpr int PW   = kTilePW / 2;          // tile pitch in words (two samples each)
    static constexpr int NA   = 4 + 2 * NH;           // source samples per row
    static constexpr int NB   = NA + NG - 1;          // compare samples per row
    static constexpr int OA   = (kHaloX - NH) & 3;    // sample offset of a[0] inside its first quad
    static constexpr int FB   = (OB - NH) & 3;        // sample offset of b[0] inside its first quad (OB = (12 + dx0) & 3)
    static constexpr int NWA  = (OA + NA + 1) / 2;    // words covering the source window
    static constexpr int NWB  = (FB + NB + 1) / 2;
    static constexpr int OP   = OB & 3;               // the output row's compare pixels start at sample kHaloX + dx0 of the row
    static constexpr int NWP  = (OP + NG + 3 + 1) / 2;
    static constexpr float kBias = 8388608.0f;
    static_assert(NH >= 1 && NH <= 3, "patch-row sums must stay below 2^23");

    int      V[NG][4];
    uint32_t hist[N][NG][4];                          // patch-row sums as bits of (2^23 + sum): the biases cancel in V
    const uint32_t *arow, *brow, *prow, *orow;
    const ACC &acc;
    uint32_t lut_lane_addr;
    float wscale;
    double origin_tune;

    __device__ __forceinline__ V3Group16(const uint32_t *cur, const uint32_t *cmp, const ACC &acc_, uint32_t lut_lane_addr_, float wscale_,
                                         double origin_tune_, int seg_y0, int lane, int dy, int dx0)
        : acc(acc_), lut_lane_addr(lut_lane_addr_), wscale(wscale_), origin_tune(origin_tune_)
    {
#pragma unroll
        for (int g = 0; g < NG; g++)
#pragma unroll
            for (int i = 0; i < 4; i++)
            {
                V[g][i] = 0;
#pragma unroll
                for (int k = 0; k < N; k++) hist[k][g][i] = kVBias;
            }
        const int fa = kHaloX - NH, fb = kHaloX - NH + dx0, fp = kHaloX + dx0;      // first sample of each window, relative to 4 * lane
        arow = cur + (seg_y0 - NH + kHalo) * PW + 2 * lane + 2 * (fa >> 2);
        brow = cmp + (seg_y0 - NH + kHalo + dy) * PW + 2 * lane + 2 * (fb >> 2);
        prow = cmp + (seg_y0 + kHalo + dy) * PW + 2 * lane + 2 * (fp >> 2);
        orow = cur + (seg_y0 + kHalo) * PW + 2 * lane + kHaloX / 2;
    }

    static __device__ __forceinline__ bool is_origin(int g) { return ORG >= 0 && g == ORG; }

    template <int K, bool OUT>
    __device__ __forceinline__ void step(int r)
    {
        uint32_t wa[NWA], wb[NWB];
#pragma unroll
        for (int j = 0; j < NWA; j++) wa[j] = arow[j];
#pragma unroll
        for (int j = 0; j < NWB; j++) wb[j] = brow[j];
        arow += PW;
        brow += PW;
        uint32_t accv[8];
        if (OUT) acc.load(r, accv);
        float a[NA], b[NB];
#pragma unroll
        for (int j = 0; j < NA; j++) a[j] = half_as_biased_float(wa[(OA + j) >> 1], (OA + j) & 1);
#pragma unroll
        for (int j = 0; j < NB; j++) b[j] = half_as_biased_float(wb[(FB + j) >> 1], (FB + j) & 1);

        // hs[i] = sum of d^2 over samples i .. i + 2NH of the row = the common middle M (samples 3 .. 2NH, carrying the
        // 2^23 bias of the stored sums) + L[i] (samples i .. 2, i <= 2) + R[i - 1] (samples 2NH+1 .. 2NH+i, i >= 1).
        // Every value is an integer below 2^24: all of it is exact in any order.
#pragma unroll
        for (int g = 0; g < NG; g++)
        {
            if (ORG != kOrgNone && is_origin(g)) continue;
            float d[NA];
#pragma unroll
            for (int j = 0; j < NA; j++) d[j] = __fsub_rn(a[j], b[j + g]);          // exact: both are 2^23 + sample
            float M = kBias;
#pragma unroll
            for (int j = 3; j <= 2 * NH; j++) M = __fmaf_rn(d[j], d[j], M);
            float L[3], R[3];
            L[2] = __fmul_rn(d[2], d[2]);
            L[1] = __fmaf_rn(d[1], d[1], L[2]);
            L[0] = __fmaf_rn(d[0], d[0], L[1]);
            R[0] = __fmul_rn(d[2 * NH + 1], d[2 * NH + 1]);
            R[1] = __fmaf_rn(d[2 * NH + 2], d[2 * NH + 2], R[0]);
            R[2] = __fmaf_rn(d[2 * NH + 3], d[2 * NH + 3], R[1]);
#pragma unroll
            for (int i = 0; i < 4; i++)
            {
                float h = M;
                if (i <= 2) h = __fadd_rn(h, L[i]);
                if (i >= 1) h = __fadd_rn(h, R[i - 1]);
                const uint32_t hb = __float_as_uint(h);
                V[g][i] = V[g][i] + (int)hb - (int)hist[K][g][i];
                hist[K][g][i] = hb;
            }
        }
        if (OUT)
        {
            uint32_t wp[NWP];
#pragma unroll
            for (int j = 0; j < NWP; j++) wp[j] = prow[r * PW + j];
            uint64_t pix2[NG + 1];                        // (compare pixel j, compare pixel j + 2) as floats
#pragma unroll
            for (int j = 0; j < NG + 1; j++)
                pix2[j] = v3_add2(v3_pack2(half_as_biased_float(wp[(OP + j) >> 1], (OP + j) & 1),
                                           half_as_biased_float(wp[(OP + j + 2) >> 1], (OP + j + 2) & 1)),
                                  v3_pack2(-kBias, -kBias));
            acc.wait_load(accv);
            uint64_t W[NG][2];
#pragma unroll
            for (int g = 0; g < NG; g++)
            {
                if (ORG != kOrgNone && is_origin(g)) continue;
                float t[4];
#pragma unroll
                for (int i = 0; i < 4; i++)
                    asm("mul.rn.sat.f32 %0, %1, %2;" : "=f"(t[i]) : "f"(__int2float_rn(V[g][i])), "f"(wscale));
#pragma unroll
                for (int h = 0; h < 2; h++)
                {
                    float u0, u1, w0, w1;
                    v3_unpack2(v3_add2_rz(v3_pack2(t[h], t[h + 2]), v3_pack2(65536.0f, 65536.0f)), u0, u1);
                    asm("ld.shared.f32 %0, [%1];" : "=f"(w0) : "r"((__float_as_uint(u0) << 7) + lut_lane_addr));
                    asm("ld.shared.f32 %0, [%1];" : "=f"(w1) : "r"((__float_as_uint(u1) << 7) + lut_lane_addr));
                    W[g][h] = v3_pack2(w0, w1);
                }
            }
            uint64_t ws2[2], ps2[2];
#pragma unroll
            for (int h = 0; h < 2; h++)
            {
                ws2[h] = v3_pack2(__uint_as_float(accv[2 * h]), __uint_as_float(accv[2 * h + 1]));
                ps2[h] = v3_pack2(__uint_as_float(accv[4 + 2 * h]), __uint_as_float(accv[4 + 2 * h + 1]));
            }
#pragma unroll
            for (int g = 0; g < NG; g++)
            {
                if (ORG != kOrgNone && is_origin(g))
                {
                    const uint32_t c0 = orow[r * PW], c1 = orow[r * PW + 1];
#pragma unroll
                    for (int h = 0; h < 2; h++)
                    {
                        float wa_, wb_, pa, pb;
                        v3_unpack2(ws2[h], wa_, wb_);
                        v3_unpack2(ps2[h], pa, pb);
                        add_origin(wa_, pa, origin_tune, (int)((c0 >> (16 * h)) & 0xffffu));      // pixel h
                        add_origin(wb_, pb, origin_tune, (int)((c1 >> (16 * h)) & 0xffffu));      // pixel h + 2
                        ws2[h] = v3_pack2(wa_, wb_);
                        ps2[h] = v3_pack2(pa, pb);
                    }
                }
                else
                {
#pragma unroll
                    for (int h = 0; h < 2; h++)
                    {
                        ws2[h] = v3_add2(ws2[h], W[g][h]);
                        ps2[h] = v3_add2(ps2[h], v3_mul2(W[g][h], pix2[g + h]));
                    }
                }
            }
#pragma unroll
            for (int h = 0; h < 2; h++)
            {
                float x, y;
                v3_unpack2(ws2[h], x, y);
                accv[2 * h] = __float_as_uint(x); accv[2 * h + 1] = __float_as_uint(y);
                v3_unpack2(ps2[h], x, y);
                accv[4 + 2 * h] = __float_as_uint(x); accv[4 + 2 * h + 1] = __float_as_uint(y);
            }
            acc.store(r, accv);
        }
    }

    template <int... Ks>
    __device__ __forceinline__ void warm_up(std::integer_sequence<int, Ks...>) { (step<Ks, false>(0), ...); }
    template <int... Ms>
    __device__ __forceinline__ void rows_from(int r0, int rows, std::integer_sequence<int, Ms...>)
    {
        ((r0 + Ms < rows ? step<(2 * NH + Ms) % N, true>(r0 + Ms) : (void)0), ...);
    }
    __device__ __forceinline__ void run(int rows)
    {
        warm_up(std::make_integer_sequence<int, 2 * NH>{});
#pragma unroll 1
        for (int r0 = 0; r0 < rows; r0 += N) rows_from(r0, rows, std::make_integer_sequence<int, N>{});
        acc.wait_store();
    }
};

template <int NH, int NG, int OB, int ORG, class ACC>
__device__ __forceinline__ void v3_group16(const uint32_t *__restrict__ cur, const uint32_t *__restrict__ cmp, const ACC &acc,
                                           uint32_t lut_lane_addr, float wscale, double origin_tune,
                                           int seg_y0, int rows, int lane, int dy, int dx0)
{
    V3Group16<NH, NG, OB, ORG, ACC> g(cur, cmp, acc, lut_lane_addr, wscale, origin_tune, seg_y0, lane, dy, dx0);
    g.run(rows);
}

template <int NH, int NW, int RS, int NBUF>
__global__ void __launch_bounds__(NW * 32, 1) nlmeans_v3w_kernel(const __grid_constant__ FusedParams fp)
{
    if (*fp.range_flag != 0u) return;               // samples above 10 bit seen: the integer kernel takes over
    constexpr int kThreads = NW * 32;
    using L = V3Layout<NW, RS, NBUF, 2>;
    int pl = 0;
    while (pl + 1 < fp.nplanes && (int)blockIdx.x >= fp.first_tile[pl + 1]) pl++;
    const KernelParams &p = fp.k[pl];
    const CUtensorMap *maps = fp.maps[pl];
    const int tile = (int)blockIdx.x - fp.first_tile[pl];
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *cur  = smem + L::kOffCur;
    float *lut    = reinterpret_cast<float *>(smem + L::kOffLut);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + L::kOffBar);
    uint32_t *tmem_base_slot = reinterpret_cast<uint32_t *>(smem + L::kOffBar + 8 * (1 + NBUF));

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int X0 = (tile % fp.tiles_x[pl]) * kTileW, Y0 = (tile / fp.tiles_x[pl]) * L::kTH;
    const int gx = X0 + kBorder - kHaloX, gy = Y0 + kBorder - kHalo;

    if (tid == 0)
    {
        for (int b = 0; b < 1 + NBUF; b++) mbar_init(bar + b, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    if (warp == 0)
    {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" :: "r"(smem_u32(tmem_base_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (tid == 0)
    {
        mbar_expect_tx(bar, L::kTileBytes);
        for (int l = 0; l < L::kLoads; l++) tma_load_2d(cur + l * L::kBoxRows * L::kRowBytes, &maps[0], gx, gy + l * L::kBoxRows, bar);
        for (int b = 0; b < NBUF && 1 + b < p.nf; b++)
        {
            mbar_expect_tx(bar + 1 + b, L::kTileBytes);
            for (int l = 0; l < L::kLoads; l++)
                tma_load_2d(smem + L::kOffCmp + b * L::kTileBytes + l * L::kBoxRows * L::kRowBytes, &maps[1 + b], gx, gy + l * L::kBoxRows, bar + 1 + b);
        }
    }
    for (int i = tid; i < kLutEntries * 32; i += kThreads)
    {
        const int e = i >> 5;
        lut[i] = e < HBCU_NLMEANS_EXPSIZE ? p.exptable[e] : 0.f;
    }

    const int seg_y0 = warp * RS;
    int rows = p.h - (Y0 + seg_y0);
    rows = rows < 0 ? 0 : (rows > RS ? RS : rows);
    V3Acc acc;
    acc.taddr = *tmem_base_slot + ((uint32_t)(warp & 3) << 21) + (uint32_t)((warp >> 2) * RS * 8);
    uint32_t z[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
    for (int r = 0; r < RS; r++) acc.store(r, z);
    acc.wait_store();
    mbar_wait(bar, 0);
    __syncthreads();

    const float wscale = p.wfact * 0.0078125f;                         // wfact / 128, exact
    const uint32_t lut_lane_addr = smem_u32(lut) + (uint32_t)lane * 4u - (0x47800000u << 7);
    const uint32_t *cw = reinterpret_cast<const uint32_t *>(cur);
    for (int f = 0; f < p.nf; f++)
    {
        const uint32_t *bw = cw;
        const int buf = (f - 1) % NBUF;
        if (f > 0)
        {
            mbar_wait(bar + 1 + buf, (uint32_t)(((f - 1) / NBUF) & 1));
            bw = reinterpret_cast<const uint32_t *>(smem + L::kOffCmp + buf * L::kTileBytes);
        }
        if (rows > 0)
        {
            for (int dy = -p.r_half; dy <= p.r_half; dy++)
            {
                for (int dx0 = -p.r_half; dx0 <= p.r_half; dx0 += kGroup)
                {
                    const int ng  = min(kGroup, p.r_half - dx0 + 1);
                    const int org = (f == 0 && dy == 0 && dx0 <= 0 && dx0 + ng > 0) ? -dx0 : kOrgNone;
                    const int ob  = (12 + dx0) & 3;
#define X(NG_, OB_, ORG_)                                                                                                   \
                    if (ng == NG_ && ob == OB_ && org == ORG_)                                                              \
                        v3_group16<NH, NG_, OB_, ORG_>(cw, bw, acc, lut_lane_addr, wscale, p.origin_tune, seg_y0, rows, lane, dy, dx0); \
                    else
                    V3_GROUP_SHAPES(X)
#undef X
                    { /* unreachable: the launcher checked v3_group_known() for every group of this range */ }
                }
            }
        }
        if (f > 0 && f + NBUF < p.nf)
        {
            __syncthreads();
            if (tid == 0)
            {
                fence_proxy_async();
                mbar_expect_tx(bar + 1 + buf, L::kTileBytes);
                for (int l = 0; l < L::kLoads; l++)
                    tma_load_2d(smem + L::kOffCmp + buf * L::kTileBytes + l * L::kBoxRows * L::kRowBytes, &maps[f + NBUF], gx, gy + l * L::kBoxRows, bar + 1 + buf);
            }
        }
    }

    const int x = lane * 4;
    uint16_t *dst = reinterpret_cast<uint16_t *>(p.dst);
    const uint16_t *cur16 = reinterpret_cast<const uint16_t *>(cur);
    for (int r = 0; r < rows; r++)
    {
        const int oy = seg_y0 + r;
        const int y = Y0 + oy;
        uint32_t accv[8];
        acc.load(r, accv);
        acc.wait_load(accv);
        uint16_t o[4];
#pragma unroll
        for (int i = 0; i < 4; i++)
            o[i] = finish_pixel<uint16_t>(__uint_as_float(accv[v3_acc_slot(i)]), __uint_as_float(accv[4 + v3_acc_slot(i)]),
                                          cur16[(oy + kHalo) * kTilePW + x + kHaloX + i]);
        uint16_t *drow = dst + (size_t)y * p.dpitch + X0 + x;
        if (X0 + x + 3 < p.w)
            *reinterpret_cast<ushort4 *>(drow) = make_ushort4(o[0], o[1], o[2], o[3]);
        else
        {
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (X0 + x + i < p.w) drow[i] = o[i];
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
    {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" :: "r"(*tmem_base_slot) : "memory");
    }
}
