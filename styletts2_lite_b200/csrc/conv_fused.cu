// Fused  [AdaIN affine + Snake / LeakyReLU]  ->  Conv1d / ConvTranspose1d (tcgen05)  ->
// [bias + residual + scale + accumulate + InstanceNorm partial statistics]   for sm_100a.
//
// Replaces, in one kernel, the chain of Modules/hifigan.py:67-73 (AdaINResBlock1 iteration:
// n1/n2 -> Snake -> c1/c2 -> + x) and :329-334 (Snake -> ups -> + x_source).  Per 128-row tile:
//   * the raw fp32 activation rows (128 + (k-1)*dilation halo) are fetched from HBM exactly once --
//     by TMA into an fp32 staging ring when the layer has <= 64 input channels, by batched 128-bit
//     loads otherwise;
//   * transform warps apply the per-(b,c) AdaIN affine y = a*x + b and the activation in registers
//     and write the 128-byte-swizzled K-major bf16/fp16 A operand to shared memory (zero padding =
//     rows written as zeros);
//   * every conv tap is one group of UMMAs whose A descriptor start address is shifted by whole
//     128-byte rows (dilation = row shift), accumulating in TMEM (2 accumulators);
//   * weights are resident in shared memory when all taps fit, else stream through a TMA ring;
//   * the epilogue drains TMEM through a swizzled per-warp staging tile so that residual reads and
//     output writes are 128-byte row segments, and emits per-tile (sum, sum of squares) per channel
//     so the next AdaIN needs no extra pass over the tensor.
// Algorithmic HBM bytes per element: 4 (x) + 4 (y) [+ 4 residual]; HBM-bound for C <= 128.
//
// One persistent CTA per SM, 16 warps (128 registers each):
//   warp 0      TMA producer (weights + fp32 activation tiles)     warp 1    TMEM allocator + MMA issuer (elect.sync lane)
//   warps 2-7   transform (6)                                      warps 8-15  epilogue (2 groups x 4 TMEM lane quarters)
// so tile i+1 is being fetched/transformed while tile i is in the tensor core and tiles i-1, i-2 are
// being stored by the two epilogue groups.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"
#include "tc_ptx.cuh"
#include "fused_ptx.cuh"

namespace st2 {

static constexpr int LW = 6;                              // transform warps
static constexpr int EG = 2;                              // epilogue groups (one per TMEM accumulator)
static constexpr int EW = 4 * EG;                         // epilogue warps
static constexpr int W_LOAD0 = 2;                         // first transform warp
static constexpr int W_EPI0 = W_LOAD0 + LW;               // first epilogue warp (8)
static constexpr int F_THREADS = (W_EPI0 + EW) * 32;      // 512
static constexpr int F_KC = 64;
static constexpr int F_MT = 128;                          // rows per tile
static constexpr int NSTG = 2;                            // fp32 staging buffers (TMA activation path)

struct FusedParams {
    // input + transform
    const float* x; int ld_x; int Tin;
    const float* coef;        // [B][2][coef_ld]: a, b
    int coef_ld;
    const float* alpha;       // [Cin] snake alpha (ACT_SNAKE)
    float slope;              // ACT_LRELU
    int Cin;                  // real input channels
    int kchunks;              // CinPad / 64
    int x16in;                // input tensor is 16-bit (is_bf16 selects bf16 / fp16)
    int y16out;               // output tensor is written as 16-bit
    int k32;                  // 1: Cin == 32 -> 64-byte operand rows (K = 32, SWIZZLE_64B) instead of zero-padding K to 64
    int xstage;               // 1: activations arrive by TMA into the fp32 staging ring (kchunks == 1)
    // geometry (ConvArgs contract, in_stride == 1)
    int B, M, Tout, Cout;
    int ntaps, tap_step, in_off;
    int phases, w_step, out_stride, out_pad;
    int halo_min;             // smallest input-row offset of any tap relative to the tile's first row
    int rows;                 // 128 + span  (rows of the A tile)
    int bn;                   // N tile (CoutPad or 256)
    int ntile_n;
    int mtiles;               // ceil(M / 128)
    int num_tiles;            // B * phases * mtiles * ntile_n
    int stages;               // weight ring depth (resident mode: number of resident [bn x 64] tiles)
    int resident;             // 1: every tap of every phase stays in shared memory for the whole kernel
    int ktaps_total;          // taps stored in the weight tensor (ntaps * phases)
    int tmem_cols;
    int is_bf16;
    // epilogue
    const float* bias;
    const float* res; int ld_res; int res_shift;
    float* y; int ld_y;
    float scale; int accumulate; int mirror;
    float2* stats;            // [B][phases*mtiles*4][Cout] partial (sum, sumsq) per (tile, row quarter), or nullptr
    long long* trace;         // debug: [5 roles][64 tiles][8 events] clock64 of CTA 0 (nullptr = off)
};

#define TRACE(role, seq, ev)                                                                                        \
    do {                                                                                                            \
        if (p.trace != nullptr && blockIdx.x == 0 && (seq) < 64) p.trace[((role) * 64 + (seq)) * 8 + (ev)] = clock64(); \
    } while (0)

__device__ __forceinline__ void epi_bar_sync(int group) { asm volatile("bar.sync %0, 128;" ::"r"(1 + group) : "memory"); }

template <int ACT>
__device__ __forceinline__ float fused_act(float v, float p0, float p1) {
    if (ACT == ACT_LRELU) return v >= 0.f ? v : v * p0;
    if (ACT == ACT_SNAKE) {
        float sn = __sinf(p0 * v);
        return fmaf(p1 * sn, sn, v);
    }
    return v;
}


// Division-free walk over this CTA's tiles: tile = blockIdx.x + i*gridDim.x, decomposed as
// (b, ph, mt, nt) with nt fastest, then mt, ph, b.
struct TileIter {
    int tile, b, ph, mt, nt;
    int d_b, d_ph, d_mt, d_nt;       // decomposition of gridDim.x
    __device__ __forceinline__ void init(const FusedParams& p) {
        const int per_ph = p.mtiles * p.ntile_n, per_b = p.phases * per_ph;
        tile = blockIdx.x;
        b = tile / per_b; int r = tile - b * per_b;
        ph = r / per_ph; r -= ph * per_ph;
        mt = r / p.ntile_n; nt = r - mt * p.ntile_n;
        int g = gridDim.x;
        d_b = g / per_b; g -= d_b * per_b;
        d_ph = g / per_ph; g -= d_ph * per_ph;
        d_mt = g / p.ntile_n; d_nt = g - d_mt * p.ntile_n;
    }
    __device__ __forceinline__ bool valid(const FusedParams& p) const { return tile < p.num_tiles; }
    __device__ __forceinline__ void next(const FusedParams& p) {
        tile += gridDim.x;
        nt += d_nt; if (nt >= p.ntile_n) { nt -= p.ntile_n; ++mt; }
        mt += d_mt; if (mt >= p.mtiles) { mt -= p.mtiles; ++ph; }
        ph += d_ph; if (ph >= p.phases) { ph -= p.phases; ++b; }
        b += d_b;
    }
};


template <int ACT>
__global__ void __launch_bounds__(F_THREADS, 1)
conv_fused_kernel(const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_x, const FusedParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const uint32_t arow = p.k32 ? 64u : 128u;                     // bytes per operand row (K = 32 or 64 16-bit values)
    const uint32_t a_bytes = ((uint32_t)p.rows * arow + 1023u) & ~1023u;
    const uint32_t b_stage_bytes = (uint32_t)p.bn * arow;
    const uint32_t xes = p.x16in ? 2u : 4u;                      // bytes per input element
    const uint32_t x_row_bytes = (uint32_t)p.Cin * xes;                                  // staging row (xstage only)
    const uint32_t x_bytes = p.xstage ? (((uint32_t)p.rows * x_row_bytes + 1023u) & ~1023u) : 0u;
    uint8_t* smem_a = smem;                                       // 2 x [rows][64] 16-bit, SWIZZLE_128B
    uint8_t* smem_b = smem_a + 2 * a_bytes;                       // resident taps or ring of [bn][64]
    uint8_t* smem_x = smem_b + (size_t)p.stages * b_stage_bytes;  // NSTG x [rows][Cin] fp32 (xstage only)
    float* staging = reinterpret_cast<float*>(smem_x + (size_t)NSTG * x_bytes);             // [EW][32 rows][32 cols]
    float2* tstats = reinterpret_cast<float2*>(staging + EW * 32 * 32);                      // [EG][4][bn]
    uint64_t* bars = reinterpret_cast<uint64_t*>(tstats + EG * 4 * p.bn);
    uint64_t* b_full = bars;                    // [stages]
    uint64_t* b_empty = bars + p.stages;        // [stages]
    uint64_t* a_full = bars + 2 * p.stages;     // [2]
    uint64_t* a_empty = a_full + 2;             // [2]
    uint64_t* acc_full = a_full + 4;            // [2]
    uint64_t* acc_empty = a_full + 6;           // [2]
    uint64_t* x_full = a_full + 8;              // [NSTG]
    uint64_t* x_empty = a_full + 8 + NSTG;      // [NSTG]
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(a_full + 8 + 2 * NSTG);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&map_b);
        if (p.xstage) prefetch_tmap(&map_x);
        const int nb = p.resident ? 1 : p.stages;
        for (int s = 0; s < nb; ++s) {
            mbar_init(&b_full[s], 1);
            mbar_init(&b_empty[s], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&a_full[i], LW);
            mbar_init(&a_empty[i], 1);
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], 4);
        }
        for (int i = 0; i < NSTG; ++i) {
            mbar_init(&x_full[i], 1);
            mbar_init(&x_empty[i], LW);
        }
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                     "r"((uint32_t)p.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // channels >= Cin of a 32-channel layer are never written by the transform warps: zero both A tiles once
    for (uint32_t i = threadIdx.x; i < 2 * a_bytes / 16; i += F_THREADS)
        reinterpret_cast<uint4*>(smem_a)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        // ===== TMA producer: weights (resident or ring) and, for single-chunk layers, the fp32 activation tiles =====
        if (elect_one_sync()) {
            if (p.resident) {
                // all taps (of all phases) once: slot = widx * kchunks + kc
                mbar_expect_tx(&b_full[0], (uint32_t)p.ktaps_total * p.kchunks * b_stage_bytes);
                for (int w = 0; w < p.ktaps_total; ++w)
                    for (int kc = 0; kc < p.kchunks; ++kc)
                        tma_load_3d(smem_b + (size_t)(w * p.kchunks + kc) * b_stage_bytes, &map_b, &b_full[0], kc * F_KC, 0, w);
            }
            int stage = 0;
            uint32_t phase = 0, n = 0;
            TileIter ti;
            for (ti.init(p); ti.valid(p); ti.next(p), ++n) {
                if (p.xstage) {
                    const uint32_t s = n % NSTG;
                    mbar_wait(&x_empty[s], ((n / NSTG) & 1) ^ 1);
                    mbar_expect_tx(&x_full[s], (uint32_t)p.rows * x_row_bytes);
                    tma_load_3d(smem_x + (size_t)s * x_bytes, &map_x, &x_full[s], 0, ti.mt * F_MT + p.halo_min, ti.b);
                }
                if (!p.resident)
                    for (int kc = 0; kc < p.kchunks; ++kc)
                        for (int j = 0; j < p.ntaps; ++j) {
                            mbar_wait(&b_empty[stage], phase ^ 1);
                            mbar_expect_tx(&b_full[stage], b_stage_bytes);
                            tma_load_3d(smem_b + (size_t)stage * b_stage_bytes, &map_b, &b_full[stage], kc * F_KC, ti.nt * p.bn,
                                        ti.ph + j * p.w_step);
                            if (++stage == p.stages) { stage = 0; phase ^= 1; }
                        }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (elect_one_sync()) {
            const uint32_t idesc = umma_idesc(128, p.bn, p.is_bf16);
            const uint32_t a_lo0 = desc_lo(smem_u32(smem_a));
            const uint32_t a_buf_step = a_bytes >> 4;
            const uint32_t b_lo0 = desc_lo(smem_u32(smem_b));
            const uint32_t b_step = b_stage_bytes >> 4;
            const int row_u = (int)(arow >> 4);                      // descriptor units (16 B) per operand row
            const int row0 = (p.in_off - p.halo_min) * row_u;
            const int row_step = p.tap_step * row_u;
            // K-major descriptor hi word: SBO = 8 rows (>>4) | version 1 @ bit 46 | SWIZZLE_128B (2) or SWIZZLE_64B (4) @ bit 61
            const uint32_t dhi = p.k32 ? ((512u >> 4) | (1u << 14) | (4u << 29)) : kDescHi;
            const uint32_t b_res_step = (uint32_t)(p.w_step * p.kchunks) * b_step;
            int stage = 0;
            uint32_t phase = 0;
            uint32_t cc = 0, tcnt = 0;
            if (p.resident) {
                mbar_wait(&b_full[0], 0);
                tc_fence_after();
            }
            TileIter ti;
            for (ti.init(p); ti.valid(p); ti.next(p), ++tcnt) {
                const uint32_t acc = tcnt & 1;
                const uint32_t d_tmem = tmem_base + acc * (uint32_t)p.bn;
                TRACE(1, tcnt, 0);
                mbar_wait(&acc_empty[acc], ((tcnt >> 1) & 1) ^ 1);       // epilogue drained this accumulator
                tc_fence_after();
                TRACE(1, tcnt, 1);
                uint32_t accum = 0;
                for (int kc = 0; kc < p.kchunks; ++kc, ++cc) {
                    const uint32_t buf = cc & 1;
                    mbar_wait(&a_full[buf], (cc >> 1) & 1);
                    tc_fence_after();
                    if (kc == 0) TRACE(1, tcnt, 2);
                    uint32_t a_lo = a_lo0 + buf * a_buf_step + (uint32_t)row0;
                    if (p.resident) {
                        // resident weights: no barrier inside the tap loop -> branch-free, unrolled issue
                        uint32_t b_lo = b_lo0 + (uint32_t)(ti.ph * p.kchunks + kc) * b_step;     // widx = ph + j*w_step
                        if (p.k32) {
#pragma unroll 4
                            for (int j = 0; j < p.ntaps; ++j) {
                                umma_f16_lohi(d_tmem, a_lo, b_lo, dhi, idesc, accum);
                                umma_f16_lohi(d_tmem, a_lo + 2, b_lo + 2, dhi, idesc, 1u);
                                accum = 1u;
                                a_lo += (uint32_t)row_step;
                                b_lo += b_res_step;
                            }
                        } else {
#pragma unroll 2
                            for (int j = 0; j < p.ntaps; ++j) {
                                umma_f16_lohi(d_tmem, a_lo, b_lo, dhi, idesc, accum);
                                umma_f16_lohi(d_tmem, a_lo + 2, b_lo + 2, dhi, idesc, 1u);
                                umma_f16_lohi(d_tmem, a_lo + 4, b_lo + 4, dhi, idesc, 1u);
                                umma_f16_lohi(d_tmem, a_lo + 6, b_lo + 6, dhi, idesc, 1u);
                                accum = 1u;
                                a_lo += (uint32_t)row_step;
                                b_lo += b_res_step;
                            }
                        }
                    } else {
                        for (int j = 0; j < p.ntaps; ++j) {
                            mbar_wait(&b_full[stage], phase);
                            tc_fence_after();
                            const uint32_t b_lo = b_lo0 + (uint32_t)stage * b_step;
                            umma_f16_lohi(d_tmem, a_lo, b_lo, dhi, idesc, accum);
                            umma_f16_lohi(d_tmem, a_lo + 2, b_lo + 2, dhi, idesc, 1u);
                            umma_f16_lohi(d_tmem, a_lo + 4, b_lo + 4, dhi, idesc, 1u);
                            umma_f16_lohi(d_tmem, a_lo + 6, b_lo + 6, dhi, idesc, 1u);
                            accum = 1u;
                            a_lo += (uint32_t)row_step;
                            umma_commit(&b_empty[stage]);
                            if (++stage == p.stages) { stage = 0; phase ^= 1; }
                        }
                    }
                    umma_commit(&a_empty[buf]);          // A tile consumed
                }
                umma_commit(&acc_full[acc]);             // accumulator complete
                TRACE(1, tcnt, 5);
            }
        }
    } else if (warp < W_EPI0) {
        // ===== transform: x -> act(a*x+b) -> swizzled 16-bit A tile =====
        const int lt = (warp - W_LOAD0) * 32 + lane;      // 0..191
        const int cin_last = p.Cin - (p.kchunks - 1) * F_KC;
        const uint32_t smem_a_u32 = smem_u32(smem_a);
        const uint32_t smem_x_u32 = smem_u32(smem_x);
        uint32_t cc = 0;
        int lseq = 0;
        int cached_b = -1;
        XfCoef cf;
        TileIter ti;
        for (ti.init(p); ti.valid(p); ti.next(p), ++lseq) {
            const int t_base = ti.mt * F_MT + p.halo_min;
            if (lt == 0) TRACE(0, lseq, 0);
            for (int kc = 0; kc < p.kchunks; ++kc, ++cc) {
                const uint32_t buf = cc & 1;
                const int cch = (kc == p.kchunks - 1) ? cin_last : F_KC;
                const int lpr_shift = (cch == 64) ? 4 : 3;                  // float4 lanes per row: 16 or 8
                const int rpp = (LW * 32) >> lpr_shift;                     // rows per pass: 12 or 24
                const int rl = lt >> lpr_shift;
                const int c4 = (lt & ((1 << lpr_shift) - 1)) * 4;
                const int cg = kc * F_KC + c4;
                if (p.kchunks > 1 || ti.b != cached_b) {                    // per-(b,c) coefficients: reload only when they change
                    const float* ca = p.coef + (size_t)ti.b * 2 * p.coef_ld;
                    const float4 a4 = __ldg(reinterpret_cast<const float4*>(ca + cg));
                    const float4 b4 = __ldg(reinterpret_cast<const float4*>(ca + p.coef_ld + cg));
                    cf.a01 = make_float2(a4.x, a4.y); cf.a23 = make_float2(a4.z, a4.w);
                    cf.b01 = make_float2(b4.x, b4.y); cf.b23 = make_float2(b4.z, b4.w);
                    if (ACT == ACT_SNAKE) {
                        const float4 al = __ldg(reinterpret_cast<const float4*>(p.alpha + cg));
                        cf.al01 = make_float2(al.x, al.y); cf.al23 = make_float2(al.z, al.w);
                        cf.ia01 = make_float2(__fdividef(1.f, al.x), __fdividef(1.f, al.y));
                        cf.ia23 = make_float2(__fdividef(1.f, al.z), __fdividef(1.f, al.w));
                    } else {
                        cf.al01 = make_float2(p.slope, p.slope); cf.al23 = cf.al01; cf.ia01 = cf.al01; cf.ia23 = cf.al01;
                    }
                    cached_b = ti.b;
                }
                // A-tile byte address of (row r, this thread's 8-byte slot):
                //   SWIZZLE_128B: r*128 + ((chunk ^ (r & 7)) << 4) + sub      SWIZZLE_64B: r*64 + ((chunk ^ ((r >> 1) & 3)) << 4) + sub
                const uint32_t cidx = (uint32_t)(c4 >> 3), sub = (uint32_t)(c4 & 4) * 2u;
                const uint32_t abase = smem_a_u32 + buf * a_bytes + sub;
                const uint32_t sw_shift = p.k32 ? 1u : 0u, sw_mask = p.k32 ? 3u : 7u;
#define A_ADDR(r) (abase + (uint32_t)(r) * arow + ((cidx ^ (((uint32_t)(r) >> sw_shift) & sw_mask)) << 4))
                if (p.xstage) {
                    // ---- staged path: fp32 rows already in shared memory (TMA), no global latency exposed
                    const uint32_t s = cc % NSTG;                           // kchunks == 1: one staging tile per tile
                    mbar_wait_warp(&x_full[s], (cc / NSTG) & 1);
                    if (lt == 0) TRACE(0, lseq, 1);
                    mbar_wait_warp(&a_empty[buf], ((cc >> 1) & 1) ^ 1);
                    if (lt == 0) TRACE(0, lseq, 2);
                    uint32_t xaddr = smem_x_u32 + s * x_bytes + (uint32_t)rl * x_row_bytes + (uint32_t)c4 * xes;
                    const uint32_t xstep = (uint32_t)rpp * x_row_bytes;
                    int t = t_base + rl;
                    for (int r = rl; r < p.rows; r += 2 * rpp) {            // two independent rows per iteration (ILP)
                        const bool has1 = (r + rpp) < p.rows;
                        float4 v0, v1 = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (p.x16in) {
                            v0 = unpack16x4(lds64(xaddr), p.is_bf16);
                            if (has1) v1 = unpack16x4(lds64(xaddr + xstep), p.is_bf16);
                        } else {
                            v0 = lds128(xaddr);
                            if (has1) v1 = lds128(xaddr + xstep);
                        }
                        uint2 o0 = transform4<ACT>(v0, cf, p.is_bf16);
                        uint2 o1 = transform4<ACT>(v1, cf, p.is_bf16);
                        if (t < 0 || t >= p.Tin) o0 = make_uint2(0u, 0u);   // conv zero padding
                        if (t + rpp < 0 || t + rpp >= p.Tin) o1 = make_uint2(0u, 0u);
                        sts64(A_ADDR(r), o0.x, o0.y);
                        if (has1) sts64(A_ADDR(r + rpp), o1.x, o1.y);
                        xaddr += 2 * xstep;
                        t += 2 * rpp;
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&x_empty[s]);                // staging tile consumed
                } else {
                    // ---- direct path: batched 128-bit global loads (whole tile in flight), then transform
                    const char* xp = reinterpret_cast<const char*>(p.x) + (((size_t)ti.b * p.Tin + t_base + rl) * p.ld_x + cg) * xes;
                    const size_t xstep = (size_t)rpp * p.ld_x * xes;
                    constexpr int U = 16;                                   // 16 x 12 rows >= 128 + 64
                    float4 v[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int r = rl + u * rpp;
                        const int t = t_base + r;
                        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (r < p.rows && t >= 0 && t < p.Tin) {
                            if (p.x16in) v[u] = unpack16x4(__ldg(reinterpret_cast<const uint2*>(xp + u * xstep)), p.is_bf16);
                            else v[u] = __ldg(reinterpret_cast<const float4*>(xp + u * xstep));
                        }
                    }
                    if (lt == 0 && kc == 0) TRACE(0, lseq, 1);
                    mbar_wait_warp(&a_empty[buf], ((cc >> 1) & 1) ^ 1);     // loads are in flight while we wait for the buffer
                    if (lt == 0 && kc == 0) TRACE(0, lseq, 2);
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int r = rl + u * rpp;
                        const int t = t_base + r;
                        if (r < p.rows) {
                            uint2 o = transform4<ACT>(v[u], cf, p.is_bf16);
                            if (t < 0 || t >= p.Tin) o = make_uint2(0u, 0u);
                            sts64(A_ADDR(r), o.x, o.y);
                        }
                    }
                }
#undef A_ADDR
                if (lt == 0 && kc == 0) TRACE(0, lseq, 3);
                fence_proxy_async();            // generic-proxy smem writes -> visible to the tensor core (async proxy)
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[buf]);
            }
        }
    } else {
        // ===== epilogue: TMEM -> staging -> (+bias, +res, accumulate, scale) -> global, statistics =====
        // group g (4 warps = 4 TMEM lane quarters) owns accumulator g and every other tile of this CTA
        const int ew = warp - W_EPI0;                     // 0..7
        const int grp = ew >> 2;                          // 0..1
        const int q = warp & 3;                           // TMEM lane quarter this warp may access
        const int et = (ew & 3) * 32 + lane;              // thread id within the group
        const uint32_t stg_u32 = smem_u32(staging + ew * (32 * 32));
        const int rr = lane >> 3;                         // 0..3: row within a 4-row pass
        const uint32_t l7 = (uint32_t)lane & 7u;
        const int c4o = (int)l7 * 4;                      // column within the 32-column chunk
        // staging tile [32 rows][32 cols] fp32, 16-byte slots XOR-swizzled by (row & 7): conflict-free both ways
        const uint32_t st_w = stg_u32 + (uint32_t)lane * 128u;                       // row = lane (TMEM drain)
        const uint32_t st_r0 = stg_u32 + (uint32_t)rr * 128u + ((l7 ^ (uint32_t)rr) << 4);          // rows rr, rr+8, ...
        const uint32_t st_r1 = stg_u32 + (uint32_t)(rr + 4) * 128u + ((l7 ^ (uint32_t)(rr + 4)) << 4);  // rows rr+4, rr+12, ...
        const int ystep = 4 * p.out_stride * p.ld_y;      // element distance between consecutive row passes
        const int rstep = 4 * p.out_stride * p.ld_res;
        const bool do_scale = p.scale != 1.f;
        const float2 sc2 = make_float2(p.scale, p.scale);
        uint32_t tcnt = 0;
        TileIter ti;
        for (ti.init(p); ti.valid(p); ti.next(p), ++tcnt) {
            if ((int)(tcnt & 1) != grp) continue;
            const int n0 = ti.nt * p.bn;
            const uint32_t acc = tcnt & 1;
            if (et == 0) TRACE(2 + grp, tcnt, 0);
            // rows of this lane: m = m_first + 4*it  ->  t = t_first + 4*it*out_stride ; validity as a bit mask
            const int m_first = ti.mt * F_MT + q * 32 + rr;
            const int t_first = m_first * p.out_stride + ti.ph - p.out_pad;
            uint32_t vmask = 0;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int m = m_first + it * 4;
                const int t = t_first + it * 4 * p.out_stride;
                if (m < p.M && t >= (p.mirror ? 1 : 0) && t < p.Tout) vmask |= 1u << it;   // mirror: row 0 is written by the row-2 thread only
            }
            if (et == 0) TRACE(2 + grp, tcnt, 4);
            float* ytile = p.y + ((size_t)ti.b * p.Tout + t_first) * p.ld_y;
            const float* rtile = p.res ? p.res + ((size_t)ti.b * p.Tout + t_first) * p.ld_res : nullptr;
            bool waited = false;
            for (int cc0 = 0; cc0 < p.bn; cc0 += 32) {
                const int co = n0 + cc0 + c4o;
                const uint32_t cmask = (co < p.Cout) ? vmask : 0u;
                float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (p.bias != nullptr && cmask) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias + co));
                const float2 bias01 = make_float2(bias4.x, bias4.y), bias23 = make_float2(bias4.z, bias4.w);
                if (et == 0 && cc0 == 0) TRACE(2 + grp, tcnt, 6);
                // residual (+ accumulate) rows of all 8 passes in one batch of loads; for the first column chunk they are in
                // flight while the tensor core is still working on this tile
                float4 rv[8];
                {
                    const float* rp = rtile ? rtile + co : nullptr;
                    const float* yo = ytile + co;
                    // all loads are issued before any of them is consumed (a predicated-off consumer still waits on the
                    // scoreboard of its sources, which would serialise the loads)
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        rv[it] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (((cmask >> it) & 1u) && rp != nullptr) rv[it] = ldg_stream(rp + it * rstep);
                    }
                    if (p.accumulate) {
                        float4 old[8];
#pragma unroll
                        for (int it = 0; it < 8; ++it) {
                            old[it] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if ((cmask >> it) & 1u) old[it] = ldg_stream(yo + it * ystep);
                        }
#pragma unroll
                        for (int it = 0; it < 8; ++it) {
                            rv[it].x += old[it].x; rv[it].y += old[it].y; rv[it].z += old[it].z; rv[it].w += old[it].w;
                        }
                    }
                }
                if (!waited) {
                    if (et == 0) TRACE(2 + grp, tcnt, 1);
                    mbar_wait_warp(&acc_full[acc], (tcnt >> 1) & 1);
                    tc_fence_after();
                    waited = true;
                    if (et == 0) TRACE(2 + grp, tcnt, 2);
                }
                {
                    float v[32];
                    tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * (uint32_t)p.bn + (uint32_t)cc0, v);
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        sts128(st_w + (((uint32_t)i ^ l7) << 4), v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                }
                __syncwarp();
                float2 s1a = make_float2(0.f, 0.f), s1b = s1a, s2a = s1a, s2b = s1a;
                float* yo = ytile + co;
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                    const float4 a = lds128(((it & 1) ? st_r1 : st_r0) + (uint32_t)(it >> 1) * 1024u);
                    if (!((cmask >> it) & 1u)) continue;
                    float2 o01 = fadd2(fadd2(make_float2(a.x, a.y), bias01), make_float2(rv[it].x, rv[it].y));
                    float2 o23 = fadd2(fadd2(make_float2(a.z, a.w), bias23), make_float2(rv[it].z, rv[it].w));
                    if (do_scale) {
                        o01 = fmul2(o01, sc2);
                        o23 = fmul2(o23, sc2);
                    }
                    if (p.y16out)
                        *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(p.y) + (yo - p.y) + it * ystep) =
                            make_uint2(pack16(o01.x, o01.y, p.is_bf16), pack16(o23.x, o23.y, p.is_bf16));
                    else
                        *reinterpret_cast<float4*>(yo + it * ystep) = make_float4(o01.x, o01.y, o23.x, o23.y);
                    s1a = fadd2(s1a, o01); s1b = fadd2(s1b, o23);
                    s2a = ffma2(o01, o01, s2a); s2b = ffma2(o23, o23, s2b);
                    if (p.mirror && t_first + it * 4 * p.out_stride == 2) {
                        // ReflectionPad1d((1,0)): the conv value of (shifted) row 2 also lands in row 0 (with row 0's residual)
                        float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (p.res != nullptr) r0 = *reinterpret_cast<const float4*>(p.res + (size_t)ti.b * p.Tout * p.ld_res + co);
                        float2 m01 = fadd2(fadd2(make_float2(a.x, a.y), bias01), make_float2(r0.x, r0.y));
                        float2 m23 = fadd2(fadd2(make_float2(a.z, a.w), bias23), make_float2(r0.z, r0.w));
                        if (do_scale) { m01 = fmul2(m01, sc2); m23 = fmul2(m23, sc2); }
                        *reinterpret_cast<float4*>(p.y + (size_t)ti.b * p.Tout * p.ld_y + co) = make_float4(m01.x, m01.y, m23.x, m23.y);
                        s1a = fadd2(s1a, m01); s1b = fadd2(s1b, m23);
                        s2a = ffma2(m01, m01, s2a); s2b = ffma2(m23, m23, s2b);
                    }
                }
                if (p.stats != nullptr) {
                    float s1[4] = {s1a.x, s1a.y, s1b.x, s1b.y}, s2[4] = {s2a.x, s2a.y, s2b.x, s2b.y};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        s1[i] += __shfl_xor_sync(0xffffffffu, s1[i], 8);
                        s2[i] += __shfl_xor_sync(0xffffffffu, s2[i], 8);
                        s1[i] += __shfl_xor_sync(0xffffffffu, s1[i], 16);
                        s2[i] += __shfl_xor_sync(0xffffffffu, s2[i], 16);
                    }
                    // one partial per (tile, TMEM lane quarter): written straight to global, no cross-warp barrier
                    if (lane < 8 && co < p.Cout) {
                        float2* sp = p.stats + (((size_t)ti.b * (p.phases * p.mtiles) + (size_t)ti.ph * p.mtiles + ti.mt) * 4 + q) * p.Cout + co;
                        *reinterpret_cast<float4*>(sp) = make_float4(s1[0], s2[0], s1[1], s2[1]);
                        *reinterpret_cast<float4*>(sp + 2) = make_float4(s1[2], s2[2], s1[3], s2[3]);
                    }
                }
                __syncwarp();
            }
            // accumulator drained: hand it back to the MMA warp
            if (et == 0) TRACE(2 + grp, tcnt, 3);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[acc]);
            if (et == 0) TRACE(2 + grp, tcnt, 5);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols)
                     : "memory");
    }
}

// ---------------------------------------------------------------- coefficients from float2 tile partials
// grid (ceil(Cpad/32), B), block (32 channels x 32 slices of the partial list): each thread sums every 32nd partial
// (8 independent loads in flight), then a fixed-order tree over the 32 slices -> deterministic.
__global__ void __launch_bounds__(1024)
adain_coef_f2_kernel(const float2* __restrict__ partial, int nparts, const float* __restrict__ h, int ld_h, int h_off,
                     float* __restrict__ coef, int T, int C, int Cpad, const float* __restrict__ x_offset,
                     const float* __restrict__ stat_shift) {
    __shared__ double ssum[32][33], ssq[32][33];
    pdl_trigger();
    pdl_wait();                 // the partials come from the kernel before this one
    const int cx = threadIdx.x & 31, py = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + cx;
    const int b = blockIdx.y;
    double s = 0, ss = 0;
    if (c < C) {
        const float2* pp = partial + (size_t)b * nparts * C + c;
        int i = py;
        for (; i + 7 * 32 < nparts; i += 8 * 32) {
            float2 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = __ldg(pp + (size_t)(i + u * 32) * C);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                s += (double)v[u].x;
                ss += (double)v[u].y;
            }
        }
        for (; i < nparts; i += 32) {
            const float2 v = __ldg(pp + (size_t)i * C);
            s += (double)v.x;
            ss += (double)v.y;
        }
    }
    ssum[py][cx] = s;
    ssq[py][cx] = ss;
    __syncthreads();
    if (py != 0 || c >= Cpad) return;
    float a = 0.f, bb = 0.f;
    if (c < C) {
        for (int i = 1; i < 32; ++i) {
            s += ssum[i][cx];
            ss += ssq[i][cx];
        }
        const double mean = s / (double)T;
        double var = ss / (double)T - mean * mean;
        if (var < 0) var = 0;
        const double rstd = 1.0 / sqrt(var + 1e-5);
        const double gamma = (double)h[(size_t)b * ld_h + h_off + c];
        const double beta = (double)h[(size_t)b * ld_h + h_off + C + c];
        const double ad = (1.0 + gamma) * rstd;
        a = (float)ad;
        // partials of x - stat_shift: mean(x) = mean + stat_shift, the variance is that of the partials;
        // stored tensor = x - x_offset: a * x + b = a * (x - x_offset) + (b + a * x_offset)
        const double d = (stat_shift ? (double)stat_shift[c] : 0.0) - (x_offset ? (double)x_offset[c] : 0.0);
        bb = (float)(beta - (mean + d) * ad);
    }
    coef[((size_t)b * 2 + 0) * Cpad + c] = a;
    coef[((size_t)b * 2 + 1) * Cpad + c] = bb;
}

int launch_adain_coef_f2(const void* partial, int nparts, const float* h, int ld_h, int h_off, float* coef, int B, int T,
                         int C, int Cpad, cudaStream_t st, const float* x_offset, const float* stat_shift) {
    dim3 grid(cdiv(Cpad, 32), B);
    // programmatic dependent launch for small grids (one-sentence latency): the CTAs may be scheduled while the producing conv
    // drains.  Large batches gain nothing and lose SMs to the next conv's early CTAs (conv_pipe.cu)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(1024); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    const bool pdl = (int64_t)grid.x * grid.y <= 64;
    cfg.attrs = &attr; cfg.numAttrs = pdl ? 1 : 0;
    ST2_CUDA_CHECK(cudaLaunchKernelEx(&cfg, adain_coef_f2_kernel, (const float2*)partial, nparts, h, ld_h, h_off, coef, T, C, Cpad, x_offset,
                                      stat_shift));
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---------------------------------------------------------------- host side
int make_weight_map(CUtensorMap* map, int is_bf16, const void* w16, int cin_pad, int cout_pad, int ktaps, int bn);
int make_weight_map_k32(CUtensorMap* map, int is_bf16, const void* w16, int cin_pad, int cout_pad, int ktaps, int bn);
int make_act16_map_3d(CUtensorMap* map, int is_bf16, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                      uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t b0, uint32_t b1);
int make_f32_map_3d(CUtensorMap* map, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                    uint64_t stride2_bytes, uint32_t b0, uint32_t b1);

int fused_stats_parts(const ConvArgs& a) { return a.phases * cdiv(a.M, F_MT) * 4; }   // one per (tile, 32-row quarter)

bool conv_fused_supported(const ConvArgs& a) {
    if (a.in_stride != 1 || a.w16 == nullptr || a.w16_cin_pad % F_KC != 0 || a.w16_cout_pad % 32 != 0) return false;
    if (a.Cin % 4 != 0 || a.ld_x % 4 != 0 || a.Cout % 4 != 0 || a.ld_y % 4 != 0) return false;
    if (a.res != nullptr && (a.ld_res % 4 != 0 || a.res_shift != 0)) return false;
    const int last = a.Cin - (a.w16_cin_pad / F_KC - 1) * F_KC;
    if (last != 32 && last != 64) return false;          // 8 or 16 float4 lanes per row
    const int span = (a.ntaps - 1) * (a.tap_step < 0 ? -a.tap_step : a.tap_step);
    return span <= 64;
}

int launch_conv_fused(const ConvArgs& a, const float* coef, int coef_ld, int act, float slope, const float* alpha,
                      void* stats_out, cudaStream_t st) {
    ST2_REQUIRE(conv_fused_supported(a), "conv_fused: unsupported geometry");
    if (conv_pipe_supported(a)) return launch_conv_pipe(a, coef, coef_ld, act, slope, alpha, stats_out, st);
    FusedParams p;
    memset(&p, 0, sizeof(p));
    p.x = a.x; p.ld_x = a.ld_x; p.Tin = a.Tin;
    p.x16in = a.x16in; p.y16out = a.y16out;
    ST2_REQUIRE(!(a.y16out && (a.accumulate || a.mirror)), "conv_fused: 16-bit output cannot accumulate / mirror");
    ST2_REQUIRE(!a.res16 && a.acc_src == nullptr, "conv_fused: a 16-bit residual / separate accumulate source is only supported by the TMA pipeline kernel");
    p.coef = coef; p.coef_ld = coef_ld; p.alpha = alpha; p.slope = slope;
    p.Cin = a.Cin; p.kchunks = a.w16_cin_pad / F_KC;
    p.B = a.B; p.M = a.M; p.Tout = a.Tout; p.Cout = a.Cout;
    p.ntaps = a.ntaps; p.tap_step = a.tap_step; p.in_off = a.in_off;
    p.phases = a.phases; p.w_step = a.w_step; p.out_stride = a.out_stride; p.out_pad = a.out_pad;
    const int span = (a.ntaps - 1) * (a.tap_step < 0 ? -a.tap_step : a.tap_step);
    p.halo_min = a.in_off + (a.tap_step < 0 ? (a.ntaps - 1) * a.tap_step : 0);
    p.rows = F_MT + span;
    int bn = a.w16_cout_pad;
    if (bn > 256) {
        bn = 256;
        while (a.w16_cout_pad % bn != 0) bn -= 32;
    }
    p.bn = bn;
    p.ntile_n = a.w16_cout_pad / bn;
    p.mtiles = cdiv(a.M, F_MT);
    p.num_tiles = a.B * a.phases * p.mtiles * p.ntile_n;
    int cols = 32;
    while (cols < 2 * bn) cols <<= 1;
    p.tmem_cols = cols;
    p.is_bf16 = a.fmt16 == DT_BF16 ? 1 : 0;
    p.bias = a.bias; p.res = a.res; p.ld_res = a.ld_res; p.res_shift = a.res_shift;
    p.y = a.y; p.ld_y = a.ld_y; p.scale = a.scale; p.accumulate = a.accumulate; p.mirror = a.mirror;
    p.stats = (float2*)stats_out;
    // shared-memory plan (one persistent CTA per SM, <= ~224 KB)
    const int64_t budget = 224 * 1024;
    p.k32 = (a.Cin == 32 && a.w16_cin_pad == 64) ? 1 : 0;
    const int64_t arow = p.k32 ? 64 : 128;
    const int64_t a_bytes = ((int64_t)p.rows * arow + 1023) & ~(int64_t)1023;
    const int64_t b_stage = (int64_t)bn * arow;
    const int64_t base_fixed = 2 * a_bytes + EW * 32 * 32 * 4 + (int64_t)EG * 4 * bn * 8 + 160 * 8 + 1024;
    // activations by TMA into an fp32 staging ring for single-chunk layers (C <= 64), when the ring fits
    const int64_t x_bytes = (((int64_t)p.rows * a.Cin * (a.x16in ? 2 : 4)) + 1023) & ~(int64_t)1023;
    p.xstage = (p.kchunks == 1 && a.ld_x * (a.x16in ? 2 : 4) % 16 == 0) ? 1 : 0;
    int64_t fixed = base_fixed + (p.xstage ? NSTG * x_bytes : 0);
    const int ktaps_total = a.phases > 1 ? a.ntaps * a.phases : a.ntaps;
    p.ktaps_total = ktaps_total;
    const int64_t resident_tiles = (int64_t)ktaps_total * p.kchunks;
    // weights resident when every tap of every phase fits, else a ring with what is left (>= 4 stages; drop the
    // staging ring first if it would starve the weight ring)
    p.resident = (p.ntile_n == 1 && fixed + resident_tiles * b_stage <= budget && resident_tiles * b_stage < (1 << 20)) ? 1 : 0;
    const bool resident_without_stage = (p.ntile_n == 1 && base_fixed + resident_tiles * b_stage <= budget &&
                                         resident_tiles * b_stage < (1 << 20));
    // resident weights beat the staging ring: a ring shallower than two tiles of taps starves the tensor core
    if (!p.resident && p.xstage && (resident_without_stage || (budget - fixed) / b_stage < 6)) {
        p.xstage = 0;
        fixed = base_fixed;
        p.resident = (p.ntile_n == 1 && fixed + resident_tiles * b_stage <= budget && resident_tiles * b_stage < (1 << 20)) ? 1 : 0;
    }
    int stages;
    if (p.resident) {
        stages = (int)resident_tiles;
    } else {
        stages = (int)((budget - fixed) / b_stage);
        if (stages > 16) stages = 16;
        if (stages < 2) stages = 2;
    }
    p.stages = stages;
    const size_t smem = (size_t)fixed + (size_t)stages * b_stage;
    ST2_REQUIRE(smem <= 227 * 1024, "conv_fused: shared-memory plan %zu exceeds 227 KB", smem);
    CUtensorMap map_b, map_x;
    int e = p.k32 ? make_weight_map_k32(&map_b, p.is_bf16, a.w16, a.w16_cin_pad, a.w16_cout_pad, ktaps_total, bn)
                  : make_weight_map(&map_b, p.is_bf16, a.w16, a.w16_cin_pad, a.w16_cout_pad, ktaps_total, bn);
    if (e != ST2_OK) return e;
    if (p.xstage) {
        if (a.x16in)
            e = make_act16_map_3d(&map_x, p.is_bf16, a.x, (uint64_t)a.Cin, (uint64_t)a.Tin, (uint64_t)a.B, (uint64_t)a.ld_x * 2,
                                  (uint64_t)a.Tin * a.ld_x * 2, (uint32_t)a.Cin, (uint32_t)p.rows);
        else
            e = make_f32_map_3d(&map_x, a.x, (uint64_t)a.Cin, (uint64_t)a.Tin, (uint64_t)a.B, (uint64_t)a.ld_x * 4,
                                (uint64_t)a.Tin * a.ld_x * 4, (uint32_t)a.Cin, (uint32_t)p.rows);
        if (e != ST2_OK) return e;
    } else {
        map_x = map_b;
    }
    static bool attr_done[kMaxDevices] = {};
    const int num_sms = device_num_sms();
    if (!attr_done[current_device_slot()]) {
        ST2_CUDA_CHECK(cudaFuncSetAttribute(conv_fused_kernel<ACT_NONE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        ST2_CUDA_CHECK(cudaFuncSetAttribute(conv_fused_kernel<ACT_LRELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        ST2_CUDA_CHECK(cudaFuncSetAttribute(conv_fused_kernel<ACT_SNAKE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        attr_done[current_device_slot()] = true;
    }
    int grid = num_sms;
    if (grid > p.num_tiles) grid = p.num_tiles;
    if (tune().verbose)
        fprintf(stderr, "conv_fused: Cin=%d Cout=%d taps=%d step=%d phases=%d mtiles=%d ntile_n=%d bn=%d tiles=%d grid=%d resident=%d "
                "stages=%d xstage=%d res=%d acc=%d x16=%d y16=%d smem=%zu\n",
                a.Cin, a.Cout, p.ntaps, p.tap_step, p.phases, p.mtiles, p.ntile_n, p.bn, p.num_tiles, grid, p.resident, p.stages,
                p.xstage, a.res != nullptr ? 1 : 0, p.accumulate, p.x16in, p.y16out, smem);
    switch (act) {
        case ACT_NONE: conv_fused_kernel<ACT_NONE><<<grid, F_THREADS, smem, st>>>(map_b, map_x, p); break;
        case ACT_LRELU: conv_fused_kernel<ACT_LRELU><<<grid, F_THREADS, smem, st>>>(map_b, map_x, p); break;
        case ACT_SNAKE:
            ST2_REQUIRE(alpha != nullptr, "conv_fused: snake needs alpha");
            conv_fused_kernel<ACT_SNAKE><<<grid, F_THREADS, smem, st>>>(map_b, map_x, p);
            break;
        default: set_error("conv_fused: bad act %d", act); return ST2_ERR_INVALID;
    }
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

}  // namespace st2
