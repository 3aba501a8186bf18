// Row-per-thread fused kernel for the 32- and 64-channel convolutions of AdaINResBlock1 (Modules/hifigan.py:65-74):
//   y = (conv1d(snake(a*x + b), w) + bias [+ res] [+ old]) * scale,  InstanceNorm partial statistics of y
// with every stage-private tensor (x, res, old, usually y) stored as fp16 (DESIGN.md section 3).  These layers are 22 of the
// 45.7 ms of a 64 x 5 s forward on conv_pipe.cu and sit at 2-3x their byte floor there: ncu shows its epilogue executing ~360
// instructions per 32x32 chunk (residual ring, transposition through shared memory, per-tile statistics partials) and the
// transform warps re-transforming the halo of every 128-row tile.  This kernel changes the decomposition:
//   * tiles: a CTA owns a CONTIGUOUS range of macro tiles (1, 2 or 4 MMA sub-tiles of 128 rows that share one transformed
//     operand buffer of sub*128 + span rows), so the halo is transformed once per macro tile and every role walks rows in order;
//   * residual / accumulate sources never touch a compute warp: their fp16 tiles land by TMA in the K-major UMMA layout and are
//     added into the accumulator by the tensor core itself (D += R * I with a resident fp16 identity tile; exact in fp32);
//   * epilogue: one thread = one output row (the TMEM drain layout).  No shared memory: 16 accumulator columns at a time go
//     TMEM -> registers -> scale/bias -> fp16 pack -> 32 contiguous bytes of the row in global memory (the four stores of a
//     chunk fill every 32-byte sector they touch), and the InstanceNorm (sum, sum of squares) of the 32 channels a warp owns
//     stay in 64 registers per thread ACROSS tiles; they are reduced over the 32 lanes by a fixed-order butterfly only when the
//     utterance changes -- one partial per (CTA, utterance, epilogue warp) instead of one per (tile, 32-row quarter), which also
//     shrinks what the coefficient kernel reads from ~45 MB to a few hundred KB;
//   * activation blocks go through PRIVATE, SELF-FED rings (one per transform warp, depth xd): the warp that consumes a slot
//     issues the TMA load that refills it, so there is no producer thread in the activation path (the first build had one
//     thread test-waiting and issuing 9 blocks + 4 residual tiles per macro tile: ncu showed the transform warps at an mbarrier
//     in 44 % of all samples), no empty barrier and no sequence-number spin; blocks are always processed in whole batches of 8
//     passes (the operand buffer has slack rows for the overshoot), so the ragged path only runs next to the zero padding.
// Roles (20 warps; 96 registers at launch, re-split by setmaxnreg to 80-88 / 120 for the epilogue): warp 0 residual-tile
// producer, warp 1 TMEM allocator + MMA issuer, 18 - 4*NCH transform warps, 4*NCH epilogue warps (NCH = C / 32; epilogue warp
// ew drains TMEM lane quarter warp & 3 of column chunk ew >> 2 of every sub-tile).
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"
#include "tc_ptx.cuh"
#include "fused_ptx.cuh"

namespace st2 {

static constexpr int RW_THREADS = 640;                    // 20 warps (ptxas grants 96 registers from 545 threads up)
static constexpr int RW_X0 = 2;                          // first transform warp
static constexpr int RW_MAXGRID = 160;                   // statistics buffers are sized for at most this many CTAs

// where the partials of an utterance live in the statistics buffer of a conv_row launch (see flush() and RowStatsDesc)
struct RowStatsInfo { int grid, J, nwarp, mmt, tq, tr, C; };

struct RowParams {
    // transform
    const float* coef; int coef_ld;
    const float* alpha;
    // geometry
    int B, M, ntaps, tap_step, halo_min, a_row0;
    int sub;                    // MMA sub-tiles (128 rows) per macro tile
    int R, nblk, tail_rows;     // activation blocks: R rows each, nblk per macro tile, the last one loads tail_rows rows
    int xslot;                  // bytes per activation ring slot
    int a_bytes;                // bytes per operand buffer (nblk * R rows)
    int na;                     // operand buffers (macro tiles in flight between transform and MMA): 2 .. 4
    int lw, xd;                 // active transform warps, depth of each private activation ring
    int nacc, nacc_log2, tmem_cols;
    int nres, nr;               // fp16 sources added by the identity MMA (0, 1, 2), residual ring stages
    int mmt;                    // macro tiles per utterance
    int tq, tr;                 // macro tiles per CTA: CTAs [0, tr) own tq + 1, the rest tq (contiguous ranges)
    int J;                      // statistics slots per CTA (utterances a CTA can touch)
    // epilogue
    const float* bias; float scale;
    void* y; int ld_y;
    // bias_mma (C = 32, scale == 1): the bias enters the accumulator through one extra tcgen05.mma -- D = ONES[128 x 16] x
    // BIAS[16 x C] with bias_hi / bias_lo (an fp16 pair per channel) in rows k = 0, 1 -- instead of 8 shared-memory loads and 16
    // packed FMAs per row in the epilogue, the busiest role of the 32-channel layers
    int bias_mma;
    // AdaIN coefficients computed in the kernel (cin_part != nullptr) from the partials of the conv_row launch that produced x,
    // instead of read from `coef`: no coefficient launch between two convs of a resblock
    const float2* cin_part; RowStatsInfo cin_si; const float* cin_h; int cin_ld_h, cin_h_off, cin_T;
    float2* stats;              // [grid][J][4 * NCH epilogue warps][32] (sum, sum of squares) or nullptr
};

__device__ __forceinline__ bool rw_mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}

// Snake constants of 4 consecutive channels (see conv_pipe.cu): yb = a*x + (b + c), t = (2*alpha*a)*x + 2*alpha*b,
// out = yb - c*cos(t) with c = 1/(2*alpha)
struct RXf { float2 a01, a23, b01, b23, ta01, ta23, tb01, tb23, nc01, nc23; };

template <bool BF16>
__device__ __forceinline__ uint2 row_snake4(const float4 v, const RXf& c) {
    const float2 x01 = make_float2(v.x, v.y), x23 = make_float2(v.z, v.w);
    float2 y01 = ffma2(c.a01, x01, c.b01), y23 = ffma2(c.a23, x23, c.b23);
    const float2 t01 = ffma2(c.ta01, x01, c.tb01), t23 = ffma2(c.ta23, x23, c.tb23);
    const float2 s01 = make_float2(__cosf(t01.x), __cosf(t01.y)), s23 = make_float2(__cosf(t23.x), __cosf(t23.y));
    y01 = ffma2(c.nc01, s01, y01);
    y23 = ffma2(c.nc23, s23, y23);
    return make_uint2(pack16(y01.x, y01.y, BF16 ? 1 : 0), pack16(y23.x, y23.y, BF16 ? 1 : 0));
}

// sum over the 32 lanes of v[c] for every c; lane l returns the total of column l (fixed order -> deterministic)
__device__ __forceinline__ float row_reduce_scatter32(float (&v)[32], int lane) {
#define RW_STAGE(OFF, N)                                                            \
    {                                                                               \
        const bool up = (lane & OFF) != 0;                                          \
        _Pragma("unroll") for (int i = 0; i < N; ++i) {                             \
            const float send = up ? v[i] : v[i + N];                                \
            const float keep = up ? v[i + N] : v[i];                                \
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, OFF);                  \
        }                                                                           \
    }
    RW_STAGE(16, 16)
    RW_STAGE(8, 8)
    RW_STAGE(4, 4)
    RW_STAGE(2, 2)
    RW_STAGE(1, 1)
#undef RW_STAGE
    return v[0];
}


__device__ __forceinline__ int row_cta_start(const RowStatsInfo& s, int c) { return c * s.tq + (c < s.tr ? c : s.tr); }
__device__ __forceinline__ int row_cta_of(const RowStatsInfo& s, int t) {
    const int big = s.tr * (s.tq + 1);
    return t < big ? t / (s.tq + 1) : s.tr + (t - big) / s.tq;
}

// AdaIN coefficients of (utterance b, channel c) from the per-(CTA, utterance, epilogue warp) partials a conv_row launch wrote
// (layout: flush() of the kernel below): a = (1 + gamma) * rstd, b = beta - mean * a.  Sums in double, fixed order.
__device__ __forceinline__ void row_coef_from_partials(const float2* __restrict__ partial, const RowStatsInfo& si,
                                                       const float* __restrict__ h, int ld_h, int h_off, int T, int b, int c,
                                                       float* a_out, float* b_out) {
    const int C = si.C;
    const int c_lo = row_cta_of(si, b * si.mmt), c_hi = row_cta_of(si, (b + 1) * si.mmt - 1);
    const int chunk = c >> 5, col = c & 31;
    const int per_cta = si.nwarp / (C >> 5);
    double s = 0, ss = 0;
    for (int cta = c_lo; cta <= c_hi; ++cta) {
        const int j = b - row_cta_start(si, cta) / si.mmt;
        const float2* pp = partial + (((size_t)cta * si.J + j) * si.nwarp + chunk * per_cta) * 32 + col;
        float2 v[8];
#pragma unroll
        for (int wq = 0; wq < 8; ++wq) v[wq] = wq < per_cta ? __ldg(pp + wq * 32) : make_float2(0.f, 0.f);
#pragma unroll
        for (int wq = 0; wq < 8; ++wq) { s += (double)v[wq].x; ss += (double)v[wq].y; }
    }
    const double mean = s / (double)T;
    double var = ss / (double)T - mean * mean;
    if (var < 0) var = 0;
    const double rstd = 1.0 / sqrt(var + 1e-5);
    const double gamma = (double)h[(size_t)b * ld_h + h_off + c];
    const double beta = (double)h[(size_t)b * ld_h + h_off + C + c];
    const double ad = (1.0 + gamma) * rstd;
    *a_out = (float)ad;
    *b_out = (float)(beta - mean * ad);
}

template <bool BF16, bool X16, bool Y16, int NCH, bool BM>
__global__ void __launch_bounds__(RW_THREADS, 1)
conv_row_kernel(const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_x,
                const __grid_constant__ CUtensorMap map_xt, const __grid_constant__ CUtensorMap map_r,
                const __grid_constant__ CUtensorMap map_o, const RowParams p) {
    constexpr int C = 32 * NCH;
    constexpr int NEW = 4 * NCH;                           // epilogue warps: four TMEM lane quarters per 32-column chunk
    constexpr int NTW = 18 - NEW;                          // transform warps: 14 (C = 32) or 10 (C = 64)
    constexpr int W_EPI0 = RW_X0 + NTW;                    // first epilogue warp
    constexpr uint32_t arow = NCH == 1 ? 64u : 128u;       // bytes per operand row (K = C, 16-bit)
    constexpr uint32_t btile = (uint32_t)C * arow;         // one tap [C][C]: 2 KB / 8 KB
    constexpr uint32_t rtile = 128u * arow;                // one residual sub-tile [128][C] fp16: 8 KB / 16 KB
    constexpr int KS = C / 16;                             // K = 16 steps per tap
    constexpr uint32_t xes = X16 ? 2u : 4u;
    constexpr uint32_t xrow = (uint32_t)C * xes;           // bytes per activation row in a ring slot
    constexpr uint32_t PASS = X16 ? 256u : 512u;           // slot bytes one warp pass covers (128 elements)

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* smem_a = smem;                                              // na x [a_rows][C] 16-bit, swizzled
    uint8_t* smem_w = smem_a + (size_t)p.na * p.a_bytes;                // ntaps x [C][C] resident taps
    uint8_t* smem_i = smem_w + (size_t)p.ntaps * btile;                  // fp16 identity [C][C]
    uint8_t* smem_bt = smem_i + btile;                                   // bias_mma: fp16 bias tile [C][C] (k = 0, 1 used) + 512 B of ones
    uint8_t* smem_r = smem_bt + (BM ? btile + 1024u : 0u);      // nr x nres x [128][C] fp16 residual tiles
    uint8_t* smem_x = smem_r + (size_t)p.nr * p.nres * rtile;            // lw x xd activation slots
    const int nxs = p.lw * p.xd;
    float* bias_s = reinterpret_cast<float*>(smem_x + (size_t)nxs * p.xslot);   // [C] bias * scale
    float* coef_s = bias_s + C;                                                  // [J][2][C] in-kernel AdaIN coefficients (<= 2 KB)
    uint64_t* bars = reinterpret_cast<uint64_t*>(coef_s + (p.cin_part != nullptr ? p.J * 2 * C : 0));
    uint64_t* w_full = bars;                    // [1]
    uint64_t* a_full = bars + 1;                // [4 operand buffers]
    uint64_t* a_empty = a_full + 4;             // [4]
    uint64_t* acc_full = a_empty + 4;           // [8]
    uint64_t* acc_empty = acc_full + 8;         // [8]
    uint64_t* r_full = acc_empty + 8;           // [nr]
    uint64_t* r_empty = r_full + p.nr;          // [nr]
    uint64_t* x_full = r_empty + p.nr;          // [nxs]
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(x_full + nxs);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    // this CTA's contiguous range of macro tiles
    const int cta = blockIdx.x;
    const int m_lo = cta * p.tq + (cta < p.tr ? cta : p.tr);
    const int m_n = p.tq + (cta < p.tr ? 1 : 0);
    const int sub_rows = p.sub * 128;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&map_b);
        prefetch_tmap(&map_x);
        prefetch_tmap(&map_xt);
        if (p.nres >= 1) prefetch_tmap(&map_r);
        if (p.nres >= 2) prefetch_tmap(&map_o);
        mbar_init(w_full, 1);
        // operand buffers are handed over per macro tile: filled by its nblk blocks, emptied by the MMA of its last sub-tile
        for (int i = 0; i < p.na; ++i) {
            mbar_init(&a_full[i], (uint32_t)p.nblk);
            mbar_init(&a_empty[i], 1u);
        }
        for (int i = 0; i < 8; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], (uint32_t)(4 * NCH));   // the warps that drain one accumulator
        }
        for (int i = 0; i < p.nr; ++i) {
            mbar_init(&r_full[i], 1);
            mbar_init(&r_empty[i], 1);
        }
        for (int i = 0; i < nxs; ++i) mbar_init(&x_full[i], 1);
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                     "r"((uint32_t)p.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // fp16 identity tile in the K-major swizzled B layout: element (n, k = n) of row n
    for (uint32_t i = threadIdx.x; i < btile / 16; i += blockDim.x) reinterpret_cast<uint4*>(smem_i)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (BM) {
        for (uint32_t i = threadIdx.x; i < btile / 16; i += blockDim.x) reinterpret_cast<uint4*>(smem_bt)[i] = make_uint4(0u, 0u, 0u, 0u);
        // one 8-row group of fp16 ones: the A descriptor of the bias MMA has a zero group stride, all 16 row groups read these 512 B
        for (uint32_t i = threadIdx.x; i < 512u / 16; i += blockDim.x)
            reinterpret_cast<uint4*>(smem_bt + btile)[i] = make_uint4(0x3C003C00u, 0x3C003C00u, 0x3C003C00u, 0x3C003C00u);
    }
    __syncthreads();
    if (threadIdx.x < C) {
        const uint32_t n = threadIdx.x;
        const uint32_t sw = NCH == 1 ? ((n >> 1) & 3u) : (n & 7u);
        const uint32_t off = n * arow + (((n >> 3) ^ sw) << 4) + (n & 7u) * 2u;
        *reinterpret_cast<uint16_t*>(smem_i + off) = 0x3C00u;            // fp16 1.0
        bias_s[n] = (p.bias != nullptr ? p.bias[n] : 0.f) * p.scale;
        if (BM) {
            // row n of the K-major bias tile: (hi, lo) at k = 0, 1 -- 16-byte chunk 0 of the row, at its swizzled position
            const float bv = bias_s[n];
            const __half hi = __float2half_rn(bv);
            const __half lo = __float2half_rn(bv - __half2float(hi));
            const __half2 pr = __halves2half2(hi, lo);
            *reinterpret_cast<uint32_t*>(smem_bt + n * arow + ((0u ^ sw) << 4)) = *reinterpret_cast<const uint32_t*>(&pr);
        }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;
    pdl_trigger();
    pdl_wait();
    if (p.cin_part != nullptr) {
        // the AdaIN coefficients of this CTA's utterances, before the roles split (all 96 registers, nothing of the hot loops live):
        // one (utterance, channel) per thread, ~24 partials each from L2
        const int b_lo = m_lo / p.mmt, b_hi = (m_lo + m_n - 1) / p.mmt;
        for (int idx = threadIdx.x; idx < (b_hi - b_lo + 1) * C; idx += blockDim.x) {
            const int jj = idx / C, cc = idx - jj * C;
            float av, bv;
            row_coef_from_partials(p.cin_part, p.cin_si, p.cin_h, p.cin_ld_h, p.cin_h_off, p.cin_T, b_lo + jj, cc, &av, &bv);
            coef_s[(jj * 2 + 0) * C + cc] = av;
            coef_s[(jj * 2 + 1) * C + cc] = bv;
        }
        __syncthreads();
    }
    // register split (the kernel launches with 96 per thread): the two epilogue warpgroups (warps 12-19) keep a whole 32-column
    // accumulator chunk plus 64 statistics registers, everybody else gives 16 back:  3 x 128 x 80 + 2 x 128 x 120 = 640 x 96
    // (each setmaxnreg dominates the code of its roles, so ptxas allocates the two regions with their own budgets)
    if (warp < W_EPI0) {
    // 640 x 96 = (16 x 32) x 88 + 128 x 120 (C = 32)  =  (12 x 32) x 80 + 256 x 120 (C = 64)
    if (NCH == 1) asm volatile("setmaxnreg.dec.sync.aligned.u32 88;" ::: "memory");
    else asm volatile("setmaxnreg.dec.sync.aligned.u32 80;" ::: "memory");
    if (warp == 0) {
        // ===== producer: resident weights, then the residual-tile queue (activations are loaded by their consumers) =====
        if (elect_one_sync()) {
            mbar_expect_tx(w_full, (uint32_t)p.ntaps * btile);
            for (int w = 0; w < p.ntaps; ++w) tma_load_3d(smem_w + (size_t)w * btile, &map_b, w_full, 0, 0, w);
            if (p.nres != 0) {
                // (macro tile, sub-tile) -> stage
                int r_b = m_lo / p.mmt, r_mm = m_lo - r_b * p.mmt;
                uint32_t r_stage = 0, r_par = 0;
                const uint32_t r_tx = (uint32_t)p.nres * rtile;
                for (int r_m = 0; r_m < m_n; ++r_m) {
                    for (int r_s = 0; r_s < p.sub && r_mm * sub_rows + r_s * 128 < p.M; ++r_s) {
                        mbar_wait(&r_empty[r_stage], r_par ^ 1u);
                        uint8_t* dst = smem_r + (size_t)r_stage * p.nres * rtile;
                        mbar_expect_tx(&r_full[r_stage], r_tx);
                        const int row = r_mm * sub_rows + r_s * 128;
                        tma_load_3d(dst, &map_r, &r_full[r_stage], 0, row, r_b);
                        if (p.nres == 2) tma_load_3d(dst + rtile, &map_o, &r_full[r_stage], 0, row, r_b);
                        if (++r_stage == (uint32_t)p.nr) { r_stage = 0; r_par ^= 1u; }
                    }
                    if (++r_mm == p.mmt) { r_mm = 0; ++r_b; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (elect_one_sync()) {
            const uint32_t idesc = umma_idesc(128, C, BF16 ? 1 : 0);
            const uint32_t idesc_id = umma_idesc(128, C, 0);              // fp16 residual x fp16 identity
            const uint32_t dhi = NCH == 1 ? ((512u >> 4) | (1u << 14) | (4u << 29)) : kDescHi;
            const uint32_t a_lo0 = desc_lo(smem_u32(smem_a));
            const uint32_t a_buf_step = (uint32_t)p.a_bytes >> 4;
            const uint32_t w_lo0 = desc_lo(smem_u32(smem_w));
            const uint32_t i_lo = desc_lo(smem_u32(smem_i));
            const uint32_t bt_lo = desc_lo(smem_u32(smem_bt)), ones_lo = desc_lo(smem_u32(smem_bt + btile));
            const uint32_t r_lo0 = desc_lo(smem_u32(smem_r));
            const uint32_t r_stage_step = ((uint32_t)p.nres * rtile) >> 4;
            const uint32_t row_step = (uint32_t)(p.tap_step * (int)(arow >> 4));
            mbar_wait(w_full, 0);
            tc_fence_after();
            uint32_t sc = 0;                            // sub-tile counter -> accumulator sc % nacc
            uint32_t r_stage = 0, r_par = 0;
            int b = m_lo / p.mmt, mm = m_lo - b * p.mmt;
            uint32_t buf = 0, buf_par = 0;              // operand buffer of macro tile mc: mc % na, fill parity (mc / na) & 1
            for (int mc = 0; mc < m_n; ++mc) {
                for (int s = 0; s < p.sub; ++s) {
                    // the buffer is waited for exactly once per fill (a parity wait only tells adjacent phases apart) and handed
                    // back also when its last sub-tiles lie past the end of the utterance and contract nothing
                    if (s == 0) mbar_wait(&a_full[buf], buf_par);
                    tc_fence_after();
                    if (mm * sub_rows + s * 128 >= p.M) {
                        if (s == p.sub - 1) umma_commit(&a_empty[buf]);
                        continue;
                    }
                    const uint32_t acc = sc & (uint32_t)(p.nacc - 1);
                    const uint32_t d_tmem = tmem_base + acc * (uint32_t)C;
                    mbar_wait(&acc_empty[acc], ((sc >> p.nacc_log2) & 1u) ^ 1u);
                    tc_fence_after();
                    uint32_t accum = 0;
                    if (BM) {
                        // A: the ones group, SBO = 0 (same swizzle mode as the other operands); B: the bias tile, k-step 0
                        umma_f16_lohi2(d_tmem, ones_lo, (1u << 14) | (4u << 29), bt_lo, dhi, idesc_id, 0u);
                        accum = 1u;
                    }
                    if (p.nres) {
                        mbar_wait(&r_full[r_stage], r_par);
                        tc_fence_after();
                        uint32_t r_lo = r_lo0 + r_stage * r_stage_step;
                        for (int src = 0; src < p.nres; ++src, r_lo += rtile >> 4) {
#pragma unroll
                            for (int ks = 0; ks < KS; ++ks) {
                                umma_f16_lohi(d_tmem, r_lo + 2u * ks, i_lo + 2u * ks, dhi, idesc_id, accum);
                                accum = 1u;
                            }
                        }
                        umma_commit(&r_empty[r_stage]);
                        if (++r_stage == (uint32_t)p.nr) { r_stage = 0; r_par ^= 1u; }
                    }
                    uint32_t a_lo = a_lo0 + buf * a_buf_step + (uint32_t)(s * 128 + p.a_row0) * (arow >> 4);
                    uint32_t b_lo = w_lo0;
                    for (int j = 0; j < p.ntaps; ++j) {
#pragma unroll
                        for (int ks = 0; ks < KS; ++ks) {
                            umma_f16_lohi(d_tmem, a_lo + 2u * ks, b_lo + 2u * ks, dhi, idesc, accum);
                            accum = 1u;
                        }
                        a_lo += row_step;
                        b_lo += btile >> 4;
                    }
                    umma_commit(&acc_full[acc]);
                    if (s == p.sub - 1) umma_commit(&a_empty[buf]);
                    ++sc;
                }
                if (++buf == (uint32_t)p.na) { buf = 0; buf_par ^= 1u; }
                if (++mm == p.mmt) { mm = 0; ++b; }
            }
        }
    } else {
        // ===== transform: activation block -> AdaIN affine + Snake -> swizzled 16-bit operand rows =====
        const int tw = warp - RW_X0;
        if (tw < p.lw) {
            constexpr int lpr_shift = NCH == 1 ? 3 : 4;             // lanes per row: 8 or 16
            constexpr int rpp = 32 >> lpr_shift;                    // rows per pass: 4 or 2
            constexpr int BROWS = 8 * rpp;                          // rows per batch of 8 passes: 32 or 16
            const int rl = lane >> lpr_shift;
            const int c4 = (lane & ((1 << lpr_shift) - 1)) * 4;
            const uint32_t smem_a_u32 = smem_u32(smem_a);
            const uint32_t smem_x_u32 = smem_u32(smem_x);
            const uint32_t cidx = (uint32_t)(c4 >> 3), csub = (uint32_t)(c4 & 4) * 2u;
            uint32_t aoff[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const uint32_t Rr = (uint32_t)(rl + u * rpp);
                const uint32_t sw = NCH == 1 ? ((Rr >> 1) & 3u) : (Rr & 7u);
                aoff[u] = Rr * arow + ((cidx ^ sw) << 4) + csub;
            }
            // this warp's blocks: g = tw, tw + lw, ... -> (macro tile mi of this CTA, blk); two cursors walk them, the load
            // cursor xd blocks ahead of the compute cursor
            const int b0 = m_lo / p.mmt, mm0 = m_lo - b0 * p.mmt;
            int mi = 0, blk = tw, b = b0, mm = mm0;                 // compute cursor
            while (blk >= p.nblk) { blk -= p.nblk; ++mi; if (++mm == p.mmt) { mm = 0; ++b; } }
            int l_mi = mi, l_blk = blk, l_b = b, l_mm = mm;         // load cursor
            uint32_t l_i = 0;                                       // ring slot the next load goes to
            auto issue_load = [&]() {                               // lane 0 only; the slot is free (this warp consumed it)
                const uint32_t slot = (uint32_t)tw * (uint32_t)p.xd + l_i;
                const bool tail = (l_blk == p.nblk - 1);
                const uint32_t nrows = tail ? (uint32_t)p.tail_rows : (uint32_t)p.R;
                mbar_expect_tx(&x_full[slot], nrows * xrow);
                tma_load_3d(smem_x + (size_t)slot * p.xslot, tail ? &map_xt : &map_x, &x_full[slot], 0,
                            l_mm * sub_rows + p.halo_min + l_blk * p.R, l_b);
            };
            auto advance_load = [&]() {
                if (++l_i == (uint32_t)p.xd) l_i = 0;
                l_blk += p.lw;
                while (l_blk >= p.nblk) { l_blk -= p.nblk; ++l_mi; if (++l_mm == p.mmt) { l_mm = 0; ++l_b; } }
            };
            for (int i = 0; i < p.xd; ++i) {                        // prologue: fill the ring
                if (l_mi < m_n && lane == 0) issue_load();
                if (l_mi < m_n) advance_load();
            }
            uint32_t xi = 0, xpar = 0;                              // ring cursor of the compute side
            int cached_b = -1;
            RXf cf;
            const int cld = p.cin_part != nullptr ? C : p.coef_ld;
            const float* cbase = p.cin_part != nullptr ? coef_s - (ptrdiff_t)(m_lo / p.mmt) * 2 * C : p.coef;
            while (mi < m_n) {
                if (b != cached_b) {
                    // utterance b: from the coefficient buffer, or from the table this CTA computed (generic loads either way)
                    const float* ca = cbase + (ptrdiff_t)b * 2 * cld;
                    const float4 a4 = *reinterpret_cast<const float4*>(ca + c4);
                    const float4 b4 = *reinterpret_cast<const float4*>(ca + cld + c4);
                    const float4 al = __ldg(reinterpret_cast<const float4*>(p.alpha + c4));
                    const float4 c = make_float4(__fdividef(0.5f, al.x), __fdividef(0.5f, al.y), __fdividef(0.5f, al.z), __fdividef(0.5f, al.w));
                    cf.a01 = make_float2(a4.x, a4.y); cf.a23 = make_float2(a4.z, a4.w);
                    cf.ta01 = make_float2(2.f * al.x * a4.x, 2.f * al.y * a4.y); cf.ta23 = make_float2(2.f * al.z * a4.z, 2.f * al.w * a4.w);
                    cf.tb01 = make_float2(2.f * al.x * b4.x, 2.f * al.y * b4.y); cf.tb23 = make_float2(2.f * al.z * b4.z, 2.f * al.w * b4.w);
                    cf.b01 = make_float2(b4.x + c.x, b4.y + c.y); cf.b23 = make_float2(b4.z + c.z, b4.w + c.w);
                    cf.nc01 = make_float2(-c.x, -c.y); cf.nc23 = make_float2(-c.z, -c.w);
                    cached_b = b;
                }
                const uint32_t fill = (uint32_t)mi / (uint32_t)p.na, buf = (uint32_t)mi - fill * (uint32_t)p.na;
                const uint32_t slot = (uint32_t)tw * (uint32_t)p.xd + xi;
                const int r0 = blk * p.R;                                        // first operand row of this block
                const int nvalid = (blk == p.nblk - 1) ? p.tail_rows : p.R;      // rows the TMA box really loaded
                const int t0 = mm * sub_rows + p.halo_min + r0;                  // time index of operand row r0
                mbar_wait_warp(&x_full[slot], xpar);
                mbar_wait_warp(&a_empty[buf], (fill & 1u) ^ 1u);
                uint32_t xaddr = smem_x_u32 + slot * (uint32_t)p.xslot + (uint32_t)rl * xrow + (uint32_t)c4 * xes;
                uint32_t abase = smem_a_u32 + buf * (uint32_t)p.a_bytes + (uint32_t)r0 * arow;
                // whole batches: rows past nvalid read stale slot bytes and land in slack operand rows no MMA reads
                for (int rb = 0; rb < nvalid; rb += BROWS, xaddr += 8 * PASS, abase += (uint32_t)BROWS * arow) {
                    float4 v[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (X16) v[u] = unpack16x4(lds64(xaddr + (uint32_t)u * PASS), 0);
                        else v[u] = lds128(xaddr + (uint32_t)u * PASS);
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const uint2 o = row_snake4<BF16>(v[u], cf);
                        sts64(abase + aoff[u], o.x, o.y);
                    }
                }
                if (t0 < 0 || t0 + nvalid > p.M) {
                    // zero padding of the convolution (after the activation): rows outside [0, M) of the utterance
                    __syncwarp();
                    const uint32_t abuf = smem_a_u32 + buf * (uint32_t)p.a_bytes + csub;
                    for (int r = rl; r < nvalid; r += rpp) {
                        const int t = t0 + r;
                        if (t < 0 || t >= p.M) {
                            const uint32_t Rr = (uint32_t)(r0 + r);
                            const uint32_t sw = NCH == 1 ? ((Rr >> 1) & 3u) : (Rr & 7u);
                            sts64(abuf + Rr * arow + ((cidx ^ sw) << 4), 0u, 0u);
                        }
                    }
                }
                fence_proxy_async();
                __syncwarp();                                        // every lane has read the slot and written its rows
                if (lane == 0) {
                    mbar_arrive(&a_full[buf]);
                    if (l_mi < m_n) issue_load();                    // refill the slot just consumed (l_i == xi)
                }
                if (l_mi < m_n) advance_load();
                if (++xi == (uint32_t)p.xd) { xi = 0; xpar ^= 1u; }
                blk += p.lw;
                while (blk >= p.nblk) { blk -= p.nblk; ++mi; if (++mm == p.mmt) { mm = 0; ++b; } }
            }
        }
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 120;" ::: "memory");
        // ===== epilogue: one thread = one output row; statistics in registers across tiles =====
        const int ew = warp - W_EPI0;                     // 0 .. NEW-1
        const int q = warp & 3;                           // TMEM lane quarter this warp may access
        const int ch = ew >> 2;                           // 32-column chunk this warp owns
        const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ch * 32);
        const uint32_t bias_u32 = smem_u32(bias_s) + (uint32_t)(ch * 32) * 4u;
        const float2 sc2 = make_float2(p.scale, p.scale);
        constexpr size_t yes = Y16 ? 2 : 4;               // bytes per output element
        const size_t sub_bytes = (size_t)128 * p.ld_y * yes;
        float2 s1[16], s2[16];                            // (sum, sum of squares) of channel pairs (2i, 2i + 1) of this row
#pragma unroll
        for (int i = 0; i < 16; ++i) { s1[i] = make_float2(0.f, 0.f); s2[i] = make_float2(0.f, 0.f); }
        const int b_first = m_lo / p.mmt;
        int b = b_first, mm = m_lo - b_first * p.mmt;
        uint32_t sc = 0;
        auto flush = [&](int bb) {
            if (p.stats != nullptr) {
                float a1[32];
#pragma unroll
                for (int i = 0; i < 16; ++i) { a1[2 * i] = s1[i].x; a1[2 * i + 1] = s1[i].y; }
                const float t1 = row_reduce_scatter32(a1, lane);
#pragma unroll
                for (int i = 0; i < 16; ++i) { a1[2 * i] = s2[i].x; a1[2 * i + 1] = s2[i].y; }
                const float t2 = row_reduce_scatter32(a1, lane);
                p.stats[(((size_t)cta * p.J + (bb - b_first)) * NEW + ew) * 32 + lane] = make_float2(t1, t2);
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) { s1[i] = make_float2(0.f, 0.f); s2[i] = make_float2(0.f, 0.f); }
        };
        // BM (a kernel variant): the accumulator already holds conv + bias and scale is 1, so a row goes from TMEM to the
        // statistics and the store with no arithmetic of its own
        for (int mc = 0; mc < m_n; ++mc) {
            int m = mm * sub_rows + q * 32 + lane;                              // output row of this thread in sub-tile 0
            uint8_t* yrow = reinterpret_cast<uint8_t*>(p.y) + (((size_t)b * p.M + (size_t)m) * p.ld_y + ch * 32) * yes;
            for (int s = 0; s < p.sub && mm * sub_rows + s * 128 < p.M; ++s, ++sc, m += 128, yrow += sub_bytes) {
                const uint32_t acc = sc & (uint32_t)(p.nacc - 1);
                mbar_wait_warp(&acc_full[acc], (sc >> p.nacc_log2) & 1u);
                tc_fence_after();
                float v[32];
                tmem_ld32(t_lane + acc * (uint32_t)C, v);
                // the accumulator chunk is in registers: hand it back to the MMA warp
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[acc]);
                if (m < p.M) {
                    float2 o[16];
                    if (BM) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) o[i] = make_float2(v[2 * i], v[2 * i + 1]);
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float4 bs = lds128(bias_u32 + (uint32_t)(i * 16));
                            o[2 * i] = ffma2(make_float2(v[4 * i], v[4 * i + 1]), sc2, make_float2(bs.x, bs.y));
                            o[2 * i + 1] = ffma2(make_float2(v[4 * i + 2], v[4 * i + 3]), sc2, make_float2(bs.z, bs.w));
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        s1[i] = fadd2(s1[i], o[i]);
                        s2[i] = ffma2(o[i], o[i], s2[i]);
                    }
                    if (Y16) {
                        uint4* dst = reinterpret_cast<uint4*>(yrow);
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            dst[i] = make_uint4(pack16(o[4 * i].x, o[4 * i].y, 0), pack16(o[4 * i + 1].x, o[4 * i + 1].y, 0),
                                                pack16(o[4 * i + 2].x, o[4 * i + 2].y, 0), pack16(o[4 * i + 3].x, o[4 * i + 3].y, 0));
                    } else {
                        float4* dst = reinterpret_cast<float4*>(yrow);
#pragma unroll
                        for (int i = 0; i < 8; ++i) dst[i] = make_float4(o[2 * i].x, o[2 * i].y, o[2 * i + 1].x, o[2 * i + 1].y);
                    }
                }
                __syncwarp();                              // re-converge before the next .aligned TMEM load
            }
            if (++mm == p.mmt) {
                flush(b);
                mm = 0;
                ++b;
            }
        }
        if (mm != 0) flush(b);                            // the range ended inside utterance b
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols)
                     : "memory");
    }
}

// ---------------------------------------------------------------- coefficients from the per-(CTA, utterance, warp) partials
// grid (B), block 256: thread (c, slice) sums every `nsl`-th partial of channel c in double, then a fixed-order tree over the
// slices.  The CTAs that hold partials of utterance b are those whose macro-tile range meets [b*mmt, (b+1)*mmt).
__global__ void __launch_bounds__(256)
adain_coef_row_kernel(const float2* __restrict__ partial, const RowStatsInfo si, const float* __restrict__ h, int ld_h, int h_off,
                      float* __restrict__ coef, int T, int Cpad) {
    __shared__ double ssum[256], ssq[256];
    pdl_trigger();
    pdl_wait();
    const int C = si.C;
    const int nsl = 256 / C;                     // slices per channel: 8 (C = 32) or 4 (C = 64)
    const int c = threadIdx.x % C, sl = threadIdx.x / C;
    const int b = blockIdx.x;
    const int c_lo = row_cta_of(si, b * si.mmt), c_hi = row_cta_of(si, (b + 1) * si.mmt - 1);
    const int chunk = c >> 5, col = c & 31;
    const int per_cta = si.nwarp / (C >> 5);     // epilogue warps that hold partials of this column chunk: 8 (C = 32) or 4 (C = 64)
    const int nparts = (c_hi - c_lo + 1) * per_cta;
    double s = 0, ss = 0;
    for (int i = sl; i < nparts; i += nsl) {
        const int cta = c_lo + i / per_cta, wq = i - (i / per_cta) * per_cta;
        const int j = b - row_cta_start(si, cta) / si.mmt;
        const float2 v = __ldg(partial + (((size_t)cta * si.J + j) * si.nwarp + chunk * per_cta + wq) * 32 + col);
        s += (double)v.x;
        ss += (double)v.y;
    }
    ssum[threadIdx.x] = s;
    ssq[threadIdx.x] = ss;
    __syncthreads();
    if (sl != 0) return;
    for (int i = 1; i < nsl; ++i) {
        s += ssum[i * C + c];
        ss += ssq[i * C + c];
    }
    const double mean = s / (double)T;
    double var = ss / (double)T - mean * mean;
    if (var < 0) var = 0;
    const double rstd = 1.0 / sqrt(var + 1e-5);
    const double gamma = (double)h[(size_t)b * ld_h + h_off + c];
    const double beta = (double)h[(size_t)b * ld_h + h_off + C + c];
    const double ad = (1.0 + gamma) * rstd;
    coef[((size_t)b * 2 + 0) * Cpad + c] = (float)ad;
    coef[((size_t)b * 2 + 1) * Cpad + c] = (float)(beta - mean * ad);
}

// ---------------------------------------------------------------- host side
int make_weight_map(CUtensorMap* map, int is_bf16, const void* w16, int cin_pad, int cout_pad, int ktaps, int bn);
int make_weight_map_k32(CUtensorMap* map, int is_bf16, const void* w16, int cin_pad, int cout_pad, int ktaps, int bn);
int make_map_3d_sw(CUtensorMap* map, int dtype, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                   uint64_t stride2_bytes, uint32_t b0, uint32_t b1, int swizzle_bytes);

static int row_num_sms() { return device_num_sms(); }

static bool row_geometry_ok(const ConvArgs& a) {
    if (a.in_stride != 1 || a.mirror || a.res_shift != 0 || a.phases != 1) return false;
    if (a.out_stride != 1 || a.out_pad != 0 || a.tap_step <= 0 || a.M != a.Tout || a.Tin != a.Tout) return false;
    if (!(a.Cin == 32 || a.Cin == 64) || a.Cout != a.Cin) return false;
    if (a.w16 == nullptr || a.w16_cin_pad != 64 || a.w16_cout_pad != a.Cout) return false;
    if (a.ld_x != a.Cin) return false;
    if (a.res != nullptr && (!a.res16 || a.ld_res != a.Cout)) return false;            // residual only as an fp16 tile
    if (a.accumulate && !(a.res != nullptr && a.acc_src != nullptr && a.acc16)) return false;   // old values only as an fp16 tile
    if (!a.accumulate && a.acc_src != nullptr) return false;
    if (a.ld_y % 8 != 0) return false;
    const int span = (a.ntaps - 1) * a.tap_step;
    return span <= 64 && a.in_off <= 0 && a.in_off + span >= 0;
}

// geometry + shared-memory plan; false if it does not fit
static bool row_plan(const ConvArgs& a, RowParams& p, size_t* smem_out, int* grid_out) {
    memset(&p, 0, sizeof(p));
    const int C = a.Cin, nch = C / 32;
    const int arow = nch == 1 ? 64 : 128;
    const int btile = C * arow, rtile = 128 * arow;
    const int span = (a.ntaps - 1) * a.tap_step;
    p.B = a.B; p.M = a.M; p.ntaps = a.ntaps; p.tap_step = a.tap_step;
    p.halo_min = a.in_off; p.a_row0 = 0;
    p.nres = (a.res != nullptr ? 1 : 0) + (a.accumulate ? 1 : 0);
    p.nacc = nch == 1 ? 8 : 4;
    p.nacc_log2 = nch == 1 ? 3 : 2;
    p.tmem_cols = 256;
    // the bias through the tensor core: 32-channel layers with scale 1 (every conv of a resblock but the last of a stage); the
    // 64-channel layers run 8 epilogue warps and have no shared memory to spare for an 8 KB bias tile
    p.bias_mma = (nch == 1 && a.bias != nullptr && a.scale == 1.f) ? 1 : 0;
    const int ntw = 18 - 4 * nch;
    const int xes = a.x16in ? 2 : 4;
    const int brows = nch == 1 ? 32 : 16;                  // rows per transform batch
    const int64_t budget = 224 * 1024 + (p.bias_mma ? 2048 : 0);      // + 1 KB of alignment slack = 227 KB at most
    bool ok = false;
    // 4 KB activation blocks (two transform batches per barrier round trip: 2 KB blocks measured 0.36 vs 0.30 ms on the
    // 64-channel k = 3 layer) with the largest macro tile that fits (the halo is transformed once per macro tile), then the
    // deepest rings; 2 KB blocks only where nothing else fits
    for (int slot_bytes = 4096; slot_bytes >= 2048 && !ok; slot_bytes >>= 1) {
        for (int sub = 4; sub >= 1 && !ok; sub >>= 1) {
            if (tune().row_sub && sub != tune().row_sub) continue;
            const int mr = sub * 128 + span;
            int R = slot_bytes / (C * xes);
            R = R / brows * brows;
            if (R < brows) R = brows;
            const int nblk = cdiv(mr, R);
            const int tail = mr - (nblk - 1) * R;
            const int64_t a_bytes = ((int64_t)nblk * R * arow + 1023) & ~(int64_t)1023;
            const int xslot = R * C * xes;
            // three operand buffers for single-sub-tile macro tiles when they fit (the MMA of tile m otherwise gates the
            // transform of tile m + 2 after every 128 rows)
            for (int na = sub == 1 ? 3 : 2; na >= 2 && !ok; --na) {
                const int lw_max = na * nblk < ntw ? na * nblk : ntw;
                const int64_t fixed = na * a_bytes + (int64_t)a.ntaps * btile + btile + 4096 + (p.bias_mma ? btile + 1024 : 0);
                const int nr_max = p.nres ? 4 : 0, nr_min = p.nres ? 2 : 0;
                // as many transform warps as have a ring (at least 10; 7 for the smallest macro tile) with the deepest rings that fit
                for (int lw = lw_max; lw >= (lw_max < 10 ? lw_max : (sub == 1 ? 7 : 10)) && !ok; --lw) {
                    for (int nr = nr_max; nr >= nr_min && !ok; --nr) {
                        for (int xd = 3; xd >= 2 && !ok; --xd) {
                            const int64_t tot = fixed + (int64_t)nr * p.nres * rtile + (int64_t)lw * xd * xslot;
                            if (tot <= budget) {
                                p.sub = sub; p.R = R; p.nblk = nblk; p.tail_rows = tail; p.xslot = xslot; p.a_bytes = (int)a_bytes;
                                p.lw = lw; p.xd = xd; p.nr = nr; p.na = na;
                                *smem_out = (size_t)tot + 1024;
                                ok = true;
                            }
                        }
                    }
                }
            }
        }
    }
    if (!ok) return false;
    p.mmt = cdiv(a.M, p.sub * 128);
    const int64_t nt = (int64_t)a.B * p.mmt;
    int grid = row_num_sms();
    if (grid > RW_MAXGRID) grid = RW_MAXGRID;
    if (grid > nt) grid = (int)nt;
    p.tq = (int)(nt / grid); p.tr = (int)(nt % grid);
    p.J = (p.tq + 1 + p.mmt - 1) / p.mmt + 1;
    p.bias = a.bias; p.scale = a.scale;
    p.y = a.y; p.ld_y = a.ld_y;
    *grid_out = grid;
    return true;
}

bool conv_row_can_launch(const ConvArgs& a) {
    if (!row_geometry_ok(a)) return false;
    RowParams p;
    size_t smem;
    int grid;
    return row_plan(a, p, &smem, &grid);
}

// dispatch policy: small problems (one-sentence latency: fewer than 4 macro tiles per SM) stay on conv_pipe.cu, whose 128-row
// tiles spread them over more SMs.  Tune::row_always drops that threshold (geometry and plan still apply), so the decoder's
// reference fixtures, a few utterances long, can run every 32 / 64-channel resblock conv on this kernel.
bool conv_row_supported(const ConvArgs& a) {
    if (!row_geometry_ok(a)) return false;
    RowParams p;
    size_t smem;
    int grid;
    if (!row_plan(a, p, &smem, &grid)) return false;
    return tune().row_always || (int64_t)a.B * p.mmt >= 4 * (int64_t)row_num_sms();
}

// bytes of the statistics buffer a conv_row launch of this geometry writes (upper bound over devices with <= RW_MAXGRID SMs)
int64_t conv_row_stats_bytes(int B, int T, int C) {
    // J <= B + 1 slots per CTA; 8 epilogue warps x 32 columns x float2
    const int64_t per_cta = (int64_t)(B + 1) * 8 * 32 * 8;
    (void)T; (void)C;
    return (int64_t)RW_MAXGRID * per_cta;
}

// can a launch of this geometry compute its AdaIN coefficients itself (RowCoefSrc)?  The table of its utterances must fit 2 KB
bool conv_row_inline_coef_ok(const ConvArgs& a) {
    if (!row_geometry_ok(a) || tune().no_row_inline_coef) return false;
    RowParams p;
    size_t smem;
    int grid;
    if (!row_plan(a, p, &smem, &grid)) return false;
    return p.J * 2 * a.Cin * 4 <= 2048;
}

int launch_conv_row(const ConvArgs& a, const float* coef, int coef_ld, int act, const float* alpha, void* stats_out,
                    RowStatsDesc* desc, cudaStream_t st, const RowCoefSrc* src) {
    RowParams p;
    size_t smem = 0;
    int grid = 0;
    ST2_REQUIRE(row_geometry_ok(a) && row_plan(a, p, &smem, &grid), "conv_row: unsupported geometry");
    ST2_REQUIRE(act == ACT_SNAKE && alpha != nullptr, "conv_row: only the Snake transform is built");
    p.coef = coef; p.coef_ld = coef_ld; p.alpha = alpha;
    p.cin_part = nullptr;
    if (src != nullptr) {
        ST2_REQUIRE(src->partial != nullptr && src->h != nullptr && src->desc.C == a.Cin && p.J * 2 * a.Cin * 4 <= 2048,
                    "conv_row: in-kernel coefficients need row partials of the same channel count and <= 2 KB of them per CTA");
        p.cin_part = (const float2*)src->partial;
        p.cin_si.grid = src->desc.grid; p.cin_si.J = src->desc.J; p.cin_si.nwarp = src->desc.nwarp; p.cin_si.mmt = src->desc.mmt;
        p.cin_si.tq = src->desc.tq; p.cin_si.tr = src->desc.tr; p.cin_si.C = src->desc.C;
        p.cin_h = src->h; p.cin_ld_h = src->ld_h; p.cin_h_off = src->h_off; p.cin_T = src->T;
    }
    p.stats = (float2*)stats_out;
    const int C = a.Cin, nch = C / 32;
    const int is_bf16 = a.fmt16 == DT_BF16 ? 1 : 0;
    CUtensorMap map_b, map_x, map_xt, map_r, map_o;
    int e = nch == 1 ? make_weight_map_k32(&map_b, is_bf16, a.w16, a.w16_cin_pad, a.w16_cout_pad, a.ntaps, C)
                     : make_weight_map(&map_b, is_bf16, a.w16, a.w16_cin_pad, a.w16_cout_pad, a.ntaps, C);
    if (e != ST2_OK) return e;
    const int xdt = a.x16in ? 2 : 0;
    const uint64_t xes = a.x16in ? 2 : 4;
    e = make_map_3d_sw(&map_x, xdt, a.x, (uint64_t)C, (uint64_t)a.Tin, (uint64_t)a.B, (uint64_t)a.ld_x * xes,
                       (uint64_t)a.Tin * a.ld_x * xes, (uint32_t)C, (uint32_t)p.R, 0);
    if (e != ST2_OK) return e;
    e = make_map_3d_sw(&map_xt, xdt, a.x, (uint64_t)C, (uint64_t)a.Tin, (uint64_t)a.B, (uint64_t)a.ld_x * xes,
                       (uint64_t)a.Tin * a.ld_x * xes, (uint32_t)C, (uint32_t)p.tail_rows, 0);
    if (e != ST2_OK) return e;
    map_r = map_x;
    map_o = map_x;
    const int sw = nch == 1 ? 64 : 128;
    if (a.res != nullptr) {
        e = make_map_3d_sw(&map_r, 2, a.res, (uint64_t)C, (uint64_t)a.Tout, (uint64_t)a.B, (uint64_t)a.ld_res * 2,
                           (uint64_t)a.Tout * a.ld_res * 2, (uint32_t)C, 128, sw);
        if (e != ST2_OK) return e;
    }
    if (a.accumulate) {
        e = make_map_3d_sw(&map_o, 2, a.acc_src, (uint64_t)C, (uint64_t)a.Tout, (uint64_t)a.B, (uint64_t)a.ld_y * 2,
                           (uint64_t)a.Tout * a.ld_y * 2, (uint32_t)C, 128, sw);
        if (e != ST2_OK) return e;
    }
    if (desc != nullptr) {
        desc->grid = grid; desc->J = p.J; desc->nwarp = 4 * nch; desc->mmt = p.mmt; desc->tq = p.tq; desc->tr = p.tr; desc->C = C;
    }
    if (tune().verbose)
        fprintf(stderr, "conv_row: C=%d taps=%d step=%d x16=%d y16=%d nres=%d sub=%d R=%d nblk=%d tail=%d na=%d lw=%d xd=%d nr=%d smem=%zu grid=%d mmt=%d tq=%d tr=%d J=%d inline=%d\n",
                C, p.ntaps, p.tap_step, a.x16in, a.y16out, p.nres, p.sub, p.R, p.nblk, p.tail_rows, p.na, p.lw, p.xd, p.nr, smem, grid, p.mmt,
                p.tq, p.tr, p.J, p.cin_part != nullptr ? 1 : 0);
    ST2_REQUIRE(stats_out == nullptr || (int64_t)grid * p.J * (4 * nch) * 32 * 8 <= conv_row_stats_bytes(a.B, a.Tout, C),
                "conv_row: statistics buffer too small");
    // the opt-in to > 48 KB of dynamic shared memory is per device: once per (device, variant)
    static bool attr_done[kMaxDevices][32] = {};
    const int dev = current_device_slot();
#define ROW_LAUNCH(BF, X, Y, N, M)                                                                                               \
    do {                                                                                                                         \
        bool& done = attr_done[dev][(M ? 16 : 0) + (BF ? 8 : 0) + (X ? 4 : 0) + (Y ? 2 : 0) + (N - 1)];                          \
        if (!done) {                                                                                                             \
            ST2_CUDA_CHECK(cudaFuncSetAttribute(conv_row_kernel<BF, X, Y, N, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); \
            done = true;                                                                                                         \
        }                                                                                                                        \
        conv_row_kernel<BF, X, Y, N, M><<<grid, RW_THREADS, smem, st>>>(map_b, map_x, map_xt, map_r, map_o, p);                  \
    } while (0)
#define ROW_LAUNCH_M(BF, X, Y, N) do { if (N == 1 && p.bias_mma) ROW_LAUNCH(BF, X, Y, N, (N == 1)); else ROW_LAUNCH(BF, X, Y, N, false); } while (0)
#define ROW_LAUNCH_Y(BF, X, N) do { if (a.y16out) ROW_LAUNCH_M(BF, X, true, N); else ROW_LAUNCH_M(BF, X, false, N); } while (0)
    const bool bf = is_bf16 != 0, x16 = a.x16in != 0;
    if (nch == 1) {
        if (bf) { if (x16) ROW_LAUNCH_Y(true, true, 1); else ROW_LAUNCH_Y(true, false, 1); }
        else { if (x16) ROW_LAUNCH_Y(false, true, 1); else ROW_LAUNCH_Y(false, false, 1); }
    } else {
        if (bf) { if (x16) ROW_LAUNCH_Y(true, true, 2); else ROW_LAUNCH_Y(true, false, 2); }
        else { if (x16) ROW_LAUNCH_Y(false, true, 2); else ROW_LAUNCH_Y(false, false, 2); }
    }
#undef ROW_LAUNCH_Y
#undef ROW_LAUNCH_M
#undef ROW_LAUNCH
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

int launch_adain_coef_row(const void* partial, const RowStatsDesc& d, const float* h, int ld_h, int h_off, float* coef, int B,
                          int T, int C, int Cpad, cudaStream_t st) {
    ST2_REQUIRE(C == d.C && (C == 32 || C == 64) && Cpad == C, "adain_coef_row: bad channel count");
    RowStatsInfo si;
    si.grid = d.grid; si.J = d.J; si.nwarp = d.nwarp; si.mmt = d.mmt; si.tq = d.tq; si.tr = d.tr; si.C = d.C;
    adain_coef_row_kernel<<<B, 256, 0, st>>>((const float2*)partial, si, h, ld_h, h_off, coef, T, Cpad);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

}  // namespace st2
