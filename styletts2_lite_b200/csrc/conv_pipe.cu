// Fully TMA-fed fused  [AdaIN affine + Snake / LeakyReLU] -> Conv1d / ConvTranspose1d (tcgen05) ->
// [bias + residual + accumulate + scale + InstanceNorm partial statistics]  kernel for sm_100a: every conv of
// AdaINResBlock1 (Modules/hifigan.py:65-74) with up to 128 channels and the generator `ups` with stride*Cout <= 256
// (:292-294, :329-334) -- 92 of the 100 fused launches of a hifigan forward; conv_fused.cu runs the rest.
//
// conv_fused.cu left three latency chains exposed (measured with its role timeline): the transform warps waited
// for whole-tile loads, the epilogue warps waited ~1.5 us for their residual rows, and one producer thread
// serialised weight and activation loads.  Here no compute warp ever touches global memory for input:
//   * activations arrive by TMA in blocks of <= 12 KB (a few equal blocks per tile, multiples of 8 rows; fp32, or fp16 for
//     the intra-block tensor of the resblocks) through a ring of `nx` slots that is independent of the tile geometry;
//     blocks are dealt round-robin to the transform warps, which work in batches of 8 row passes (8 independent 128-bit
//     loads, then 8 independent activation chains -> the Snake chain is hidden by ILP, not by occupancy);
//   * residual (+ accumulate) rows arrive by TMA as 128-byte-swizzled [128 rows x 32 ch] fp32 boxes through a ring
//     of `nr` stages; the epilogue adds them in the TMEM-drain layout and reuses the very same stage as its
//     transposition buffer, so the only global accesses of the epilogue are full-line stores;
//   * one producer thread multiplexes three independent queues (weights, activation blocks, residual boxes) with
//     non-blocking mbarrier tests, so a full weight ring never delays an activation prefetch;
//   * 2-4 operand buffers and 4 TMEM accumulators (2 for N > 128) decouple transform, MMA and epilogue; pipe_plan()
//     splits the 227 KB of shared memory between operand buffers, weights (resident or ring) and the two rings;
//   * layers that stream their weights (128 channels) run two consecutive tiles against every weight stage (p.pair).
// The activation and residual rings are plain FIFOs shared by several consumer warps.  An mbarrier parity wait only
// tells adjacent phases apart and a consumer can be two fills ahead of a slot it does not own, so the producer
// publishes the sequence number of every fill in a shared-memory word before issuing it; a consumer first sees
// "its" sequence number (the previous fill has then landed and been consumed) and only then waits on the barrier.
// ConvTranspose1d(k = taps*stride, stride): its `stride` polyphase sub-convolutions read the same input rows, so their
// weights are stacked along N (N = stride*Cout) and row m of the accumulator is exactly the `stride` consecutive output
// rows m*stride - pad ... of the channels-last tensor, i.e. a dense [M][stride*Cout] matrix at a constant element offset.
// Roles (one persistent CTA per SM): warp 0 producer, warp 1 TMEM allocator + MMA issuer, warps 2-7 transform,
// warps 8.. epilogue in groups of 4 (one TMEM lane quarter per warp): 2 groups (512 threads, 128 registers) or 3 groups
// (640 threads, 96 registers; the 32-channel layers with a residual, which are epilogue-bound).
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"
#include "tc_ptx.cuh"
#include "fused_ptx.cuh"

namespace st2 {

static constexpr int P_LW = 6;                           // transform warps
static constexpr int P_W_X0 = 2;                         // first transform warp
static constexpr int P_W_EPI0 = P_W_X0 + P_LW;           // first epilogue warp (8)
// threads: (8 + 4*EG) warps.  EG = 2 epilogue groups (512 threads, 128 registers) is the default; the 32-channel layers with
// a residual are epilogue-bound and run EG = 3 (640 threads, 96 registers): 0.53 -> 0.47 ms on the k=3 layer, while
// transform-bound layers lose with the smaller register budget.
static constexpr int P_MT = 128;                         // rows per tile
static constexpr int P_XSLOT_MAX = 12288;                 // largest activation ring slot
static constexpr int P_RBOX = P_MT * 32 * 4;             // one residual box: 128 rows x 32 fp32

struct PipeParams {
    // transform
    const float* coef; int coef_ld;
    const float* alpha; float slope;
    int Cin, kchunks, cch;      // cch: channels per K chunk (64, or 32 for 32-channel layers)
    int x16in, is_bf16, k32;
    // geometry
    int B, M, Tin, Cout;
    int ntaps, tap_step, halo_min, rows;
    int xr, nblk, tail_rows;    // activation blocks: xr rows each, nblk per (tile, chunk), the last one tail_rows
    int xslot;                  // bytes per activation ring slot (xr rows)
    int lw;                     // active transform warps = min(6, na * nblk): a warp's consecutive blocks are then at most
                                // na operand fills apart, so its a_empty parity wait is never more than one phase behind
    int bn, nt, mtiles, num_tiles;   // bn columns per accumulator; nt > 1: N passes over the operand tile (Cout = nt * bn)
    int wstages, resident, tmem_cols;
    int na, nacc, nacc_log2;    // operand (A) buffers 2..4, TMEM accumulators 2 or 4
    int eg;                     // epilogue groups of the kernel variant launched (2 or 3)
    int pair;                   // 1: the MMA warp runs two consecutive tiles against every weight stage (streamed weights,
                                //    2 K chunks, 4 operand buffers, 4 accumulators): half the weight traffic into shared memory
    int nx, nr, nres;           // ring depths; nres = residual sources per stage (0, 1, or 2 = residual + old y)
    int r16;                    // the residual tensor is fp16 (the running tensor of AdaINResBlock1): four [32 rows x 32 ch] boxes
    int o16;                    // the old values of an accumulate layer are fp16 (partial sums of a stage), same box layout
    // epilogue
    const float* bias;
    float* y; int ld_y; float scale; int y16out;   // y already shifted by -out_pad*cdiv rows for a transposed conv
    int ostride, opad, Tout, cdiv, cshift;          // output row of (m, column c): t = m*ostride + c/cdiv - opad, valid in [0,Tout); cdiv = 1 << cshift
    int a_row0;                                     // operand row of tap 0 for output row 0 of the tile
    long long ybatch;                               // elements between consecutive utterances of y
    float2* stats;              // [B][mtiles*4][Cout] (sum, sumsq) per (tile, 32-row quarter) or nullptr
};

__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
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

// tile = blockIdx.x + i*gridDim.x  ->  (b, mt), advanced without divisions
struct PTile {
    int tile, b, mt, d_b, d_mt;
    __device__ __forceinline__ void init(const PipeParams& p) {
        tile = blockIdx.x;
        b = tile / p.mtiles; mt = tile - b * p.mtiles;
        d_b = gridDim.x / p.mtiles; d_mt = gridDim.x - d_b * p.mtiles;
    }
    __device__ __forceinline__ bool valid(const PipeParams& p) const { return tile < p.num_tiles; }
    __device__ __forceinline__ void next(const PipeParams& p) {
        tile += gridDim.x;
        mt += d_mt; if (mt >= p.mtiles) { mt -= p.mtiles; ++b; }
        b += d_b;
    }
};

// per-thread transform constants for 4 consecutive channels (two packed pairs each).
// Snake: y + sin^2(alpha*y)/alpha with y = a*x + b  ==  (a*x + b + c) - c*cos(2*alpha*(a*x + b)),  c = 1/(2*alpha)
//   -> yb = a*x + (b + c);  t = (2*alpha*a)*x + 2*alpha*b;  out = yb + nc*cos(t)        (3 packed FMAs + 2 MUFU per pair)
struct PXf { float2 a01, a23, b01, b23, ta01, ta23, tb01, tb23, nc01, nc23; };

template <int ACT, bool BF16>
__device__ __forceinline__ uint2 pipe_transform4(const float4 v, const PXf& c) {
    const float2 x01 = make_float2(v.x, v.y), x23 = make_float2(v.z, v.w);
    float2 y01 = ffma2(c.a01, x01, c.b01), y23 = ffma2(c.a23, x23, c.b23);
    if (ACT == ACT_SNAKE) {
        const float2 t01 = ffma2(c.ta01, x01, c.tb01), t23 = ffma2(c.ta23, x23, c.tb23);
        const float2 s01 = make_float2(__cosf(t01.x), __cosf(t01.y)), s23 = make_float2(__cosf(t23.x), __cosf(t23.y));
        y01 = ffma2(c.nc01, s01, y01);
        y23 = ffma2(c.nc23, s23, y23);
    } else if (ACT == ACT_LRELU) {
        const float2 z01 = fmul2(y01, c.ta01), z23 = fmul2(y23, c.ta23);    // slope < 1: lrelu(y) = max(y, slope*y)
        y01 = make_float2(fmaxf(y01.x, z01.x), fmaxf(y01.y, z01.y));
        y23 = make_float2(fmaxf(y23.x, z23.x), fmaxf(y23.y, z23.y));
    }
    return make_uint2(pack16(y01.x, y01.y, BF16 ? 1 : 0), pack16(y23.x, y23.y, BF16 ? 1 : 0));
}

// Epilogue rows of one 32x32 chunk in the transposed layout: this lane owns 4 channels of rows rr + 4*it.
// o = a*scale + bias*scale, 128-byte row segments to global, running (sum, sum of squares) per channel.
template <bool FULL, bool Y16>
__device__ __forceinline__ void pipe_store_rows(uint32_t st_r0, uint32_t st_r1, float* yo, int ystep, uint32_t vmask, float2 sc2,
                                                float2 bs01, float2 bs23, float2& s1a, float2& s1b, float2& s2a, float2& s2b) {
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const float4 a = lds128(((it & 1) ? st_r1 : st_r0) + (uint32_t)(it >> 1) * 1024u);
        if (!FULL && !((vmask >> it) & 1u)) continue;
        const float2 o01 = ffma2(make_float2(a.x, a.y), sc2, bs01);
        const float2 o23 = ffma2(make_float2(a.z, a.w), sc2, bs23);
        if (Y16)   // fp16 storage of the intra-block tensor: yo is a half pointer in disguise (element offsets are the same)
            *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(yo) + (size_t)it * ystep) =
                make_uint2(pack16(o01.x, o01.y, 0), pack16(o23.x, o23.y, 0));
        else
            *reinterpret_cast<float4*>(yo + (size_t)it * ystep) = make_float4(o01.x, o01.y, o23.x, o23.y);
        s1a = fadd2(s1a, o01); s1b = fadd2(s1b, o23);
        s2a = ffma2(o01, o01, s2a); s2b = ffma2(o23, o23, s2b);
    }
}

template <int ACT, bool BF16, bool X16, int EG>
__global__ void __launch_bounds__((P_W_EPI0 + 4 * EG) * 32, 1)
conv_pipe_kernel(const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_x,
                 const __grid_constant__ CUtensorMap map_xt, const __grid_constant__ CUtensorMap map_r,
                 const __grid_constant__ CUtensorMap map_o, const PipeParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const uint32_t arow = p.k32 ? 64u : 128u;                      // bytes per operand row
    const uint32_t a_bytes = ((uint32_t)p.rows * arow + 1023u) & ~1023u;
    const uint32_t b_stage_bytes = (uint32_t)p.bn * arow;
    const uint32_t r_stage_bytes = p.nres ? (uint32_t)p.nres * P_RBOX : 0u;
    const uint32_t r_tx_bytes = r_stage_bytes - (p.r16 ? (uint32_t)P_RBOX / 2u : 0u) -             // an fp16 box is half the bytes
                                (p.nres == 2 && p.o16 ? (uint32_t)P_RBOX / 2u : 0u);
    const uint32_t r_bytes = p.nres ? (uint32_t)p.nr * r_stage_bytes : (uint32_t)(4 * p.eg) * 4096u;   // ring or per-warp staging
    uint8_t* smem_a = smem;                                        // na x [rows][K] 16-bit, swizzled
    uint8_t* smem_b = smem_a + (size_t)p.na * a_bytes;             // resident taps or ring of [bn][K]
    uint8_t* smem_r = smem_b + (size_t)p.wstages * b_stage_bytes;  // residual ring / transposition buffers
    uint8_t* smem_x = smem_r + r_bytes;                            // nx activation slots
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_x + (size_t)p.nx * p.xslot);
    uint64_t* b_full = bars;                    // [wstages]
    uint64_t* b_empty = b_full + p.wstages;     // [wstages]
    uint64_t* a_full = b_empty + p.wstages;     // [4]
    uint64_t* a_empty = a_full + 4;             // [4]
    uint64_t* acc_full = a_full + 8;            // [4]
    uint64_t* acc_empty = a_full + 12;          // [4]
    uint64_t* x_full = a_full + 16;             // [nx]
    uint64_t* x_empty = x_full + p.nx;          // [nx]
    uint64_t* r_full = x_empty + p.nx;          // [nr]
    uint64_t* r_empty = r_full + p.nr;          // [nr]
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(r_empty + p.nr);
    volatile uint32_t* x_seq = tmem_ptr_smem + 2;   // [nx] sequence number of the fill in flight / landed in each slot
    volatile uint32_t* r_seq = x_seq + p.nx;        // [nr]

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    constexpr uint32_t xes = X16 ? 2u : 4u;                        // fp32 activations, or the fp16 intra-block tensor
    constexpr uint32_t PASS = X16 ? 256u : 512u;                   // slot bytes one warp pass covers
    const uint32_t xrow = (uint32_t)p.cch * xes;                   // bytes per slot row

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&map_b);
        prefetch_tmap(&map_x);
        prefetch_tmap(&map_xt);
        if (p.nres >= 1) prefetch_tmap(&map_r);
        if (p.nres >= 2) prefetch_tmap(&map_o);
        const int nb = p.resident ? 1 : p.wstages;
        for (int s = 0; s < nb; ++s) {
            mbar_init(&b_full[s], 1);
            mbar_init(&b_empty[s], 1);
        }
        for (int i = 0; i < 4; ++i) {
            mbar_init(&a_full[i], (uint32_t)p.nblk);
            mbar_init(&a_empty[i], 1);
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], 4);
        }
        for (int i = 0; i < p.nx; ++i) {
            mbar_init(&x_full[i], 1);
            mbar_init(&x_empty[i], 1);
            x_seq[i] = 0xffffffffu;
        }
        for (int i = 0; i < p.nr; ++i) {
            mbar_init(&r_full[i], 1);
            mbar_init(&r_empty[i], 4);
            r_seq[i] = 0xffffffffu;
        }
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                     "r"((uint32_t)p.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // K columns the transform never writes (32-channel layer in a 64-wide operand) stay zero for the whole kernel
    for (uint32_t i = threadIdx.x; i < (uint32_t)p.na * a_bytes / 16; i += blockDim.x)
        reinterpret_cast<uint4*>(smem_a)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;
    // everything above (barriers, TMEM, zeroed operand buffers) is independent of the previous kernel in the stream: under
    // programmatic dependent launch it overlaps that kernel; nothing below may run before it has completed
    pdl_trigger();
    pdl_wait();

    if (warp == 0) {
        // ===== producer: three independent queues served by one thread with non-blocking barrier tests =====
        if (elect_one_sync()) {
            if (p.resident) {
                mbar_expect_tx(&b_full[0], (uint32_t)p.ntaps * p.kchunks * b_stage_bytes);
                for (int w = 0; w < p.ntaps; ++w)
                    for (int kc = 0; kc < p.kchunks; ++kc)
                        tma_load_3d(smem_b + (size_t)(w * p.kchunks + kc) * b_stage_bytes, &map_b, &b_full[0], kc * 64, 0, w);
            }
            // activation queue: block g = (tile, kc, blk) -> slot g % nx
            PTile xt; xt.init(p);
            int x_kc = 0, x_blk = 0; uint32_t x_slot = 0, x_par = 0, x_g = 0;
            bool x_done = !xt.valid(p);
            // weight queue: (tile, kc, tap)
            PTile wt; wt.init(p);
            int w_kc = 0, w_j = 0, w_nt = 0; uint32_t w_stage = 0, w_par = 0;
            bool w_done = p.resident || !wt.valid(p);
            // residual queue: box set c = (tile, chunk) -> stage c % nr
            const int nchunks = p.Cout >> 5;             // residual boxes per tile: every 32-column chunk of the row
            PTile rt; rt.init(p);
            int r_ch = 0; uint32_t r_stage = 0, r_par = 0, r_c = 0;
            bool r_done = p.nres == 0 || !rt.valid(p);
            while (!(x_done && w_done && r_done)) {
                if (!w_done && mbar_test(&b_empty[w_stage], w_par ^ 1)) {
                    mbar_expect_tx(&b_full[w_stage], b_stage_bytes);
                    tma_load_3d(smem_b + (size_t)w_stage * b_stage_bytes, &map_b, &b_full[w_stage], w_kc * 64, w_nt * p.bn, w_j);
                    if (++w_stage == (uint32_t)p.wstages) { w_stage = 0; w_par ^= 1; }
                    if (++w_j == p.ntaps) {
                        w_j = 0;
                        if (++w_kc == p.kchunks && (w_kc = 0, ++w_nt == p.nt)) {
                            w_nt = 0;
                            wt.next(p);
                            if (p.pair && wt.valid(p)) wt.next(p);       // the MMA warp covers two tiles per pass
                            w_done = !wt.valid(p);
                        }
                    }
                }
                if (!x_done && mbar_test(&x_empty[x_slot], x_par ^ 1)) {
                    const bool tail = (x_blk == p.nblk - 1);
                    const uint32_t nrows = tail ? (uint32_t)p.tail_rows : (uint32_t)p.xr;
                    x_seq[x_slot] = x_g;                               // published before the fill is issued
                    mbar_expect_tx(&x_full[x_slot], nrows * xrow);
                    tma_load_3d(smem_x + (size_t)x_slot * p.xslot, tail ? &map_xt : &map_x, &x_full[x_slot], x_kc * 64,
                                xt.mt * P_MT + p.halo_min + x_blk * p.xr, xt.b);
                    ++x_g;
                    if (++x_slot == (uint32_t)p.nx) { x_slot = 0; x_par ^= 1; }
                    if (++x_blk == p.nblk) {
                        x_blk = 0;
                        if (++x_kc == p.kchunks) { x_kc = 0; xt.next(p); x_done = !xt.valid(p); }
                    }
                }
                if (!r_done && mbar_test(&r_empty[r_stage], r_par ^ 1)) {
                    r_seq[r_stage] = r_c;
                    mbar_expect_tx(&r_full[r_stage], r_tx_bytes);
                    uint8_t* dst = smem_r + (size_t)r_stage * r_stage_bytes;
                    // columns [32*r_ch, +32) of accumulator row m are channels co0.. of output row m*ostride + phs - opad
                    //   = phase (phs - opad) mod ostride of row m + floor((phs - opad) / ostride) in the (c, phase, m, b) view
                    const int phs = (r_ch * 32) >> p.cshift, co0 = r_ch * 32 - phs * p.cdiv;
                    int u = phs - p.opad, moff = 0;
                    while (u < 0) { u += p.ostride; --moff; }
                    if (p.r16) {
                        // fp16 residual: one [32 rows x 32 ch] box (64-byte rows, SWIZZLE_64B) per TMEM lane quarter, each at the
                        // start of the 4 KB region its epilogue warp later reuses as the fp32 transposition buffer
#pragma unroll
                        for (int qq = 0; qq < 4; ++qq)
                            tma_load_4d(dst + qq * 4096, &map_r, &r_full[r_stage], co0, u, rt.mt * P_MT + moff + qq * 32, rt.b);
                    } else {
                        tma_load_4d(dst, &map_r, &r_full[r_stage], co0, u, rt.mt * P_MT + moff, rt.b);
                    }
                    if (p.nres == 2) {
                        if (p.o16) {
#pragma unroll
                            for (int qq = 0; qq < 4; ++qq)
                                tma_load_4d(dst + P_RBOX + qq * 4096, &map_o, &r_full[r_stage], co0, u, rt.mt * P_MT + moff + qq * 32, rt.b);
                        } else {
                            tma_load_4d(dst + P_RBOX, &map_o, &r_full[r_stage], co0, u, rt.mt * P_MT + moff, rt.b);
                        }
                    }
                    ++r_c;
                    if (++r_stage == (uint32_t)p.nr) { r_stage = 0; r_par ^= 1; }
                    if (++r_ch == nchunks) { r_ch = 0; rt.next(p); r_done = !rt.valid(p); }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (elect_one_sync()) {
            const uint32_t idesc = umma_idesc(128, p.bn, BF16 ? 1 : 0);
            const uint32_t a_lo0 = desc_lo(smem_u32(smem_a));
            const uint32_t a_buf_step = a_bytes >> 4;
            const uint32_t b_lo0 = desc_lo(smem_u32(smem_b));
            const uint32_t b_step = b_stage_bytes >> 4;
            const uint32_t row_step = (uint32_t)(p.tap_step * (int)(arow >> 4));   // 16-byte units per tap (wraps when negative)
            const uint32_t row0 = (uint32_t)p.a_row0 * (arow >> 4);
            // K-major descriptor hi word: SBO = 8 rows (>>4) | version 1 @ bit 46 | SWIZZLE_128B (2) or SWIZZLE_64B (4) @ bit 61
            const uint32_t dhi = p.k32 ? ((512u >> 4) | (1u << 14) | (4u << 29)) : kDescHi;
            const uint32_t b_res_step = (uint32_t)p.kchunks * b_step;
            uint32_t stage = 0, phase = 0, tcnt = 0;
            uint32_t buf = 0, buf_par = 0;              // operand buffer cursor (cc % na, (cc / na) & 1)
            if (p.resident) {
                mbar_wait(&b_full[0], 0);
                tc_fence_after();
            }
            PTile ti;
            ti.init(p);
            if (p.pair) {
                // two tiles per pass over the weight ring: operand buffers (cc & 3) of tile 0 and tile 1, accumulators
                // tcnt & 3 and (tcnt + 1) & 3; every weight stage feeds 8 MMAs instead of 4
                while (ti.valid(p)) {
                    PTile t1 = ti;
                    t1.next(p);
                    const bool two = t1.valid(p);
                    const uint32_t acc0 = tcnt & 3u, acc1 = (tcnt + 1u) & 3u;
                    const uint32_t d0 = tmem_base + acc0 * (uint32_t)p.bn, d1 = tmem_base + acc1 * (uint32_t)p.bn;
                    mbar_wait(&acc_empty[acc0], ((tcnt >> 2) & 1) ^ 1);
                    if (two) mbar_wait(&acc_empty[acc1], (((tcnt + 1u) >> 2) & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t cc0 = tcnt * (uint32_t)p.kchunks;
                    uint32_t accum = 0;
                    for (int kc = 0; kc < p.kchunks; ++kc) {
                        const uint32_t ca = cc0 + (uint32_t)kc, cb = ca + (uint32_t)p.kchunks;
                        const uint32_t ba = ca & 3u, bb = cb & 3u;
                        mbar_wait(&a_full[ba], (ca >> 2) & 1);
                        if (two) mbar_wait(&a_full[bb], (cb >> 2) & 1);
                        tc_fence_after();
                        uint32_t a0 = a_lo0 + ba * a_buf_step + row0, a1 = a_lo0 + bb * a_buf_step + row0;
                        for (int j = 0; j < p.ntaps; ++j) {
                            mbar_wait(&b_full[stage], phase);
                            tc_fence_after();
                            const uint32_t b_lo = b_lo0 + stage * b_step;
                            umma_f16_lohi(d0, a0, b_lo, dhi, idesc, accum);
                            umma_f16_lohi(d0, a0 + 2, b_lo + 2, dhi, idesc, 1u);
                            umma_f16_lohi(d0, a0 + 4, b_lo + 4, dhi, idesc, 1u);
                            umma_f16_lohi(d0, a0 + 6, b_lo + 6, dhi, idesc, 1u);
                            if (two) {
                                umma_f16_lohi(d1, a1, b_lo, dhi, idesc, accum);
                                umma_f16_lohi(d1, a1 + 2, b_lo + 2, dhi, idesc, 1u);
                                umma_f16_lohi(d1, a1 + 4, b_lo + 4, dhi, idesc, 1u);
                                umma_f16_lohi(d1, a1 + 6, b_lo + 6, dhi, idesc, 1u);
                            }
                            accum = 1u;
                            a0 += row_step;
                            a1 += row_step;
                            umma_commit(&b_empty[stage]);
                            if (++stage == (uint32_t)p.wstages) { stage = 0; phase ^= 1; }
                        }
                        umma_commit(&a_empty[ba]);
                        if (two) umma_commit(&a_empty[bb]);
                    }
                    umma_commit(&acc_full[acc0]);
                    if (two) umma_commit(&acc_full[acc1]);
                    tcnt += two ? 2u : 1u;
                    ti = t1;
                    if (two) ti.next(p);
                }
            }
            if (p.nt > 1) {
                // N passes: Cout = nt * bn columns, one accumulator per pass; the tile's operand buffers (cc & 3, all K chunks)
                // stay valid for every pass and are released in the last one; weights stream per (pass, chunk, tap)
                uint32_t au = 0;                        // accumulator use = tile * nt + pass
                for (; ti.valid(p); ti.next(p), ++tcnt) {
                    const uint32_t cc0 = tcnt * (uint32_t)p.kchunks;
                    for (int nt = 0; nt < p.nt; ++nt, ++au) {
                        const uint32_t acc = au & (uint32_t)(p.nacc - 1);
                        const uint32_t d_tmem = tmem_base + acc * (uint32_t)p.bn;
                        mbar_wait(&acc_empty[acc], ((au >> p.nacc_log2) & 1) ^ 1);
                        tc_fence_after();
                        uint32_t accum = 0;
                        for (int kc = 0; kc < p.kchunks; ++kc) {
                            const uint32_t c = cc0 + (uint32_t)kc, ab = c & 3u;
                            if (nt == 0) {
                                mbar_wait(&a_full[ab], (c >> 2) & 1);
                                tc_fence_after();
                            }
                            uint32_t a_lo = a_lo0 + ab * a_buf_step + row0;
                            for (int j = 0; j < p.ntaps; ++j) {
                                mbar_wait(&b_full[stage], phase);
                                tc_fence_after();
                                const uint32_t b_lo = b_lo0 + stage * b_step;
                                umma_f16_lohi(d_tmem, a_lo, b_lo, dhi, idesc, accum);
                                umma_f16_lohi(d_tmem, a_lo + 2, b_lo + 2, dhi, idesc, 1u);
                                umma_f16_lohi(d_tmem, a_lo + 4, b_lo + 4, dhi, idesc, 1u);
                                umma_f16_lohi(d_tmem, a_lo + 6, b_lo + 6, dhi, idesc, 1u);
                                accum = 1u;
                                a_lo += row_step;
                                umma_commit(&b_empty[stage]);
                                if (++stage == (uint32_t)p.wstages) { stage = 0; phase ^= 1; }
                            }
                            if (nt == p.nt - 1) umma_commit(&a_empty[ab]);
                        }
                        umma_commit(&acc_full[acc]);
                    }
                }
            }
            for (; ti.valid(p); ti.next(p), ++tcnt) {
                const uint32_t acc = tcnt & (uint32_t)(p.nacc - 1);
                const uint32_t d_tmem = tmem_base + acc * (uint32_t)p.bn;
                mbar_wait(&acc_empty[acc], ((tcnt >> p.nacc_log2) & 1) ^ 1);   // epilogue drained this accumulator
                tc_fence_after();
                uint32_t accum = 0;
                for (int kc = 0; kc < p.kchunks; ++kc) {
                    mbar_wait(&a_full[buf], buf_par);
                    tc_fence_after();
                    uint32_t a_lo = a_lo0 + buf * a_buf_step + row0;
                    if (p.resident) {
                        uint32_t b_lo = b_lo0 + (uint32_t)kc * b_step;
                        if (p.k32) {
#pragma unroll 4
                            for (int j = 0; j < p.ntaps; ++j) {
                                umma_f16_lohi(d_tmem, a_lo, b_lo, dhi, idesc, accum);
                                umma_f16_lohi(d_tmem, a_lo + 2, b_lo + 2, dhi, idesc, 1u);
                                accum = 1u;
                                a_lo += row_step;
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
                                a_lo += row_step;
                                b_lo += b_res_step;
                            }
                        }
                    } else {
                        for (int j = 0; j < p.ntaps; ++j) {
                            mbar_wait(&b_full[stage], phase);
                            tc_fence_after();
                            const uint32_t b_lo = b_lo0 + stage * b_step;
                            umma_f16_lohi(d_tmem, a_lo, b_lo, dhi, idesc, accum);
                            umma_f16_lohi(d_tmem, a_lo + 2, b_lo + 2, dhi, idesc, 1u);
                            umma_f16_lohi(d_tmem, a_lo + 4, b_lo + 4, dhi, idesc, 1u);
                            umma_f16_lohi(d_tmem, a_lo + 6, b_lo + 6, dhi, idesc, 1u);
                            accum = 1u;
                            a_lo += row_step;
                            umma_commit(&b_empty[stage]);
                            if (++stage == (uint32_t)p.wstages) { stage = 0; phase ^= 1; }
                        }
                    }
                    umma_commit(&a_empty[buf]);          // A tile consumed
                    if (++buf == (uint32_t)p.na) { buf = 0; buf_par ^= 1u; }
                }
                umma_commit(&acc_full[acc]);             // accumulator complete
            }
        }
    } else if (warp < P_W_EPI0) {
        // ===== transform: one warp = one activation block at a time, blocks dealt round-robin =====
        const int tw = warp - P_W_X0;
        const int lpr_shift = (p.cch == 64) ? 4 : 3;            // lanes per row: 16 or 8
        const int rpp = 32 >> lpr_shift;                        // rows per pass: 2 or 4  (one pass = PASS bytes of the slot)
        const int rl = lane >> lpr_shift;
        const int c4 = (lane & ((1 << lpr_shift) - 1)) * 4;
        const uint32_t smem_a_u32 = smem_u32(smem_a);
        const uint32_t smem_x_u32 = smem_u32(smem_x);
        // operand-tile offsets of this thread's 8 rows of a batch, relative to the batch's first row (a multiple of 8, so
        // the swizzle term only depends on the row within the batch):
        //   SWIZZLE_128B: R*128 + ((chunk ^ (R & 7)) << 4)      SWIZZLE_64B: R*64 + ((chunk ^ ((R >> 1) & 3)) << 4)
        uint32_t aoff[8];
        {
            const uint32_t cidx = (uint32_t)(c4 >> 3), sub = (uint32_t)(c4 & 4) * 2u;
            const uint32_t sw_shift = p.k32 ? 1u : 0u, sw_mask = p.k32 ? 3u : 7u;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const uint32_t R = (uint32_t)(rl + u * rpp);
                aoff[u] = R * arow + ((cidx ^ ((R >> sw_shift) & sw_mask)) << 4) + sub;
            }
        }
        const uint32_t batch_a = (uint32_t)(8 * rpp) * arow;    // operand bytes per batch of 8 passes
        PTile ti;
        ti.init(p);
        int seq = 0, kc = 0, blk = tw;
        if (tw >= p.lw) ti.tile = p.num_tiles;                  // idle warp
        while (blk >= p.nblk && ti.valid(p)) {
            blk -= p.nblk;
            if (++kc == p.kchunks) { kc = 0; ti.next(p); ++seq; }
        }
        uint32_t g = (uint32_t)tw;                              // global block number -> slot g % nx, fill g / nx
        uint32_t slot = g % (uint32_t)p.nx, xpar = (g / (uint32_t)p.nx) & 1u;
        int cached_b = -1, cached_kc = -1;
        PXf cf;
        while (ti.valid(p)) {
            const uint32_t cc = (uint32_t)(seq * p.kchunks + kc);
            const uint32_t fill = cc / (uint32_t)p.na;          // this block's operand buffer and which fill of it
            const uint32_t buf = cc - fill * (uint32_t)p.na;
            if (ti.b != cached_b || kc != cached_kc) {          // per-(b,c) coefficients: reload only when they change
                const int cg = kc * 64 + c4;
                const float* ca = p.coef + (size_t)ti.b * 2 * p.coef_ld;
                const float4 a4 = __ldg(reinterpret_cast<const float4*>(ca + cg));
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(ca + p.coef_ld + cg));
                cf.a01 = make_float2(a4.x, a4.y); cf.a23 = make_float2(a4.z, a4.w);
                cf.b01 = make_float2(b4.x, b4.y); cf.b23 = make_float2(b4.z, b4.w);
                if (ACT == ACT_SNAKE) {
                    const float4 al = __ldg(reinterpret_cast<const float4*>(p.alpha + cg));
                    const float4 c = make_float4(__fdividef(0.5f, al.x), __fdividef(0.5f, al.y), __fdividef(0.5f, al.z), __fdividef(0.5f, al.w));
                    cf.ta01 = make_float2(2.f * al.x * a4.x, 2.f * al.y * a4.y); cf.ta23 = make_float2(2.f * al.z * a4.z, 2.f * al.w * a4.w);
                    cf.tb01 = make_float2(2.f * al.x * b4.x, 2.f * al.y * b4.y); cf.tb23 = make_float2(2.f * al.z * b4.z, 2.f * al.w * b4.w);
                    cf.b01 = make_float2(b4.x + c.x, b4.y + c.y); cf.b23 = make_float2(b4.z + c.z, b4.w + c.w);
                    cf.nc01 = make_float2(-c.x, -c.y); cf.nc23 = make_float2(-c.z, -c.w);
                } else {
                    cf.ta01 = make_float2(p.slope, p.slope); cf.ta23 = cf.ta01;
                    cf.tb01 = cf.ta01; cf.tb23 = cf.ta01; cf.nc01 = cf.ta01; cf.nc23 = cf.ta01;
                }
                cached_b = ti.b; cached_kc = kc;
            }
            const int r0 = blk * p.xr;                                       // first A row of this block (multiple of 8)
            const int nrows = (blk == p.nblk - 1) ? p.tail_rows : p.xr;
            const int t0 = ti.mt * P_MT + p.halo_min + r0;                   // time index of that row
            const bool interior = (t0 >= 0) && (t0 + nrows <= p.Tin);
            while (x_seq[slot] != g) { }                                     // fill g has been issued into this slot ...
            mbar_wait_warp(&x_full[slot], xpar);                             // ... and has landed
            mbar_wait_warp(&a_empty[buf], (fill & 1) ^ 1);
            uint32_t xaddr = smem_x_u32 + slot * (uint32_t)p.xslot + (uint32_t)rl * xrow + (uint32_t)c4 * xes;
            uint32_t abase = smem_a_u32 + buf * a_bytes + (uint32_t)r0 * arow;
            int rb = 0;
            if (interior) {
                // full batches: 8 independent loads, then 8 independent activation chains, no per-row checks
                for (; rb + 8 * rpp <= nrows; rb += 8 * rpp, xaddr += 8 * PASS, abase += batch_a) {
                    float4 v[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (X16) v[u] = unpack16x4(lds64(xaddr + (uint32_t)u * PASS), 0);
                        else v[u] = lds128(xaddr + (uint32_t)u * PASS);
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const uint2 o = pipe_transform4<ACT, BF16>(v[u], cf);
                        sts64(abase + aoff[u], o.x, o.y);
                    }
                }
            }
            // ragged end of the block, and blocks that touch the zero padding of the convolution: two passes at a time
            {
                const uint32_t cidx = (uint32_t)(c4 >> 3), sub = (uint32_t)(c4 & 4) * 2u;
                const uint32_t sw_shift = p.k32 ? 1u : 0u, sw_mask = p.k32 ? 3u : 7u;
                const uint32_t abuf = smem_a_u32 + buf * a_bytes + sub;
                for (; rb < nrows; rb += 2 * rpp, xaddr += 2 * PASS) {
                    float4 v[2];
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (rb + rl + u * rpp < nrows) {
                            if (X16) v[u] = unpack16x4(lds64(xaddr + (uint32_t)u * PASS), 0);
                            else v[u] = lds128(xaddr + (uint32_t)u * PASS);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        const int r = rb + rl + u * rpp;
                        uint2 o = pipe_transform4<ACT, BF16>(v[u], cf);
                        const int t = t0 + r;
                        if (t < 0 || t >= p.Tin) o = make_uint2(0u, 0u);   // conv zero padding (after the activation)
                        const uint32_t R = (uint32_t)(r0 + r);
                        if (r < nrows) sts64(abuf + R * arow + ((cidx ^ ((R >> sw_shift) & sw_mask)) << 4), o.x, o.y);
                    }
                }
            }
            fence_proxy_async();            // generic-proxy smem writes -> visible to the tensor core (async proxy)
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&x_empty[slot]);
                mbar_arrive(&a_full[buf]);
            }
            blk += p.lw;
            while (blk >= p.nblk && ti.valid(p)) {
                blk -= p.nblk;
                if (++kc == p.kchunks) { kc = 0; ti.next(p); ++seq; }
            }
            g += (uint32_t)p.lw;
            slot += (uint32_t)p.lw;
            while (slot >= (uint32_t)p.nx) { slot -= (uint32_t)p.nx; xpar ^= 1u; }
        }
    } else {
        // ===== epilogue: TMEM -> (+ residual in the drain layout) -> transposition -> bias/scale -> global, statistics =====
        const int ew = warp - P_W_EPI0;                   // 0 .. 4*EG-1
        const int grp = ew >> 2;                          // accumulator / tile parity this group owns
        const int q = warp & 3;                           // TMEM lane quarter this warp may access
        const int rr = lane >> 3;                         // 0..3: row within a 4-row pass
        const uint32_t l7 = (uint32_t)lane & 7u;
        const int c4o = (int)l7 * 4;                      // column within the 32-column chunk
        const int nchunks = p.bn >> 5;
        const uint32_t smem_r_u32 = smem_u32(smem_r);
        const int ystep = 4 * p.ld_y;                     // element distance between consecutive row passes
        const float2 sc2 = make_float2(p.scale, p.scale);
        uint32_t rs = 0, rpar = 0, rc = 0;                // residual ring cursor: stage, parity, box-set number
        auto r_advance = [&](int n) {
            rc += (uint32_t)n;
            rs += (uint32_t)n;
            while (rs >= (uint32_t)p.nr) { rs -= (uint32_t)p.nr; rpar ^= 1u; }
        };
        uint32_t tcnt = 0, au = 0;                        // accumulator use = tile * nt + pass; groups take uses in turn
        PTile ti;
        for (ti.init(p); ti.valid(p); ti.next(p), ++tcnt) {
          for (int nt = 0; nt < p.nt; ++nt, ++au) {
            if ((int)(au % (uint32_t)EG) != grp) {
                if (p.nres) r_advance(nchunks);           // another group's accumulator
                continue;
            }
            const uint32_t acc = au & (uint32_t)(p.nacc - 1);
            const int cb = nt * p.bn;                     // first column of this pass
            const int m_first = ti.mt * P_MT + q * 32 + rr;                  // rows of this lane: m_first + 4*it
            // warp-uniform: every (row, column) of this quarter maps to an output row inside [0, Tout)
            const int m_lo = ti.mt * P_MT + q * 32;
            const bool full = m_lo + 32 <= p.M && m_lo * p.ostride - p.opad >= 0 &&
                              (m_lo + 31) * p.ostride + (p.ostride - 1) - p.opad < p.Tout;
            uint32_t vmask = 0xffu;
            const size_t yoff = (size_t)ti.b * (size_t)p.ybatch + (size_t)m_first * p.ld_y + c4o;
            float* ytile = p.y16out ? reinterpret_cast<float*>(reinterpret_cast<__half*>(p.y) + yoff) : p.y + yoff;
            float2* stile = p.stats ? p.stats + (((size_t)ti.b * p.mtiles + ti.mt) * 4 + q) * p.Cout + c4o : nullptr;
            mbar_wait_warp(&acc_full[acc], (au >> p.nacc_log2) & 1);
            tc_fence_after();
            auto run_chunks = [&](auto nres_c, auto y16_c) {
            constexpr int NRES = decltype(nres_c)::value;
            constexpr bool Y16 = decltype(y16_c)::value;
            for (int ch = 0; ch < nchunks; ++ch) {
                const int gcol = cb + ch * 32;                 // column of the row this chunk starts at
                const int phs = gcol >> p.cshift;              // polyphase index of this column chunk (0 for a plain conv)
                if (!full) {
                    vmask = 0;
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        const int m = m_first + it * 4, t = m * p.ostride + phs - p.opad;
                        if (m < p.M && t >= 0 && t < p.Tout) vmask |= 1u << it;
                    }
                }
                float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (p.bias != nullptr) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias + gcol - phs * p.cdiv + c4o));
                const float2 bs01 = fmul2(make_float2(bias4.x, bias4.y), sc2), bs23 = fmul2(make_float2(bias4.z, bias4.w), sc2);
                // [32 rows][32 cols] fp32 region of this warp, 16-byte slots XOR-swizzled by (row & 7) -- the TMA
                // SWIZZLE_128B layout of the residual box, and conflict-free for both access directions
                uint32_t tile_u32;
                if (NRES) {
                    while (r_seq[rs] != rc) { }           // box set rc has been issued into this stage ...
                    mbar_wait_warp(&r_full[rs], rpar);    // ... and has landed
                    tile_u32 = smem_r_u32 + rs * r_stage_bytes + (uint32_t)(q * 32) * 128u;
                } else {
                    tile_u32 = smem_r_u32 + (uint32_t)ew * 4096u;
                }
                const uint32_t st_w = tile_u32 + (uint32_t)lane * 128u;      // row = lane (TMEM drain layout)
                {
                    float v[32];
                    tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * (uint32_t)p.bn + (uint32_t)(ch * 32), v);
                    if (ch == nchunks - 1) {
                        // the accumulator is in registers: hand it back to the MMA warp before the stores
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&acc_empty[acc]);
                    }
                    if (NRES) {
                        if (p.r16) {
                            // row = lane of this quarter's fp16 box: 64-byte rows, 16-byte slots XOR-swizzled by (row >> 1) & 3
                            const uint32_t st_h = tile_u32 + (uint32_t)lane * 64u, sw = ((uint32_t)lane >> 1) & 3u;
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const float4 raw = lds128(st_h + (((uint32_t)i ^ sw) << 4));
                                const float4 r0 = unpack16x4(make_uint2(__float_as_uint(raw.x), __float_as_uint(raw.y)), 0);
                                const float4 r1 = unpack16x4(make_uint2(__float_as_uint(raw.z), __float_as_uint(raw.w)), 0);
                                v[8 * i] += r0.x; v[8 * i + 1] += r0.y; v[8 * i + 2] += r0.z; v[8 * i + 3] += r0.w;
                                v[8 * i + 4] += r1.x; v[8 * i + 5] += r1.y; v[8 * i + 6] += r1.z; v[8 * i + 7] += r1.w;
                            }
                            __syncwarp();                 // the fp32 rows written below overlap other lanes' fp16 rows
                        } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float4 r = lds128(st_w + (((uint32_t)i ^ l7) << 4));
                            const float2 lo = fadd2(make_float2(v[4 * i], v[4 * i + 1]), make_float2(r.x, r.y));
                            const float2 hi = fadd2(make_float2(v[4 * i + 2], v[4 * i + 3]), make_float2(r.z, r.w));
                            v[4 * i] = lo.x; v[4 * i + 1] = lo.y; v[4 * i + 2] = hi.x; v[4 * i + 3] = hi.y;
                        }
                        }
                        if (NRES == 2) {
                            if (p.o16) {
                                const uint32_t st_h = tile_u32 + (uint32_t)P_RBOX + (uint32_t)lane * 64u, sw = ((uint32_t)lane >> 1) & 3u;
#pragma unroll
                                for (int i = 0; i < 4; ++i) {
                                    const float4 raw = lds128(st_h + (((uint32_t)i ^ sw) << 4));
                                    const float4 r0 = unpack16x4(make_uint2(__float_as_uint(raw.x), __float_as_uint(raw.y)), 0);
                                    const float4 r1 = unpack16x4(make_uint2(__float_as_uint(raw.z), __float_as_uint(raw.w)), 0);
                                    v[8 * i] += r0.x; v[8 * i + 1] += r0.y; v[8 * i + 2] += r0.z; v[8 * i + 3] += r0.w;
                                    v[8 * i + 4] += r1.x; v[8 * i + 5] += r1.y; v[8 * i + 6] += r1.z; v[8 * i + 7] += r1.w;
                                }
                            } else {
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const float4 r = lds128(st_w + (uint32_t)P_RBOX + (((uint32_t)i ^ l7) << 4));
                                const float2 lo = fadd2(make_float2(v[4 * i], v[4 * i + 1]), make_float2(r.x, r.y));
                                const float2 hi = fadd2(make_float2(v[4 * i + 2], v[4 * i + 3]), make_float2(r.z, r.w));
                                v[4 * i] = lo.x; v[4 * i + 1] = lo.y; v[4 * i + 2] = hi.x; v[4 * i + 3] = hi.y;
                            }
                            }
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        sts128(st_w + (((uint32_t)i ^ l7) << 4), v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                }
                __syncwarp();
                const uint32_t st_r0 = tile_u32 + (uint32_t)rr * 128u + ((l7 ^ (uint32_t)rr) << 4);               // rows rr, rr+8, ...
                const uint32_t st_r1 = tile_u32 + (uint32_t)(rr + 4) * 128u + ((l7 ^ (uint32_t)(rr + 4)) << 4);   // rows rr+4, rr+12, ...
                float2 s1a = make_float2(0.f, 0.f), s1b = s1a, s2a = s1a, s2b = s1a;
                float* yo = Y16 ? reinterpret_cast<float*>(reinterpret_cast<__half*>(ytile) + gcol) : ytile + gcol;
                if (full) pipe_store_rows<true, Y16>(st_r0, st_r1, yo, ystep, vmask, sc2, bs01, bs23, s1a, s1b, s2a, s2b);
                else pipe_store_rows<false, Y16>(st_r0, st_r1, yo, ystep, vmask, sc2, bs01, bs23, s1a, s1b, s2a, s2b);
                if (stile != nullptr) {
                    float s1[4] = {s1a.x, s1a.y, s1b.x, s1b.y}, s2[4] = {s2a.x, s2a.y, s2b.x, s2b.y};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        s1[i] += __shfl_xor_sync(0xffffffffu, s1[i], 8);
                        s2[i] += __shfl_xor_sync(0xffffffffu, s2[i], 8);
                        s1[i] += __shfl_xor_sync(0xffffffffu, s1[i], 16);
                        s2[i] += __shfl_xor_sync(0xffffffffu, s2[i], 16);
                    }
                    // one partial per (tile, TMEM lane quarter): written straight to global, no cross-warp barrier
                    if (lane < 8) {
                        float2* sp = stile + gcol;
                        *reinterpret_cast<float4*>(sp) = make_float4(s1[0], s2[0], s1[1], s2[1]);
                        *reinterpret_cast<float4*>(sp + 2) = make_float4(s1[2], s2[2], s1[3], s2[3]);
                    }
                }
                if (NRES) {
                    fence_proxy_async();                  // our generic writes to the stage precede the next TMA fill
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&r_empty[rs]);
                    r_advance(1);
                } else {
                    __syncwarp();
                }
            }
            };
            // one specialisation per launch configuration (uniform over the grid): no per-chunk branches on kernel parameters
            if (p.nres == 0) {
                if (p.y16out) run_chunks(std::integral_constant<int, 0>{}, std::true_type{});
                else run_chunks(std::integral_constant<int, 0>{}, std::false_type{});
            } else if (p.nres == 1) {
                if (p.y16out) run_chunks(std::integral_constant<int, 1>{}, std::true_type{});
                else run_chunks(std::integral_constant<int, 1>{}, std::false_type{});
            } else {
                if (p.y16out) run_chunks(std::integral_constant<int, 2>{}, std::true_type{});
                else run_chunks(std::integral_constant<int, 2>{}, std::false_type{});
            }
          }
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

// ---------------------------------------------------------------- host side
int make_weight_map(CUtensorMap* map, int is_bf16, const void* w16, int cin_pad, int cout_pad, int ktaps, int bn);
int make_weight_map_k32(CUtensorMap* map, int is_bf16, const void* w16, int cin_pad, int cout_pad, int ktaps, int bn);
int make_map_4d_f32_sw128(CUtensorMap* map, const void* base, uint64_t C, uint64_t phases, uint64_t rows, uint64_t B,
                          uint64_t ld_bytes, uint64_t batch_bytes, uint32_t b0, uint32_t b2);
int make_map_4d_f16_sw64(CUtensorMap* map, const void* base, uint64_t C, uint64_t rows, uint64_t B, uint64_t ld_bytes,
                         uint64_t batch_bytes, uint32_t b0, uint32_t b2);
int make_map_3d_any(CUtensorMap* map, int dtype /*0 f32, 1 bf16, 2 f16*/, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                    uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t b0, uint32_t b1, int swizzle128);

static bool pipe_geometry_ok(const ConvArgs& a) {
    if (tune().no_pipe) return false;
    if (a.in_stride != 1 || a.mirror || a.res_shift != 0) return false;
    const bool tr = a.phases > 1;          // polyphase ConvTranspose1d -> dense conv with N = phases * Cout
    if (tr) {
        if (a.out_stride != a.phases || a.w_step != a.phases || a.tap_step != -1 || a.in_off != 0 || a.accumulate) return false;
        if (a.ld_y != a.Cout || (a.res != nullptr && a.ld_res != a.Cout)) return false;
        if (a.Tout % a.phases != 0 || a.out_pad < 0 || a.out_pad > a.phases) return false;
    } else if (a.out_stride != 1 || a.out_pad != 0 || a.tap_step <= 0 || a.M != a.Tout) {
        return false;
    }
    if (a.w16 == nullptr || a.w16_cin_pad % 64 != 0 || a.w16_cout_pad % 32 != 0) return false;
    {
        // columns of one accumulator row: <= 256 in one pass (192 at most in practice), else passes of 128 over an operand
        // tile that stays resident in the 4 operand buffers (<= 4 K chunks)
        const int ntot = a.phases * a.w16_cout_pad, kch = a.w16_cin_pad / 64;
        const bool one_pass = ntot <= 192;
        const bool n_pass = ntot % 128 == 0 && ntot <= 1024 && (kch == 1 || kch == 2 || kch == 4);
        if (!one_pass && !n_pass) return false;
        // measured on the 256-channel layers (N passes here vs conv_fused.cu): k=3 0.278 -> 0.165 ms, k=7 0.293 -> 0.276
        // (no residual) and 0.337 -> 0.313 (accumulate), ups 256->128 1.14 -> 0.37; k=7 with one residual and k=11 are
        // tensor-bound over there (up to 1250 TFLOP/s) and lose here, so they stay
        if (!one_pass && a.phases == 1) {
            const int nres_ = (a.res != nullptr ? 1 : 0) + (a.accumulate ? 1 : 0);
            if (a.ntaps > 7 || (a.ntaps == 7 && nres_ == 1)) return false;
        }
    }
    if (!(a.Cin == 32 || a.Cin % 64 == 0) || a.Cout % 32 != 0 || a.Cout != a.w16_cout_pad) return false;
    if ((a.Cout & (a.Cout - 1)) != 0) return false;        // column -> phase is a shift
    if (a.w16_cin_pad != (a.Cin == 32 ? 64 : a.Cin)) return false;
    // x16in / y16out: the intra-block tensor of AdaINResBlock1 stored as fp16 (plain stride-1 convs only)
    if ((a.x16in || a.res16) && tr) return false;
    if (a.acc_src != nullptr && !a.accumulate) return false;
    if (a.y16out && a.accumulate && !(a.acc_src != nullptr && a.acc16)) return false;     // fp16 in-place sums need an fp16 source
    if (a.res16 && a.res == nullptr) return false;
    if (a.ld_x % (a.x16in ? 8 : 4) != 0 || a.ld_y % 4 != 0 || (a.res != nullptr && a.ld_res % (a.res16 ? 8 : 4) != 0)) return false;
    if (a.accumulate && a.res == nullptr) return false;
    const int span = (a.ntaps - 1) * (a.tap_step < 0 ? -a.tap_step : a.tap_step);
    return span <= 64 && (tr || (a.in_off <= 0 && a.in_off + span >= 0));
}

// geometry + shared-memory plan; false if the rings do not fit next to the operand tiles and weights
static bool pipe_plan(const ConvArgs& a, PipeParams& p, size_t* smem_out) {
    memset(&p, 0, sizeof(p));
    p.Cin = a.Cin; p.kchunks = a.w16_cin_pad / 64; p.cch = a.Cin == 32 ? 32 : 64;
    p.x16in = a.x16in; p.is_bf16 = a.fmt16 == DT_BF16 ? 1 : 0;
    p.k32 = a.Cin == 32 ? 1 : 0;
    const int ph = a.phases;               // 1, or the stride of a transposed conv (columns = ph * Cout)
    const bool tr_ = a.phases > 1;
    p.B = a.B; p.M = a.M; p.Tin = a.Tin; p.Cout = ph * a.Cout;
    p.ntaps = a.ntaps; p.tap_step = a.tap_step;
    const int span = (a.ntaps - 1) * (a.tap_step < 0 ? -a.tap_step : a.tap_step);
    p.halo_min = a.in_off + (a.tap_step < 0 ? (a.ntaps - 1) * a.tap_step : 0);
    p.a_row0 = a.in_off - p.halo_min;
    p.rows = P_MT + span;
    p.ostride = a.out_stride; p.opad = a.out_pad; p.Tout = a.Tout; p.cdiv = a.Cout;
    p.cshift = 0;
    while ((1 << p.cshift) < a.Cout) ++p.cshift;
    {
        // activation blocks: the fewest equal blocks (whole passes of the owning warp) that fit a 12 KB slot
        const int rowb = p.cch * (a.x16in ? 2 : 4), rpp = 8;   // blocks are whole multiples of 8 rows (swizzle period)
        // 12 KB blocks by default; 8 KB when every residual stage holds two boxes (residual + accumulate), where the
        // smaller blocks leave room for one more stage (measured: 0.75 -> 0.60 ms on the 32-channel k=11 layer)
        int xmax = (a.res != nullptr && a.accumulate) ? 8192 : P_XSLOT_MAX;
        // measured per layer class on the B200: 8 KB blocks win by 3-14 % where the 12 KB
        // split leaves a short last block per tile -- 64 channels k=7 (0.435 -> 0.398 ms), 128 channels k=3 without residual
        // (0.362 -> 0.312) and k=7 with one residual (0.350 -> 0.338); every 32-channel layer loses 5-14 % with them
        const int nres_ = (a.res != nullptr ? 1 : 0) + (a.accumulate ? 1 : 0);
        if ((a.Cin == 64 && a.ntaps == 7) || (a.Cin == 128 && a.ntaps == 3 && nres_ == 0) || (a.Cin == 128 && a.ntaps == 7 && nres_ == 1))
            xmax = 8192;
        if (a.x16in && xmax > 8192) xmax = 8192;  // fp16 input: a 12 KB block would be a whole tile for one warp (8 KB: 1-8 % faster on the k=3 layers)
        int nblk = 1;
        for (;; ++nblk) {
            p.xr = (cdiv(p.rows, nblk) + rpp - 1) / rpp * rpp;
            if (p.xr * rowb <= xmax) break;
        }
        p.nblk = cdiv(p.rows, p.xr);
        p.tail_rows = p.rows - (p.nblk - 1) * p.xr;
        p.xslot = (p.xr * rowb + 127) / 128 * 128;
    }
    {
        const int ntot = ph * a.w16_cout_pad;
        p.nt = ntot <= 192 ? 1 : ntot / 128;
        p.bn = ntot / p.nt;
    }
    p.mtiles = cdiv(a.M, P_MT);
    p.num_tiles = a.B * p.mtiles;
    p.nacc = p.bn <= 128 ? 4 : 2;
    p.nacc_log2 = p.nacc == 4 ? 2 : 1;
    int cols = 32;
    while (cols < p.nacc * p.bn) cols <<= 1;
    p.tmem_cols = cols;
    p.nres = (a.res != nullptr ? 1 : 0) + (a.accumulate ? 1 : 0);
    p.r16 = a.res16 ? 1 : 0;
    p.o16 = (a.accumulate && a.acc_src != nullptr && a.acc16) ? 1 : 0;
    p.eg = (p.cch == 32 && p.nres > 0 && !tr_) ? 3 : 2;
    // three groups for the non-residual 32-channel layers too were measured slower, 0.385 -> 0.416 ms at k = 3 -- the
    // 96-register variant costs the transform warps more than the third group gives the epilogue
    // 3 groups need 4 accumulators: a group's previous tile is tcnt-3, so MMA(tcnt-4) -- the previous use of its accumulator
    // -- has completed when it waits; with 2 accumulators the previous use is tile tcnt-2 and the parity wait could pass early
    if (p.nacc < 4) p.eg = 2;
    p.bias = a.bias; p.scale = a.scale; p.y16out = a.y16out;
    p.y = a.y16out ? reinterpret_cast<float*>(reinterpret_cast<__half*>(a.y) - (int64_t)a.out_pad * a.ld_y)
                   : a.y - (int64_t)a.out_pad * a.ld_y;            // row m, column c  ->  y[b][m*ostride - opad][c]  (dense [M][ph*Cout])
    p.ld_y = ph * a.ld_y;
    p.ybatch = (long long)a.Tout * a.ld_y;

    // ---- shared-memory plan (one persistent CTA per SM)
    const int64_t budget = 225 * 1024;
    const int64_t arow = p.k32 ? 64 : 128;
    const int64_t a_bytes = ((int64_t)p.rows * arow + 1023) & ~(int64_t)1023;
    const int64_t b_stage = (int64_t)p.bn * arow;
    const int64_t r_stage = (int64_t)p.nres * P_RBOX;
    // tile pairs: streamed weights with exactly 2 K chunks (the 128-channel layers) -> 4 operand buffers up front
    // (measured on the 128-channel layers: conv2 with one residual 0.405 -> 0.36 ms (k=7), 0.535 -> 0.507 (k=11); layers without
    // a residual, whose epilogue staging leaves less room for the rings, and the accumulate layers lose, so only nres == 1)
    const bool pair_ok = p.nt == 1 && p.kchunks == 2 && p.bn <= 128 && p.nacc == 4 && p.nres == 1 &&
                         (int64_t)a.ntaps * p.kchunks * b_stage > 96 * 1024;
    int na = (pair_ok || p.nt > 1) ? 4 : 2;
    int64_t base = na * a_bytes + 2048 + (p.nres ? 0 : (int64_t)(4 * p.eg) * 4096);
    const int64_t w_resident = (int64_t)a.ntaps * p.kchunks * b_stage;
    const int nchunks = p.bn / 32;
    // rings: nx activation slots and nr residual stages (FIFO); minimum 3 slots / 2 stages
    const int64_t xslot = p.xslot;
    int nx = 3, nr = p.nres ? 2 : 0;
    auto rings = [&](int nx_, int nr_) { return (int64_t)nx_ * xslot + (int64_t)nr_ * r_stage; };
    p.resident = (p.nt == 1 && base + w_resident + rings(nx, nr) <= budget) ? 1 : 0;
    int64_t left;
    if (p.resident) {
        p.wstages = a.ntaps * p.kchunks;
        left = budget - base - w_resident;
    } else {
        p.wstages = 4;                       // weight ring: at least 4 stages
        left = budget - base - p.wstages * b_stage;
        if (left < rings(nx, nr)) return false;
    }
    // what is left goes to the two rings in turn (bytes in flight are what hides the HBM latency), then to the weight ring
    left -= rings(nx, nr);
    int nr_goal = p.nres ? (2 * nchunks + 2 > 8 ? 8 : 2 * nchunks + 2) : 0;
    int nx_goal = 10;
    // resident weights of a 2-chunk layer (128 channels, k = 3: 96 KB) leave little for the rings: two operand buffers and
    // deeper rings measured 0.319 -> 0.264 ms (no residual), 0.356 -> 0.310 (residual), 0.546 -> 0.478 (accumulate)
    int na_goal = (p.resident && p.kchunks >= 2) ? 2 : 4;
    for (bool grew = true; grew;) {
        grew = false;
        // a third / fourth operand buffer as soon as the rings hold ~32 KB / ~48 KB each (or all they are allowed to)
        const int64_t want = na == 2 ? 32 * 1024 : 48 * 1024;
        const bool x_ok = (int64_t)nx * xslot >= want || nx >= nx_goal;
        const bool r_ok = nr_goal == 0 || (int64_t)nr * r_stage >= want || nr >= nr_goal;
        if (na < na_goal && x_ok && r_ok && left >= a_bytes) { ++na; left -= a_bytes; grew = true; continue; }
        const bool r_first = (int64_t)nr * r_stage <= (int64_t)nx * xslot;
        if (nr < nr_goal && left >= r_stage && (r_first || nx >= nx_goal)) { ++nr; left -= r_stage; grew = true; continue; }
        if (nx < nx_goal && left >= xslot) { ++nx; left -= xslot; grew = true; continue; }
        if (nr < nr_goal && left >= r_stage) { ++nr; left -= r_stage; grew = true; }
    }
    if (!p.resident)
        while (p.wstages < 8 && left >= b_stage) { ++p.wstages; left -= b_stage; }
    p.nx = nx; p.nr = nr;
    p.na = na;
    p.pair = (pair_ok && !p.resident && na == 4) ? 1 : 0;
    p.lw = na * p.nblk < P_LW ? na * p.nblk : P_LW;
    const size_t smem = (size_t)(na * a_bytes + (int64_t)p.wstages * b_stage + (p.nres ? (int64_t)p.nr * r_stage : (int64_t)(4 * p.eg) * 4096) +
                                 (int64_t)p.nx * p.xslot + 2048 + 1024);
    if (smem > 227 * 1024) return false;
    if ((2 * p.wstages + 16 + 2 * p.nx + 2 * p.nr) * 8 + 16 + (p.nx + p.nr) * 4 > 2048) return false;
    *smem_out = smem;
    return true;
}

bool conv_pipe_supported(const ConvArgs& a) {
    if (!pipe_geometry_ok(a)) return false;
    PipeParams p;
    size_t smem;
    return pipe_plan(a, p, &smem);
}

int launch_conv_pipe(const ConvArgs& a, const float* coef, int coef_ld, int act, float slope, const float* alpha,
                     void* stats_out, cudaStream_t st) {
    PipeParams p;
    size_t smem = 0;
    ST2_REQUIRE(pipe_geometry_ok(a) && pipe_plan(a, p, &smem), "conv_pipe: unsupported geometry");
    p.coef = coef; p.coef_ld = coef_ld; p.alpha = alpha; p.slope = slope;
    p.stats = (float2*)stats_out;

    // ---- tensor maps
    CUtensorMap map_b, map_x, map_xt, map_r, map_o;
    // transposed conv: taps are stored phase-major (widx = phase + j*stride), so tap j of the stacked weight is the
    // [phases*Cout][Cin] slab starting at stored tap j*stride -- the same memory viewed with phases*Cout rows per tap
    int e = p.k32 ? make_weight_map_k32(&map_b, p.is_bf16, a.w16, a.w16_cin_pad, a.phases * a.w16_cout_pad, a.ntaps, p.bn)
                  : make_weight_map(&map_b, p.is_bf16, a.w16, a.w16_cin_pad, a.phases * a.w16_cout_pad, a.ntaps, p.bn);
    if (e != ST2_OK) return e;
    const int xdt = a.x16in ? 2 : 0;
    const uint64_t xes = a.x16in ? 2 : 4;
    e = make_map_3d_any(&map_x, xdt, a.x, (uint64_t)a.Cin, (uint64_t)a.Tin, (uint64_t)a.B, (uint64_t)a.ld_x * xes,
                        (uint64_t)a.Tin * a.ld_x * xes, (uint32_t)p.cch, (uint32_t)p.xr, 0);
    if (e != ST2_OK) return e;
    e = make_map_3d_any(&map_xt, xdt, a.x, (uint64_t)a.Cin, (uint64_t)a.Tin, (uint64_t)a.B, (uint64_t)a.ld_x * xes,
                        (uint64_t)a.Tin * a.ld_x * xes, (uint32_t)p.cch, (uint32_t)p.tail_rows, 0);
    if (e != ST2_OK) return e;
    map_r = map_x;
    map_o = map_x;
    if (a.res != nullptr && a.res16) {
        e = make_map_4d_f16_sw64(&map_r, a.res, (uint64_t)a.Cout, (uint64_t)a.Tout, (uint64_t)a.B, (uint64_t)a.ld_res * 2,
                                 (uint64_t)a.Tout * a.ld_res * 2, 32, 32);
        if (e != ST2_OK) return e;
    } else if (a.res != nullptr) {
        e = make_map_4d_f32_sw128(&map_r, a.res, (uint64_t)a.Cout, (uint64_t)a.phases, (uint64_t)(a.Tout / a.phases), (uint64_t)a.B,
                                  (uint64_t)a.ld_res * 4, (uint64_t)a.Tout * a.ld_res * 4, 32, P_MT);
        if (e != ST2_OK) return e;
    }
    if (a.accumulate) {
        const void* old = a.acc_src != nullptr ? a.acc_src : (const void*)a.y;
        if (p.o16)
            e = make_map_4d_f16_sw64(&map_o, old, (uint64_t)a.Cout, (uint64_t)a.Tout, (uint64_t)a.B, (uint64_t)a.ld_y * 2,
                                     (uint64_t)a.Tout * a.ld_y * 2, 32, 32);
        else
            e = make_map_4d_f32_sw128(&map_o, old, (uint64_t)a.Cout, 1, (uint64_t)a.Tout, (uint64_t)a.B, (uint64_t)a.ld_y * 4,
                                      (uint64_t)a.Tout * a.ld_y * 4, 32, P_MT);
        if (e != ST2_OK) return e;
    }
    // the opt-in to > 48 KB of dynamic shared memory applies to the device that is current: once per device
    static bool attr_done[kMaxDevices] = {};
    const int num_sms = device_num_sms();
    if (!attr_done[current_device_slot()]) {
#define PIPE_ATTR(A, BF, X, G) ST2_CUDA_CHECK(cudaFuncSetAttribute(conv_pipe_kernel<A, BF, X, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024))
        PIPE_ATTR(ACT_NONE, true, false, 2); PIPE_ATTR(ACT_NONE, false, false, 2);
        PIPE_ATTR(ACT_LRELU, true, false, 2); PIPE_ATTR(ACT_LRELU, false, false, 2);
        PIPE_ATTR(ACT_SNAKE, true, false, 2); PIPE_ATTR(ACT_SNAKE, false, false, 2);
        PIPE_ATTR(ACT_SNAKE, true, true, 2); PIPE_ATTR(ACT_SNAKE, false, true, 2);
        PIPE_ATTR(ACT_SNAKE, true, false, 3); PIPE_ATTR(ACT_SNAKE, false, false, 3);
        PIPE_ATTR(ACT_SNAKE, true, true, 3); PIPE_ATTR(ACT_SNAKE, false, true, 3);
#undef PIPE_ATTR
        attr_done[current_device_slot()] = true;
    }
    int grid = num_sms;
    if (grid > p.num_tiles) grid = p.num_tiles;
    ST2_REQUIRE(act != ACT_SNAKE || alpha != nullptr, "conv_pipe: snake needs alpha");
    ST2_REQUIRE(!a.x16in || act == ACT_SNAKE, "conv_pipe: 16-bit input is only built for the Snake transform");
    if (act != ACT_SNAKE) p.eg = 2;                          // the 3-group variant is only built for Snake
    cudaLaunchConfig_t lcfg = {};
    lcfg.gridDim = dim3(grid); lcfg.dynamicSmemBytes = smem; lcfg.stream = st;
    cudaLaunchAttribute lattr;
    lattr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    lattr.val.programmaticStreamSerializationAllowed = 1;
    // Only for small problems (a few tiles per CTA, i.e. one-sentence latency: 3.65 -> 3.29 ms at 1 x 3 s): in throughput
    // runs the early CTAs of this kernel sit on SMs the coefficient kernel in front of it needs, +0.8 ms per 64 x 5 s step
    const bool pdl = p.num_tiles <= 16 * num_sms;
    lcfg.attrs = &lattr; lcfg.numAttrs = pdl ? 1 : 0;
    // Cout counts the columns of one accumulator row (phases * Cout for a transposed conv); mtiles * B = tiles, walked
    // tile = blockIdx.x + i * grid
    if (tune().verbose)
        fprintf(stderr, "conv_pipe: Cin=%d Cout=%d phases=%d taps=%d step=%d rows=%d nblk=%d tail=%d xr=%d resident=%d wstages=%d na=%d "
                "nacc=%d lw=%d nx=%d nr=%d nres=%d smem=%zu mtiles=%d tiles=%d grid=%d pair=%d eg=%d nt=%d bn=%d x16=%d r16=%d o16=%d "
                "y16=%d pdl=%d\n",
                p.Cin, p.Cout, p.ostride, p.ntaps, p.tap_step, p.rows, p.nblk, p.tail_rows, p.xr, p.resident, p.wstages, p.na, p.nacc,
                p.lw, p.nx, p.nr, p.nres, smem, p.mtiles, p.num_tiles, grid, p.pair, p.eg, p.nt, p.bn, p.x16in, p.r16, p.o16,
                p.y16out, pdl ? 1 : 0);
#define PIPE_LAUNCH(A, BF, X, G)                                                                                         \
    do {                                                                                                                 \
        lcfg.blockDim = dim3((P_W_EPI0 + 4 * G) * 32);                                                                   \
        ST2_CUDA_CHECK(cudaLaunchKernelEx(&lcfg, conv_pipe_kernel<A, BF, X, G>, map_b, map_x, map_xt, map_r, map_o, p)); \
    } while (0)
    const bool bf = p.is_bf16 != 0;
    switch (act) {
        case ACT_NONE: if (bf) PIPE_LAUNCH(ACT_NONE, true, false, 2); else PIPE_LAUNCH(ACT_NONE, false, false, 2); break;
        case ACT_LRELU: if (bf) PIPE_LAUNCH(ACT_LRELU, true, false, 2); else PIPE_LAUNCH(ACT_LRELU, false, false, 2); break;
        case ACT_SNAKE:
            if (p.eg == 3) {
                if (a.x16in) { if (bf) PIPE_LAUNCH(ACT_SNAKE, true, true, 3); else PIPE_LAUNCH(ACT_SNAKE, false, true, 3); }
                else { if (bf) PIPE_LAUNCH(ACT_SNAKE, true, false, 3); else PIPE_LAUNCH(ACT_SNAKE, false, false, 3); }
            } else {
                if (a.x16in) { if (bf) PIPE_LAUNCH(ACT_SNAKE, true, true, 2); else PIPE_LAUNCH(ACT_SNAKE, false, true, 2); }
                else { if (bf) PIPE_LAUNCH(ACT_SNAKE, true, false, 2); else PIPE_LAUNCH(ACT_SNAKE, false, false, 2); }
            }
            break;
        default: set_error("conv_pipe: bad act %d", act); return ST2_ERR_INVALID;
    }
#undef PIPE_LAUNCH
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

}  // namespace st2
