// Tensor-core implicit-GEMM Conv1d / ConvTranspose1d for sm_100a: TMA -> shared memory ->
// tcgen05.mma (kind::f16, bf16 or fp16 operands) with fp32 accumulators in TMEM.
//
// Same ConvArgs contract as conv_simt.cu (stride-1 Conv1d and polyphase ConvTranspose1d; the
// strided 1->C noise_convs stay on the SIMT kernel).  GEMM view per CTA:
//     D[128 time steps, BN couts] = sum_{tap j} sum_{ci chunk of 64}  A_j[128, 64] * W_j[64, BN]
//   A: channels-last 16-bit activations x16[B][Tin][ld]; a 3-D tensor map (ci, t, b) lets TMA
//      fetch the [128 x 64] box at time coordinate m0 + j*tap_step + in_off -- dilation is a
//      coordinate shift and the conv zero padding is TMA's out-of-bounds fill (per utterance,
//      because b is its own coordinate).
//   B: weights packed at load time as [tap][CoutPad][CinPad] (K-major), box [BN x 64].
//   Both land in the canonical 128-byte-swizzled K-major layout that the UMMA shared-memory
//   descriptors address (SBO = 1024 B between 8-row groups; K advance = +32 B inside the atom).
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer (one
// elected lane), warps 2-5 = epilogue (tcgen05.ld 32x32b -> bias/residual/scale -> global).
// Two CTAs fit per SM (<= 96 KB shared, <= 256 TMEM columns each) so one CTA's epilogue overlaps
// the other's main loop.
#include <cuda.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace st2 {

static constexpr int TC_BM = 128;
static constexpr int TC_KC = 64;             // K chunk: 64 x 16-bit = one 128-byte swizzle row
static constexpr int TC_THREADS = 192;
static constexpr uint32_t A_STAGE_BYTES = TC_BM * TC_KC * 2;   // 16 KB

struct TcParams {
    const float* bias;
    const float* res; int ld_res; int res_shift;
    float* y; int ld_y; int Tout;
    int Cout, M;
    int ntaps, tap_step, in_off;
    int phases, w_step, out_stride, out_pad;
    int kchunks;                 // CinPad / 64
    int bn;                      // N tile (multiple of 16, <= 256)
    int tmem_cols;               // power of two >= bn
    int stages;
    float scale; int accumulate; int mirror;
    int is_bf16;
    int epi_gelu;                // y = GELU(acc + bias) as 16-bit values (is_bf16 selects the format), pitch ld_y elements
};

__global__ void __launch_bounds__(TC_THREADS)
conv_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const TcParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // 1024-byte aligned tiles (SWIZZLE_128B atoms)
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const uint32_t b_stage_bytes = (uint32_t)p.bn * TC_KC * 2;
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + (size_t)p.stages * A_STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + (size_t)p.stages * b_stage_bytes);
    uint64_t* full_bar = bars;                     // [stages]
    uint64_t* empty_bar = bars + p.stages;         // [stages]
    uint64_t* tmem_full_bar = bars + 2 * p.stages; // [1]
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * p.stages + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * TC_BM;
    const int n0 = blockIdx.y * p.bn;
    const int b = blockIdx.z / p.phases;
    const int ph = blockIdx.z - b * p.phases;
    const int nit = p.ntaps * p.kchunks;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&map_a);
        prefetch_tmap(&map_b);
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        mbar_init(tmem_full_bar, 1);
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                     "r"((uint32_t)p.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int it = 0; it < nit; ++it) {
                const int j = it / p.kchunks;
                const int kc = it - j * p.kchunks;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                mbar_expect_tx(&full_bar[stage], A_STAGE_BYTES + b_stage_bytes);
                tma_load_3d(smem_a + (size_t)stage * A_STAGE_BYTES, &map_a, &full_bar[stage], kc * TC_KC,
                            m0 + j * p.tap_step + p.in_off, b);
                tma_load_3d(smem_b + (size_t)stage * b_stage_bytes, &map_b, &full_bar[stage], kc * TC_KC, n0,
                            ph + j * p.w_step);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            const uint32_t idesc = umma_idesc(TC_BM, p.bn, p.is_bf16);
            int stage = 0;
            uint32_t phase = 0;
            for (int it = 0; it < nit; ++it) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint64_t adesc = umma_desc_sw128(smem_u32(smem_a + (size_t)stage * A_STAGE_BYTES));
                const uint64_t bdesc = umma_desc_sw128(smem_u32(smem_b + (size_t)stage * b_stage_bytes));
#pragma unroll
                for (int k4 = 0; k4 < TC_KC / 16; ++k4)
                    umma_f16(tmem_base, adesc + (uint64_t)(k4 * 2), bdesc + (uint64_t)(k4 * 2), idesc,
                             (it > 0 || k4 > 0) ? 1u : 0u);
                umma_commit(&empty_bar[stage]);          // frees the smem slot when these MMAs retire
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
            umma_commit(tmem_full_bar);                  // accumulator complete
        }
    } else {
        // ===== epilogue: TMEM -> registers -> global =====
        const int q = warp & 3;                          // TMEM lane quarter this warp may access
        const int row = q * 32 + lane;
        const int m = m0 + row;
        mbar_wait(tmem_full_bar, 0);
        tc_fence_after();
        const int t = m * p.out_stride + ph - p.out_pad;
        const bool row_ok = (m < p.M) && (t >= (p.mirror ? 1 : 0)) && (t < p.Tout);   // mirror: row 0 is written by the row-2 thread only
        const bool vec = (p.Cout % 4 == 0) && (p.ld_y % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.y) & 15) == 0);
        const bool vres = vec && p.res != nullptr && (p.ld_res % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.res) & 15) == 0);
        const bool vbias = p.bias != nullptr && ((reinterpret_cast<uintptr_t>(p.bias) & 15) == 0) && (n0 % 4 == 0);
        for (int c0 = 0; c0 < p.bn; c0 += 16) {
            const int co = n0 + c0;
            const bool full16 = vec && co + 16 <= p.Cout;
            // residual rows of this chunk: 128-bit loads issued before the accumulator is drained
            float4 rv[4];
            if (row_ok && full16 && vres && !(p.mirror && t == 2)) {
                const float* rp = p.res + ((size_t)b * (p.Tout >> p.res_shift) + (t >> p.res_shift)) * p.ld_res + co;
#pragma unroll
                for (int i = 0; i < 4; ++i) rv[i] = __ldg(reinterpret_cast<const float4*>(rp) + i);
            }
            float v[16];
            tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);   // warp-collective
            if (!row_ok || co >= p.Cout) continue;
            if (full16 && vbias) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + co) + i);
                    v[4 * i] += bv.x; v[4 * i + 1] += bv.y; v[4 * i + 2] += bv.z; v[4 * i + 3] += bv.w;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    if (p.bias != nullptr && co + i < p.Cout) v[i] += __ldg(p.bias + co + i);
            }
            if (p.epi_gelu) {
                // ConvNeXt MLP (vocos.py:62-63): the exact-erf GELU of the first Linear, written as the 16-bit operand of the second
                uint32_t pk[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float g0 = 0.5f * v[2 * i] * (1.f + erff(v[2 * i] * 0.70710678118654752f));
                    const float g1 = 0.5f * v[2 * i + 1] * (1.f + erff(v[2 * i + 1] * 0.70710678118654752f));
                    if (p.is_bf16) {
                        const __nv_bfloat162 h = __floats2bfloat162_rn(g0, g1);
                        pk[i] = *reinterpret_cast<const uint32_t*>(&h);
                    } else {
                        const __half2 h = __floats2half2_rn(g0, g1);
                        pk[i] = *reinterpret_cast<const uint32_t*>(&h);
                    }
                }
                uint16_t* yp16 = reinterpret_cast<uint16_t*>(p.y) + ((size_t)b * p.Tout + t) * p.ld_y + co;
                if (full16) {
                    *reinterpret_cast<uint4*>(yp16) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    *reinterpret_cast<uint4*>(yp16 + 8) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
                } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i)
                        if (co + i < p.Cout) yp16[i] = (uint16_t)(pk[i >> 1] >> ((i & 1) * 16));
                }
                continue;
            }
            const int nrep = (p.mirror && t == 2) ? 2 : 1;
            for (int rep = 0; rep < nrep; ++rep) {
                const int tt = rep == 0 ? t : 0;
                float o[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) o[i] = v[i];
                if (p.res != nullptr) {
                    if (full16 && vres && nrep == 1) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            o[4 * i] += rv[i].x; o[4 * i + 1] += rv[i].y; o[4 * i + 2] += rv[i].z; o[4 * i + 3] += rv[i].w;
                        }
                    } else {
                        const float* rp = p.res + ((size_t)b * (p.Tout >> p.res_shift) + (tt >> p.res_shift)) * p.ld_res + co;
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            if (co + i < p.Cout) o[i] += rp[i];
                    }
                }
                float* yp = p.y + ((size_t)b * p.Tout + tt) * p.ld_y + co;
                if (full16) {
#pragma unroll
                    for (int i = 0; i < 16; i += 4) {
                        float4 r = make_float4(o[i], o[i + 1], o[i + 2], o[i + 3]);
                        if (p.accumulate) {
                            float4 old = *reinterpret_cast<const float4*>(yp + i);
                            r.x += old.x; r.y += old.y; r.z += old.z; r.w += old.w;
                        }
                        r.x *= p.scale; r.y *= p.scale; r.z *= p.scale; r.w *= p.scale;
                        *reinterpret_cast<float4*>(yp + i) = r;
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i)
                        if (co + i < p.Cout) yp[i] = ((p.accumulate ? yp[i] : 0.f) + o[i]) * p.scale;
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
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

static int make_map_3d(CUtensorMap* map, int is_bf16, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                       uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t b0, uint32_t b1, int sw64 = 0) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return ST2_ERR_CUDA;
    }
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
    cuuint32_t box[3] = {b0, b1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3,
                    const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    sw64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d) dims=[%llu,%llu,%llu] strides=[%llu,%llu] box=[%u,%u]", (int)r,
                  (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
                  (unsigned long long)stride1_bytes, (unsigned long long)stride2_bytes, b0, b1);
        return ST2_ERR_CUDA;
    }
    return ST2_OK;
}

// 16-bit, no swizzle: staging tiles of a 16-bit activation tensor
int make_act16_map_3d(CUtensorMap* map, int is_bf16, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                      uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t b0, uint32_t b1) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return ST2_ERR_CUDA;
    }
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
    cuuint32_t box[3] = {b0, b1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims,
                    strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled(act16) failed (%d)", (int)r);
        return ST2_ERR_CUDA;
    }
    return ST2_OK;
}

// fp32, no swizzle: the staging tiles of the fused kernel ([rows][C] row-major in shared memory)
int make_f32_map_3d(CUtensorMap* map, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                    uint64_t stride2_bytes, uint32_t b0, uint32_t b1) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return ST2_ERR_CUDA;
    }
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
    cuuint32_t box[3] = {b0, b1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled(f32) failed (%d) dims=[%llu,%llu,%llu] strides=[%llu,%llu] box=[%u,%u]", (int)r,
                  (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
                  (unsigned long long)stride1_bytes, (unsigned long long)stride2_bytes, b0, b1);
        return ST2_ERR_CUDA;
    }
    return ST2_OK;
}

// generic 3-D map: dtype 0 = fp32, 1 = bf16, 2 = fp16; no swizzle or SWIZZLE_128B (conv_pipe.cu rings)
int make_map_3d_any(CUtensorMap* map, int dtype, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                    uint64_t stride2_bytes, uint32_t b0, uint32_t b1, int swizzle128) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return ST2_ERR_CUDA;
    }
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
    cuuint32_t box[3] = {b0, b1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUtensorMapDataType dt = dtype == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                              : (dtype == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
    CUresult r = fn(map, dt, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled(any) failed (%d) dtype=%d dims=[%llu,%llu,%llu] strides=[%llu,%llu] box=[%u,%u] sw=%d", (int)r,
                  dtype, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
                  (unsigned long long)stride1_bytes, (unsigned long long)stride2_bytes, b0, b1, swizzle128);
        return ST2_ERR_CUDA;
    }
    return ST2_OK;
}

// generic 3-D map with an explicit swizzle mode (0 none, 64 = SWIZZLE_64B, 128 = SWIZZLE_128B): the fp16 residual tiles of
// conv_row.cu, which land in shared memory in the K-major UMMA operand layout
int make_map_3d_sw(CUtensorMap* map, int dtype, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                   uint64_t stride2_bytes, uint32_t b0, uint32_t b1, int swizzle_bytes) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return ST2_ERR_CUDA;
    }
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
    cuuint32_t box[3] = {b0, b1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUtensorMapDataType dt = dtype == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                              : (dtype == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
    const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                                       : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE);
    CUresult r = fn(map, dt, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled(sw) failed (%d) dtype=%d dims=[%llu,%llu,%llu] strides=[%llu,%llu] box=[%u,%u] sw=%d", (int)r,
                  dtype, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
                  (unsigned long long)stride1_bytes, (unsigned long long)stride2_bytes, b0, b1, swizzle_bytes);
        return ST2_ERR_CUDA;
    }
    return ST2_OK;
}

// fp32 [B][T][C] tensor viewed as (c, phase, m, b) with t = m*phases + phase: 128-byte-swizzled boxes of b0 channels x b2
// rows m of one phase (the residual boxes of conv_pipe.cu; phases = 1 for a plain convolution)
int make_map_4d_f32_sw128(CUtensorMap* map, const void* base, uint64_t C, uint64_t phases, uint64_t rows, uint64_t B,
                          uint64_t ld_bytes, uint64_t batch_bytes, uint32_t b0, uint32_t b2) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return ST2_ERR_CUDA;
    }
    cuuint64_t dims[4] = {C, phases, rows, B};
    cuuint64_t strides[3] = {ld_bytes, ld_bytes * phases, batch_bytes};
    cuuint32_t box[4] = {b0, 1, b2, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled(4d) failed (%d) dims=[%llu,%llu,%llu,%llu] ld=%llu batch=%llu", (int)r,
                  (unsigned long long)C, (unsigned long long)phases, (unsigned long long)rows, (unsigned long long)B,
                  (unsigned long long)ld_bytes, (unsigned long long)batch_bytes);
        return ST2_ERR_CUDA;
    }
    return ST2_OK;
}

// fp16 [B][T][C] tensor viewed as (c, 1, t, b): 64-byte-swizzled boxes of b0 = 32 channels x b2 rows (the fp16 residual boxes
// of conv_pipe.cu; same coordinate order as make_map_4d_f32_sw128 so the producer issues both the same way)
int make_map_4d_f16_sw64(CUtensorMap* map, const void* base, uint64_t C, uint64_t rows, uint64_t B, uint64_t ld_bytes,
                         uint64_t batch_bytes, uint32_t b0, uint32_t b2) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        return ST2_ERR_CUDA;
    }
    cuuint64_t dims[4] = {C, 1, rows, B};
    cuuint64_t strides[3] = {ld_bytes, ld_bytes, batch_bytes};
    cuuint32_t box[4] = {b0, 1, b2, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled(4d f16) failed (%d) dims=[%llu,1,%llu,%llu] ld=%llu batch=%llu", (int)r,
                  (unsigned long long)C, (unsigned long long)rows, (unsigned long long)B, (unsigned long long)ld_bytes,
                  (unsigned long long)batch_bytes);
        return ST2_ERR_CUDA;
    }
    return ST2_OK;
}

int make_weight_map(CUtensorMap* map, int is_bf16, const void* w16, int cin_pad, int cout_pad, int ktaps, int bn) {
    return make_map_3d(map, is_bf16, w16, (uint64_t)cin_pad, (uint64_t)cout_pad, (uint64_t)ktaps, (uint64_t)cin_pad * 2,
                       (uint64_t)cin_pad * cout_pad * 2, TC_KC, (uint32_t)bn);
}
// K = 32 tiles (64-byte rows, SWIZZLE_64B): the first 32 input channels of every [CoutPad][CinPad] tap
int make_weight_map_k32(CUtensorMap* map, int is_bf16, const void* w16, int cin_pad, int cout_pad, int ktaps, int bn) {
    return make_map_3d(map, is_bf16, w16, (uint64_t)cin_pad, (uint64_t)cout_pad, (uint64_t)ktaps, (uint64_t)cin_pad * 2,
                       (uint64_t)cin_pad * cout_pad * 2, 32, (uint32_t)bn, 1);
}

bool conv_tc_supported(const ConvArgs& a) {
    return a.x16 != nullptr && a.w16 != nullptr && a.in_stride == 1 && a.w16_cin_pad % TC_KC == 0 &&
           a.w16_cout_pad % 16 == 0 && a.ld_x16 % 8 == 0;
}

int launch_conv_tc(const ConvArgs& a, cudaStream_t st) {
    ST2_REQUIRE(conv_tc_supported(a), "conv_tc: unsupported geometry (in_stride=%d cin_pad=%d cout_pad=%d ld=%d)",
                a.in_stride, a.w16_cin_pad, a.w16_cout_pad, a.ld_x16);
    const int is_bf16 = a.fmt16 == DT_BF16 ? 1 : 0;
    TcParams p;
    memset(&p, 0, sizeof(p));
    p.bias = a.bias; p.res = a.res; p.ld_res = a.ld_res; p.res_shift = a.res_shift;
    p.y = a.y; p.ld_y = a.ld_y; p.Tout = a.Tout; p.Cout = a.Cout; p.M = a.M;
    p.ntaps = a.ntaps; p.tap_step = a.tap_step; p.in_off = a.in_off;
    p.phases = a.phases; p.w_step = a.w_step; p.out_stride = a.out_stride; p.out_pad = a.out_pad;
    p.kchunks = a.w16_cin_pad / TC_KC;
    p.scale = a.scale; p.accumulate = a.accumulate; p.mirror = a.mirror; p.is_bf16 = is_bf16;
    p.epi_gelu = a.epi_gelu;
    ST2_REQUIRE(!a.epi_gelu || (a.res == nullptr && !a.accumulate && a.scale == 1.f && !a.mirror && a.ld_y % 8 == 0 &&
                                (reinterpret_cast<uintptr_t>(a.y) & 15) == 0),
                "conv_tc: the GELU epilogue takes no residual / accumulate / scale and needs a 16-byte aligned 16-bit output");
    // N tile: whole CoutPad up to 256, else the largest multiple-of-16 divisor <= 256
    int bn = a.w16_cout_pad;
    if (bn > 256) {
        bn = 256;
        while (a.w16_cout_pad % bn != 0) bn -= 16;
    }
    p.bn = bn;
    int cols = 32;
    while (cols < bn) cols <<= 1;
    p.tmem_cols = cols;
    const uint32_t stage_bytes = A_STAGE_BYTES + (uint32_t)bn * TC_KC * 2;
    int stages = (int)(96 * 1024 / stage_bytes);   // <= 96 KB: two CTAs per SM
    if (stages > 6) stages = 6;
    if (stages < 2) stages = 2;
    p.stages = stages;
    const size_t smem = (size_t)stages * stage_bytes + (2 * stages + 2) * sizeof(uint64_t) + 16 + 1024;

    CUtensorMap map_a, map_b;
    const int ktaps_total = a.phases > 1 ? a.ntaps * a.phases : a.ntaps;   // weight taps stored
    const uint64_t a_d0 = (uint64_t)(a.ld_x16 < a.w16_cin_pad ? a.ld_x16 : a.w16_cin_pad);
    int e = make_map_3d(&map_a, is_bf16, a.x16, a_d0, (uint64_t)a.Tin, (uint64_t)a.B, (uint64_t)a.ld_x16 * 2,
                        (uint64_t)a.Tin * a.ld_x16 * 2, TC_KC, (uint32_t)TC_BM);
    if (e != ST2_OK) return e;
    e = make_map_3d(&map_b, is_bf16, a.w16, (uint64_t)a.w16_cin_pad, (uint64_t)a.w16_cout_pad, (uint64_t)ktaps_total,
                    (uint64_t)a.w16_cin_pad * 2, (uint64_t)a.w16_cin_pad * a.w16_cout_pad * 2, TC_KC, (uint32_t)bn);
    if (e != ST2_OK) return e;

    static bool attr_set[kMaxDevices] = {};      // per device (the attribute applies to the current device)
    if (!attr_set[current_device_slot()]) {
        ST2_CUDA_CHECK(cudaFuncSetAttribute(conv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr_set[current_device_slot()] = true;
    }
    dim3 grid(cdiv(a.M, TC_BM), a.w16_cout_pad / bn, a.B * a.phases);
    conv_tc_kernel<<<grid, TC_THREADS, smem, st>>>(map_a, map_b, p);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

}  // namespace st2
