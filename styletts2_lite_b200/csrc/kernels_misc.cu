// Small layout / front-end / load-time kernels of the decoder.
#include "common.cuh"

namespace st2 {

// ---- [B,C,T] (reference layout) -> channels-last [B,T,ld] ------------------------------
__global__ void cf_to_cl_kernel(const float* __restrict__ src, float* __restrict__ dst, int ld, int C, int T) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += 8) {
        int c = c0 + i, t = t0 + threadIdx.x;
        tile[i][threadIdx.x] = (c < C && t < T) ? src[((size_t)b * C + c) * T + t] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += 8) {
        int t = t0 + i, c = c0 + threadIdx.x;
        if (t < T && c < C) dst[((size_t)b * T + t) * ld + c] = tile[threadIdx.x][i];
    }
}

int launch_cf_to_cl(const float* src, float* dst, int ld_dst, int B, int C, int T, cudaStream_t st) {
    dim3 grid(cdiv(T, 32), cdiv(C, 32), B), block(32, 8);
    cf_to_cl_kernel<<<grid, block, 0, st>>>(src, dst, ld_dst, C, T);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---- F0_conv / N_conv: Conv1d(1,1,k=3,stride=2,pad=1) (hifigan.py:434-436,458-459) --------
// Writes F0,N into the channel slots c0,c0+1 of the 514-wide and c1,c1+1 of the 1090-wide
// concat buffers (torch.cat of hifigan.py:461,469) and zeroes their padding channels.
__global__ void f0n_conv_kernel(const float* __restrict__ f0, const float* __restrict__ nn,
                                const float* __restrict__ wf, const float* __restrict__ bf,
                                const float* __restrict__ wn, const float* __restrict__ bn,
                                float* __restrict__ dst0, int ld0, int c0, int pad0_from,
                                float* __restrict__ dst1, int ld1, int c1, int pad1_from, int T) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (t >= T) return;
    const int L2 = 2 * T;
    const float* fb = f0 + (size_t)b * L2;
    const float* nb = nn + (size_t)b * L2;
    float af = bf[0], an = bn[0];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        int i = 2 * t + k - 1;
        if (i >= 0 && i < L2) {
            af = fmaf(wf[k], fb[i], af);
            an = fmaf(wn[k], nb[i], an);
        }
    }
    float* r0 = dst0 + ((size_t)b * T + t) * ld0;
    r0[c0] = af;
    r0[c0 + 1] = an;
    for (int c = pad0_from; c < ld0; ++c) r0[c] = 0.f;
    float* r1 = dst1 + ((size_t)b * T + t) * ld1;
    r1[c1] = af;
    r1[c1 + 1] = an;
    for (int c = pad1_from; c < ld1; ++c) r1[c] = 0.f;
}

int launch_f0n_conv(const float* f0, const float* n, const float* wf, const float* bf, const float* wn,
                    const float* bn, float* dst0, int ld0, int c0, int pad0_from, float* dst1, int ld1, int c1,
                    int pad1_from, int B, int T, cudaStream_t st) {
    dim3 grid(cdiv(T, 128), B);
    f0n_conv_kernel<<<grid, 128, 0, st>>>(f0, n, wf, bf, wn, bn, dst0, ld0, c0, pad0_from, dst1, ld1, c1,
                                          pad1_from, T);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---- all AdaIN fc layers at once: h[B][R] = s[B][K] @ W[R][K]^T + bias[R] ------------------
// (the 106 nn.Linear(style_dim, 2C) of hifigan.py:18,21).  CTA = 64 utterances x 4 row quads: the style vectors of up to
// 64 utterances sit in shared memory as [k][b] (conflict-free for consecutive b), every thread owns 4 consecutive output
// rows of one utterance, reads their weight rows with warp-uniform 128-bit loads and writes one float4.  Style vectors longer
// than kFcK are staged kFcK entries at a time (64 KB of shared memory); the summation order stays k = 0..K-1.
static constexpr int kFcB = 64, kFcRq = 4, kFcK = 256;
__global__ void __launch_bounds__(kFcB * kFcRq)
style_fc_kernel(const float* __restrict__ s, const float* __restrict__ W, const float* __restrict__ bias,
                float* __restrict__ h, int B, int R, int K) {
    extern __shared__ float ssm[];                    // [min(K, kFcK)][kFcB]
    const int b0 = blockIdx.y * kFcB;
    const int bb = threadIdx.x % kFcB, rq = threadIdx.x / kFcB;
    const int r = (blockIdx.x * kFcRq + rq) * 4;
    const bool active = r < R && b0 + bb < B;
    const int nr = min(4, R - r);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k0 = 0; k0 < K; k0 += kFcK) {
        const int kc = min(kFcK, K - k0);
        if (k0 > 0) __syncthreads();                  // every thread is done with the previous chunk
        for (int i = threadIdx.x; i < kc * kFcB; i += kFcB * kFcRq) {
            const int ib = i / kc, k = i - ib * kc;   // coalesced read of s, transposed write
            ssm[k * kFcB + ib] = (b0 + ib < B) ? s[(size_t)(b0 + ib) * K + k0 + k] : 0.f;
        }
        __syncthreads();
        if (!active) continue;
        for (int k = 0; k < kc; k += 4) {
            const float s0 = ssm[(k + 0) * kFcB + bb], s1 = ssm[(k + 1) * kFcB + bb], s2 = ssm[(k + 2) * kFcB + bb],
                        s3 = ssm[(k + 3) * kFcB + bb];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (j < nr) {
                    const float4 w = __ldg(reinterpret_cast<const float4*>(W + (size_t)(r + j) * K + k0 + k));   // same order as k = 0..K-1
                    acc[j] = fmaf(w.x, s0, acc[j]); acc[j] = fmaf(w.y, s1, acc[j]);
                    acc[j] = fmaf(w.z, s2, acc[j]); acc[j] = fmaf(w.w, s3, acc[j]);
                }
            }
        }
    }
    if (!active) return;
    float* hp = h + (size_t)(b0 + bb) * R + r;
    for (int j = 0; j < nr; ++j) hp[j] = acc[j] + bias[r + j];
}

int launch_style_fc(const float* s, const float* W, const float* bias, float* h, int B, int R, int K,
                    cudaStream_t st) {
    ST2_REQUIRE(K % 4 == 0 && K <= 1024, "style_fc: style_dim %d must be a multiple of 4 and <= 1024", K);
    dim3 grid(cdiv(R, 4 * kFcRq), cdiv(B, kFcB));
    const size_t smem = (size_t)min(K, kFcK) * kFcB * sizeof(float);
    static size_t max_set[kMaxDevices] = {};     // per device (the attribute applies to the current device)
    size_t& ms = max_set[current_device_slot()];
    if (smem > 48 * 1024 && smem > ms) {
        ST2_CUDA_CHECK(cudaFuncSetAttribute(style_fc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ms = smem;
    }
    style_fc_kernel<<<grid, kFcB * kFcRq, smem, st>>>(s, W, bias, h, B, R, K);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---- AdainResBlk1d.pool: depthwise ConvTranspose1d(k=3,s=2,p=1,op=1) (hifigan.py:373) ------
// w packed [3][Cpad], bias [Cpad].  y[2q] = b + x[q]*w1 ; y[2q+1] = b + x[q]*w2 + x[q+1]*w0.
__global__ void pool_dw_kernel(const float* __restrict__ x, int ld_x, const float* __restrict__ w,
                               const float* __restrict__ bias, float* __restrict__ y, int ld_y, int T, int Cpad) {
    const int cq = Cpad >> 2;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    const size_t total = (size_t)2 * T * cq;
    if (i >= total) return;
    const int to = (int)(i / cq);
    const int c = (int)(i - (size_t)to * cq) * 4;
    const int q = to >> 1;
    const float* xb = x + (size_t)b * T * ld_x;
    float4 bv = *reinterpret_cast<const float4*>(bias + c);
    float4 x0 = *reinterpret_cast<const float4*>(xb + (size_t)q * ld_x + c);
    float4 o;
    if ((to & 1) == 0) {
        float4 w1 = *reinterpret_cast<const float4*>(w + Cpad + c);
        o.x = fmaf(x0.x, w1.x, bv.x); o.y = fmaf(x0.y, w1.y, bv.y);
        o.z = fmaf(x0.z, w1.z, bv.z); o.w = fmaf(x0.w, w1.w, bv.w);
    } else {
        float4 w2 = *reinterpret_cast<const float4*>(w + 2 * Cpad + c);
        o.x = fmaf(x0.x, w2.x, bv.x); o.y = fmaf(x0.y, w2.y, bv.y);
        o.z = fmaf(x0.z, w2.z, bv.z); o.w = fmaf(x0.w, w2.w, bv.w);
        if (q + 1 < T) {
            float4 w0 = *reinterpret_cast<const float4*>(w + c);
            float4 x1 = *reinterpret_cast<const float4*>(xb + (size_t)(q + 1) * ld_x + c);
            o.x = fmaf(x1.x, w0.x, o.x); o.y = fmaf(x1.y, w0.y, o.y);
            o.z = fmaf(x1.z, w0.z, o.z); o.w = fmaf(x1.w, w0.w, o.w);
        }
    }
    *reinterpret_cast<float4*>(y + ((size_t)b * 2 * T + to) * ld_y + c) = o;
}

int launch_pool_dw(const float* x, int ld_x, const float* w, const float* bias, float* y, int ld_y, int B, int T,
                   int C, int Cpad, cudaStream_t st) {
    (void)C;
    size_t total = (size_t)2 * T * (Cpad / 4);
    dim3 grid(cdiv(total, 256), B);
    pool_dw_kernel<<<grid, 256, 0, st>>>(x, ld_x, w, bias, y, ld_y, T, Cpad);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---- hifigan tail: Snake(alphas[-1]) -> conv_post(C->1,k=7,p=3) -> tanh (hifigan.py:343-345) --
// HBM-bound on its input (4*C bytes per sample).  The Snake'd tile lives in shared memory with a pitch of C+4 floats
// (16-byte aligned rows, conflict-free 128-bit reads for consecutive rows); FAST selects sin.approx / approximate
// reciprocal for the 16-bit precisions (the fp32 parity path keeps sinf).
static constexpr int kPostTile = 256;
template <bool FAST, bool X16>
__global__ void __launch_bounds__(kPostTile)
post_hifigan_kernel(const float* __restrict__ x, int ld_x, const float* __restrict__ alpha,
                    const float* __restrict__ w /*[7][C]*/, const float* __restrict__ bias,
                    float* __restrict__ out, int S, int C) {
    extern __shared__ __align__(16) float sm[];
    const int pitch = C + 4;
    float* tile = sm;                                  // [(kPostTile+6)][C+4]
    float* sw = sm + (kPostTile + 6) * pitch;          // [7][C]
    const int b = blockIdx.y;
    const int t0 = blockIdx.x * kPostTile;
    for (int i = threadIdx.x; i < 7 * C; i += kPostTile) sw[i] = w[i];
    const int cq = C >> 2;
    for (int i = threadIdx.x; i < (kPostTile + 6) * cq; i += kPostTile) {
        int r = i / cq, c = (i - r * cq) * 4;
        int t = t0 + r - 3;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t >= 0 && t < S) {
            if (X16) {                                 // the last stage's output stored as fp16 (option fp16_out)
                const uint2 u = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(x) + ((size_t)b * S + t) * ld_x + c));
                const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
                const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
                v = make_float4(lo.x, lo.y, hi.x, hi.y);
            } else {
                v = __ldg(reinterpret_cast<const float4*>(x + ((size_t)b * S + t) * ld_x + c));
            }
            float4 al = *reinterpret_cast<const float4*>(alpha + c);
            if (FAST) {
                float s0 = __sinf(al.x * v.x), s1 = __sinf(al.y * v.y), s2 = __sinf(al.z * v.z), s3 = __sinf(al.w * v.w);
                v.x = fmaf(__fdividef(1.f, al.x) * s0, s0, v.x);
                v.y = fmaf(__fdividef(1.f, al.y) * s1, s1, v.y);
                v.z = fmaf(__fdividef(1.f, al.z) * s2, s2, v.z);
                v.w = fmaf(__fdividef(1.f, al.w) * s3, s3, v.w);
            } else {
                float s0 = sinf(al.x * v.x), s1 = sinf(al.y * v.y), s2 = sinf(al.z * v.z), s3 = sinf(al.w * v.w);
                v.x = fmaf((1.f / al.x) * s0, s0, v.x);
                v.y = fmaf((1.f / al.y) * s1, s1, v.y);
                v.z = fmaf((1.f / al.z) * s2, s2, v.z);
                v.w = fmaf((1.f / al.w) * s3, s3, v.w);
            }
        }
        *reinterpret_cast<float4*>(tile + r * pitch + c) = v;
    }
    __syncthreads();
    const int t = t0 + threadIdx.x;
    if (t >= S) return;
    float acc = bias[0];
    for (int k = 0; k < 7; ++k) {
        const float4* row = reinterpret_cast<const float4*>(tile + (threadIdx.x + k) * pitch);
        const float4* wk = reinterpret_cast<const float4*>(sw + k * C);
        for (int c = 0; c < cq; ++c) {                 // same summation order as the scalar loop
            const float4 rv = row[c], wv = wk[c];
            acc = fmaf(wv.x, rv.x, acc); acc = fmaf(wv.y, rv.y, acc);
            acc = fmaf(wv.z, rv.z, acc); acc = fmaf(wv.w, rv.w, acc);
        }
    }
    out[(size_t)b * S + t] = tanhf(acc);
}

int launch_post_hifigan(const float* x, int ld_x, const float* alpha, const float* w, const float* bias,
                        float* out, int B, int S, int C, int fast, cudaStream_t st, int x16) {
    ST2_REQUIRE(!x16 || fast, "post_hifigan: fp16 input only on the 16-bit paths");
    ST2_REQUIRE(C % 4 == 0 && C <= 64 && ld_x % 4 == 0, "post_hifigan: C=%d ld=%d unsupported", C, ld_x);
    size_t smem = ((size_t)(kPostTile + 6) * (C + 4) + 7 * C) * sizeof(float);
    if (smem > 48 * 1024) {
        ST2_CUDA_CHECK(cudaFuncSetAttribute(post_hifigan_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ST2_CUDA_CHECK(cudaFuncSetAttribute(post_hifigan_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ST2_CUDA_CHECK(cudaFuncSetAttribute(post_hifigan_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    dim3 grid(cdiv(S, kPostTile), B);
    if (x16) post_hifigan_kernel<true, true><<<grid, kPostTile, smem, st>>>(x, ld_x, alpha, w, bias, out, S, C);
    else if (fast) post_hifigan_kernel<true, false><<<grid, kPostTile, smem, st>>>(x, ld_x, alpha, w, bias, out, S, C);
    else post_hifigan_kernel<false, false><<<grid, kPostTile, smem, st>>>(x, ld_x, alpha, w, bias, out, S, C);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---- dst = a + b (pack time: a conv bias with the offset of a bias-free fp16 input folded in)
__global__ void add_vec_kernel(float* __restrict__ dst, const float* __restrict__ a, const float* __restrict__ b, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = a[i] + b[i];
}

int launch_add_vec(float* dst, const float* a, const float* b, int n, cudaStream_t st) {
    add_vec_kernel<<<cdiv(n, 256), 256, 0, st>>>(dst, a, b, n);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---- fp16 -> fp32 (debug taps of the fp16 intra-block tensor)
__global__ void half_to_float_kernel(const __half* __restrict__ src, float* __restrict__ dst, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = __half2float(src[i]);
}

int launch_half_to_float(const void* src, float* dst, int64_t n, cudaStream_t st) {
    half_to_float_kernel<<<cdiv(n, 256), 256, 0, st>>>((const __half*)src, dst, n);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---- dense copy of a pitched channels-last tensor (debug taps) ------------------------------
__global__ void copy_dense_kernel(const float* __restrict__ src, int ld, float* __restrict__ dst, int64_t rows,
                                  int C) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * C) return;
    int64_t r = i / C;
    int c = (int)(i - r * C);
    dst[i] = src[r * ld + c];
}

int launch_copy_dense(const float* src, int ld, float* dst, int64_t rows, int C, cudaStream_t st) {
    copy_dense_kernel<<<cdiv(rows * C, 256), 256, 0, st>>>(src, ld, dst, rows, C);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---- load time: weight-norm fold + repack to tap-major [k][Cin][Cout] ------------------------
// torch._weight_norm(v, g, 0): w = v * g / ||v|| with the norm over all dims but 0.
// Conv1d: v [Cout][Cin][k] (d0=Cout,d1=Cin);  ConvTranspose1d: v [Cin][Cout][k] (d0=Cin,d1=Cout).
__global__ void fold_pack_kernel(const float* __restrict__ g, const float* __restrict__ v, float* __restrict__ wp,
                                 int d0, int d1, int k, int transposed) {
    const int r = blockIdx.x;
    const int n = d1 * k;
    const float* vr = v + (size_t)r * n;
    __shared__ double red[256];
    __shared__ float s_scale;
    double ss = 0;
    if (g != nullptr)
        for (int i = threadIdx.x; i < n; i += blockDim.x) ss += (double)vr[i] * (double)vr[i];
    red[threadIdx.x] = ss;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) s_scale = (g != nullptr) ? g[r] / (float)sqrt(red[0]) : 1.f;
    __syncthreads();
    const float sc = s_scale;
    const int Cin = transposed ? d0 : d1;
    const int Cout = transposed ? d1 : d0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        int j = i / k, kk = i - j * k;          // j indexes d1
        int ci = transposed ? r : j;
        int co = transposed ? j : r;
        wp[((size_t)kk * Cin + ci) * Cout + co] = vr[i] * sc;
    }
}

int launch_fold_pack(const float* g, const float* v, float* wp, int d0, int d1, int k, int transposed,
                     cudaStream_t st) {
    fold_pack_kernel<<<d0, 256, 0, st>>>(g, v, wp, d0, d1, k, transposed);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---- load time: fp32 [k][Cin][Cout] -> 16-bit [k][CoutPad][CinPad] (K-major B operand) -------
__global__ void pack_w16_kernel(const float* __restrict__ wp, void* __restrict__ w16, int k, int Cin, int Cout,
                                int CinPad, int CoutPad, int dt) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)k * CoutPad * CinPad;
    if (i >= total) return;
    int ci = (int)(i % CinPad);
    int co = (int)((i / CinPad) % CoutPad);
    int kk = (int)(i / ((size_t)CinPad * CoutPad));
    float v = (ci < Cin && co < Cout) ? wp[((size_t)kk * Cin + ci) * Cout + co] : 0.f;
    if (dt == DT_BF16)
        reinterpret_cast<__nv_bfloat16*>(w16)[i] = __float2bfloat16_rn(v);
    else
        reinterpret_cast<__half*>(w16)[i] = __float2half_rn(v);
}

int launch_cast16(const float* src, void* dst, int64_t n, int out_dtype, cudaStream_t st) {
    // contiguous cast == pack with k=1, Cout=1, Cin=n
    pack_w16_kernel<<<cdiv(n, 256), 256, 0, st>>>(src, dst, 1, (int)n, 1, (int)n, 1, out_dtype);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

int launch_pack_w16(const float* wp, void* w16, int k, int Cin, int Cout, int CinPad, int CoutPad, int out_dtype,
                    cudaStream_t st) {
    size_t total = (size_t)k * CoutPad * CinPad;
    pack_w16_kernel<<<cdiv(total, 256), 256, 0, st>>>(wp, w16, k, Cin, Cout, CinPad, CoutPad, out_dtype);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

}  // namespace st2

namespace st2 {

// ---- generator.noise_convs[i] (hifigan.py:296-303,330): Conv1d(1 -> C, kernel k, stride s, padding p) of the
// harmonic source har[B][S] -> y[B][Tout][C] channels-last, plus per-tile (sum, sumsq) per channel for the AdaIN
// that follows (noise_res[i].adain1[0]).  HBM-bound on its output (4*C bytes per output step); weights and the
// har segment of the tile live in shared memory.
// output time steps per CTA (weights + har segment are staged once per tile): 1024 for the small strides of the late stages
// (the k = 1 conv of the last stage was bound by CTA turnover with 256: 30,000 CTAs of 16 KB of output each: 0.25 -> 0.15 ms;
// stride 2: 0.23 -> 0.20 ms), 256 for the compute-heavy early stages (stride 6 measured slower with 1024; stride 30: 256 steps
// already read 7,700 samples)
static int nc_tile(int stride) { return stride <= 2 ? 1024 : 256; }
// Y16: y is stored as fp16 (the block input of noise_res[i], read twice by its first iteration) WITHOUT the bias: with one
// input channel every output channel is bias[c] + w[.][c] * har, and a bias larger than the signal would eat the fp16 mantissa
// that the InstanceNorm behind it then magnifies (measured 4e-2 relative L2 on noise_res.3 with the bias stored).  The consumers
// add it back: the AdaIN coefficients get the offset (launch_adain_coef_f2) and the residual add of the first iteration has it
// folded into that conv's bias (decoder.cu).
// The accumulator and the (sum, sumsq) partials are of y - bias[c]: for the k = 1 conv of the last stage a channel's mean is up
// to ~500x its std with the reference initialisation, and E[y^2] - mean^2 of fp32 partials of y itself lost 3e-4 of rstd.  The
// coefficient kernel gets the bias as the statistics' shift; the bias is added only where y is stored as fp32.
template <bool Y16, int kNcTile>
__global__ void __launch_bounds__(256)
noise_conv_kernel(const float* __restrict__ har, const float* __restrict__ w /*[k][C]*/, const float* __restrict__ bias,
                  float* __restrict__ y, float2* __restrict__ stats, int S, int Tout, int C, int k, int stride, int pad,
                  int ntile) {
    extern __shared__ float sm[];
    float* sw = sm;                                   // [k][C]
    float* sh = sm + (size_t)k * C;                   // [(kNcTile-1)*stride + k]
    float* sred = sh + (kNcTile - 1) * stride + k;    // [rows_per_pass][C][2]
    const int b = blockIdx.y, tile = blockIdx.x;
    const int t0 = tile * kNcTile;
    for (int i = threadIdx.x; i < k * C; i += 256) sw[i] = w[i];
    const int seg = (kNcTile - 1) * stride + k;
    const int h0 = t0 * stride - pad;
    for (int i = threadIdx.x; i < seg; i += 256) {
        const int hi = h0 + i;
        sh[i] = (hi >= 0 && hi < S) ? har[(size_t)b * S + hi] : 0.f;
    }
    __syncthreads();
    const int cq = C >> 2;                            // channel quads
    const int rpp = 256 / cq;                         // rows per pass
    const int q = threadIdx.x % cq, rl = threadIdx.x / cq;
    const float4 bv = *reinterpret_cast<const float4*>(bias + q * 4);
    float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
    // 4 rows x 4 channels per thread: one 128-bit weight read per tap feeds 16 FMAs
    for (int r = rl; r < kNcTile; r += 4 * rpp) {
        if (t0 + r >= Tout) break;
        float4 acc[4] = {};
        const float* hp = sh + r * stride;
        const int hstep = rpp * stride;
        for (int j = 0; j < k; ++j) {
            const float4 wv = *reinterpret_cast<const float4*>(sw + (size_t)j * C + q * 4);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float hv = (r + u * rpp < kNcTile) ? hp[u * hstep + j] : 0.f;
                acc[u].x = fmaf(hv, wv.x, acc[u].x); acc[u].y = fmaf(hv, wv.y, acc[u].y);
                acc[u].z = fmaf(hv, wv.z, acc[u].z); acc[u].w = fmaf(hv, wv.w, acc[u].w);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int ru = r + u * rpp, t = t0 + ru;
            if (ru >= kNcTile || t >= Tout) break;
            if (Y16) {
                const __half2 lo = __floats2half2_rn(acc[u].x, acc[u].y), hi = __floats2half2_rn(acc[u].z, acc[u].w);
                *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(y) + ((size_t)b * Tout + t) * C + q * 4) =
                    make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
            } else {
                *reinterpret_cast<float4*>(y + ((size_t)b * Tout + t) * C + q * 4) =
                    make_float4(acc[u].x + bv.x, acc[u].y + bv.y, acc[u].z + bv.z, acc[u].w + bv.w);
            }
            s1[0] += acc[u].x; s1[1] += acc[u].y; s1[2] += acc[u].z; s1[3] += acc[u].w;
            s2[0] = fmaf(acc[u].x, acc[u].x, s2[0]); s2[1] = fmaf(acc[u].y, acc[u].y, s2[1]);
            s2[2] = fmaf(acc[u].z, acc[u].z, s2[2]); s2[3] = fmaf(acc[u].w, acc[u].w, s2[3]);
        }
    }
    if (stats == nullptr) return;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        sred[((size_t)rl * C + q * 4 + i) * 2 + 0] = s1[i];
        sred[((size_t)rl * C + q * 4 + i) * 2 + 1] = s2[i];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += 256) {
        float a = 0.f, s = 0.f;
        for (int r = 0; r < rpp; ++r) {               // fixed order: deterministic
            a += sred[((size_t)r * C + c) * 2 + 0];
            s += sred[((size_t)r * C + c) * 2 + 1];
        }
        stats[((size_t)b * ntile + tile) * C + c] = make_float2(a, s);
    }
}

int noise_conv_parts(int Tout, int stride) { return cdiv(Tout, nc_tile(stride)); }

int launch_noise_conv(const float* har, const float* w, const float* bias, float* y, void* stats, int B, int S, int Tout,
                      int C, int k, int stride, int pad, cudaStream_t st, int y16) {
    ST2_REQUIRE(C % 4 == 0 && C <= 1024 && 256 % (C / 4) == 0 && bias != nullptr, "noise_conv: unsupported C=%d", C);
    const int kNcTile = nc_tile(stride);
    const int ntile = cdiv(Tout, kNcTile);
    const int rpp = 256 / (C / 4);
    size_t smem = ((size_t)k * C + (kNcTile - 1) * stride + k + (size_t)rpp * C * 2) * sizeof(float);
    static size_t max_set[kMaxDevices] = {};     // per device (the attribute applies to the current device)
    size_t& ms = max_set[current_device_slot()];
    if (smem > 48 * 1024 && smem > ms) {
        ST2_CUDA_CHECK(cudaFuncSetAttribute(noise_conv_kernel<false, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ST2_CUDA_CHECK(cudaFuncSetAttribute(noise_conv_kernel<true, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ST2_CUDA_CHECK(cudaFuncSetAttribute(noise_conv_kernel<false, 1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ST2_CUDA_CHECK(cudaFuncSetAttribute(noise_conv_kernel<true, 1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ms = smem;
    }
    dim3 grid(ntile, B);
#define ST2_NC_LAUNCH(Y16_, TILE_) noise_conv_kernel<Y16_, TILE_><<<grid, 256, smem, st>>>(har, w, bias, y, (float2*)stats, S, Tout, C, k, stride, pad, ntile)
    if (kNcTile == 1024) { if (y16) ST2_NC_LAUNCH(true, 1024); else ST2_NC_LAUNCH(false, 1024); }
    else { if (y16) ST2_NC_LAUNCH(true, 256); else ST2_NC_LAUNCH(false, 256); }
#undef ST2_NC_LAUNCH
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

// ---- depthwise pool with a 16-bit output (operand of the tensor-core conv1 of the upsampling AdainResBlk1d)
template <int DT>
__global__ void pool_dw16_kernel(const float* __restrict__ x, int ld_x, const float* __restrict__ w,
                                 const float* __restrict__ bias, void* __restrict__ y, int ld_y, int T, int Cpad) {
    const int cq = Cpad >> 2;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    const size_t total = (size_t)2 * T * cq;
    if (i >= total) return;
    const int to = (int)(i / cq);
    const int c = (int)(i - (size_t)to * cq) * 4;
    const int q = to >> 1;
    const float* xb = x + (size_t)b * T * ld_x;
    const float4 bv = *reinterpret_cast<const float4*>(bias + c);
    const float4 x0 = *reinterpret_cast<const float4*>(xb + (size_t)q * ld_x + c);
    float4 o;
    if ((to & 1) == 0) {
        const float4 w1 = *reinterpret_cast<const float4*>(w + Cpad + c);
        o.x = fmaf(x0.x, w1.x, bv.x); o.y = fmaf(x0.y, w1.y, bv.y);
        o.z = fmaf(x0.z, w1.z, bv.z); o.w = fmaf(x0.w, w1.w, bv.w);
    } else {
        const float4 w2 = *reinterpret_cast<const float4*>(w + 2 * Cpad + c);
        o.x = fmaf(x0.x, w2.x, bv.x); o.y = fmaf(x0.y, w2.y, bv.y);
        o.z = fmaf(x0.z, w2.z, bv.z); o.w = fmaf(x0.w, w2.w, bv.w);
        if (q + 1 < T) {
            const float4 w0 = *reinterpret_cast<const float4*>(w + c);
            const float4 x1 = *reinterpret_cast<const float4*>(xb + (size_t)(q + 1) * ld_x + c);
            o.x = fmaf(x1.x, w0.x, o.x); o.y = fmaf(x1.y, w0.y, o.y);
            o.z = fmaf(x1.z, w0.z, o.z); o.w = fmaf(x1.w, w0.w, o.w);
        }
    }
    const size_t idx = ((size_t)b * 2 * T + to) * ld_y + c;
    uint2 u;
    if (DT == DT_BF16) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
        u.x = *reinterpret_cast<uint32_t*>(&lo); u.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(y) + idx) = u;
    } else {
        __half2 lo = __floats2half2_rn(o.x, o.y), hi = __floats2half2_rn(o.z, o.w);
        u.x = *reinterpret_cast<uint32_t*>(&lo); u.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(y) + idx) = u;
    }
}

int launch_pool_dw16(const float* x, int ld_x, const float* w, const float* bias, void* y, int ld_y, int out_dtype, int B,
                     int T, int Cpad, cudaStream_t st) {
    size_t total = (size_t)2 * T * (Cpad / 4);
    dim3 grid(cdiv(total, 256), B);
    if (out_dtype == DT_BF16) pool_dw16_kernel<DT_BF16><<<grid, 256, 0, st>>>(x, ld_x, w, bias, y, ld_y, T, Cpad);
    else pool_dw16_kernel<DT_F16><<<grid, 256, 0, st>>>(x, ld_x, w, bias, y, ld_y, T, Cpad);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

}  // namespace st2
