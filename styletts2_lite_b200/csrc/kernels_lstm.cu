// Recurrence of the bidirectional LSTMs of the modules in front of the Decoder: `shared` of ProsodyPredictor.F0Ntrain
// (reference models.py:407, :449), the DurationEncoder's LSTMs and predictor.lstm (models.py:470-480, :402; inference.py:243-244)
// and the TextEncoder's (models.py:255, :268-277).  Arithmetic: torch nn.LSTM, gates (i, f, g, o), zero initial state, batch_first;
// with per-utterance lengths it is nn.utils.rnn.pack_padded_sequence -> LSTM -> pad_packed_sequence.
//
// The input half of the gates (x W_ih^T + b_ih, one [B*T, 640] x [640, 2048] contraction for both directions) is
// a 1x1 convolution and runs on the conv kernels.  What is left is T strictly sequential steps of
//     gates = G[t] + h W_hh^T + b_hh ;  c = sig(f) c + sig(i) tanh(g) ;  h = sig(o) tanh(c)
// with a [4H, H] = 1 MB fp32 matrix per direction: too large for one SM's shared memory, latency bound if re-read
// from L2 every step.  One thread-block CLUSTER of 8 CTAs owns one (direction, group of 4 or 8 utterances): CTA r keeps
// the 4 x 32 gate columns of hidden units [32r, 32r+32) resident in shared memory (128 KB) for the whole sequence,
// computes its slice of the gates, updates its 32 cells and sends the 32 new h values of each utterance to
// the h buffers of all 8 CTAs through distributed shared memory.
#include "common.cuh"

#include <cooperative_groups.h>
#include <stdlib.h>

namespace cg = cooperative_groups;

namespace st2 {

constexpr int kLstmCluster = 8;      // CTAs per cluster
constexpr int kLstmThreads = 256;    // 8 warps: warp = K slice in the gate phase, = utterance in the cell phase

__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }

// G   [B][T][2][4H]   input half of the gates, direction-major inside a row (fwd 4H | rev 4H), gate order i,f,g,o
// whh [2][H][4H]      W_hh^T per direction
// bhh [2][4H]
// y   [B][T][2H]      forward h | reverse h   (channels-last, what the AdainResBlk1d stacks read)
//
// Three things keep a step near 2 us:
//  * the h exchange is `st.async` into the peers' shared memory with transaction-count mbarriers (the arrival of the data IS
//    the signal; no cluster barrier on the critical path, double-buffered h makes the reuse safe: a CTA can only send step
//    t+1 values after it received every CTA's step-t values, i.e. after every CTA finished reading the buffer being overwritten)
//  * K is split over the 8 warps (32 k each) so W_hh is read from shared memory once per step instead of four times, with
//    weights stored as (k even, k odd) pairs and packed fma.rn.f32x2 over the pair; the 8 partial sums meet in shared memory
//  * BT = 4 or 8 utterances per cluster, so small batches spread over more SMs
//
// Ragged batches (`lengths` != nullptr; pack_padded_sequence semantics of models.py:271-277, :503-509, :426-435): utterance b
// runs len_b steps, the reverse direction starts at its own last token (t = len_b - 1 - step), rows t >= len_b of y are zero
// (pad_packed_sequence).  The cluster runs max(len) steps of its utterances; a finished utterance keeps its state and re-sends
// its last h so the transaction count of every step stays the same.
__device__ __forceinline__ uint32_t lstm_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lstm_mapa(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void lstm_st_async(uint32_t remote_addr, float v, uint32_t remote_mbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(remote_addr),
                 "r"(__float_as_uint(v)), "r"(remote_mbar)
                 : "memory");
}
__device__ __forceinline__ void lstm_mbar_wait(uint32_t mbar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LSTM_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LSTM_DONE;\n"
        "bra LSTM_WAIT;\n"
        "LSTM_DONE:\n"
        "}\n" ::"r"(mbar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ float2 lstm_ffma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;"
        : "=l"(reinterpret_cast<unsigned long long&>(d))
        : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)),
          "l"(reinterpret_cast<unsigned long long&>(c)));
    return d;
}

template <int H, int BT>
__global__ void __cluster_dims__(kLstmCluster, 1, 1) __launch_bounds__(kLstmThreads, 1)
lstm_bidir_v2_kernel(const float* __restrict__ G, const float* __restrict__ whh, const float* __restrict__ bhh,
                     float* __restrict__ y, int B, int T, const int32_t* __restrict__ lengths) {
    constexpr int UL = H / kLstmCluster;        // 32 hidden units per CTA, one per lane
    constexpr int KS = kLstmThreads / 32;       // 8 K slices, one per warp
    constexpr int KW = H / KS;                  // 32 k per slice
    static_assert(UL == 32 && KW % 4 == 0, "layout");
    extern __shared__ __align__(16) float smem[];
    float4* WsA = reinterpret_cast<float4*>(smem);                 // [H/2][UL]: (i_k0, i_k1, f_k0, f_k1)
    float4* WsB = WsA + (H / 2) * UL;                              // [H/2][UL]: (g_k0, g_k1, o_k0, o_k1)
    float* hbuf = reinterpret_cast<float*>(WsB + (H / 2) * UL);    // [2][BT][H]
    float* red = hbuf + 2 * BT * H;                                // [KS][4][BT][UL] partial gate sums
    uint64_t* hfull = reinterpret_cast<uint64_t*>(red + KS * 4 * BT * UL);   // [2]

    cg::cluster_group cluster = cg::this_cluster();
    const uint32_t rank = cluster.block_rank();
    const int dir = blockIdx.y;
    const int b0 = blockIdx.z * BT;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    const float* wsrc = whh + (size_t)dir * H * 4 * H;             // [k][4H]
    for (int idx = tid; idx < (H / 2) * UL; idx += kLstmThreads) {
        const int kp = idx / UL, ul = idx % UL;
        const float* w0 = wsrc + (size_t)(2 * kp) * 4 * H + rank * UL + ul;
        const float* w1 = w0 + 4 * H;
        WsA[idx] = make_float4(w0[0], w1[0], w0[H], w1[H]);
        WsB[idx] = make_float4(w0[2 * H], w1[2 * H], w0[3 * H], w1[3 * H]);
    }
    for (int idx = tid; idx < BT * H; idx += kLstmThreads) hbuf[idx] = 0.f;            // h_0 = 0 (buffer 0)
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(lstm_smem_u32(&hfull[0])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(lstm_smem_u32(&hfull[1])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // cell phase: thread (utterance cb = warp, unit = lane) for warps < BT
    const int cb = warp;
    const bool cell = warp < BT;
    float c_state = 0.f, h_last = 0.f;
    int steps = T, len = T;                     // steps of this cluster, length of this cell thread's utterance
    if (lengths != nullptr) {
        steps = 0;
#pragma unroll
        for (int b = 0; b < BT; ++b) {
            if (b0 + b >= B) break;
            const int lb = min(max(__ldg(lengths + b0 + b), 0), T);
            steps = max(steps, lb);
            if (b == cb) len = lb;
        }
        if (!cell || b0 + cb >= B) len = steps;
    }
    float bias[4] = {0.f, 0.f, 0.f, 0.f};
    uint32_t r_h[kLstmCluster], r_bar[kLstmCluster];
#pragma unroll
    for (int r = 0; r < kLstmCluster; ++r) {
        r_h[r] = lstm_mapa(lstm_smem_u32(hbuf), (uint32_t)r);
        r_bar[r] = lstm_mapa(lstm_smem_u32(hfull), (uint32_t)r);
    }
    if (cell) {
#pragma unroll
        for (int g = 0; g < 4; ++g) bias[g] = bhh[dir * 4 * H + g * H + rank * UL + lane];
    }
    cluster.sync();                 // barriers initialised and h_0 zeroed everywhere before the first remote store

    constexpr uint32_t kStepBytes = (uint32_t)BT * H * 4u;          // what one step delivers into one CTA's h buffer
    for (int step = 0; step < steps; ++step) {
        const bool act = step < len;
        const int t = dir ? len - 1 - step : step;
        const int cur = step & 1, nxt = cur ^ 1;
        if (tid == 0)               // arm the buffer this step fills (its previous phase completed before step-1 started)
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(lstm_smem_u32(&hfull[nxt])), "r"(kStepBytes)
                         : "memory");
        float gin[4] = {0.f, 0.f, 0.f, 0.f};
        if (cell && act && b0 + cb < B) {
            const float* gp = G + (((size_t)(b0 + cb) * T + t) * 2 + dir) * 4 * H + rank * UL + lane;
#pragma unroll
            for (int g = 0; g < 4; ++g) gin[g] = __ldg(gp + g * H);
        }
        if (step > 0) lstm_mbar_wait(lstm_smem_u32(&hfull[cur]), (uint32_t)(((step - 1) >> 1) & 1));   // h_{t-1} has landed
        // gate phase: this warp's K slice of h W_hh^T for all BT utterances, (k even, k odd) pairs on the packed FMA
        float2 acc[4][BT];
#pragma unroll
        for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int b = 0; b < BT; ++b) acc[g][b] = make_float2(0.f, 0.f);
        const float* hc = hbuf + (size_t)cur * BT * H + warp * KW;
        const float4* wa = WsA + (warp * KW / 2) * UL + lane;
        const float4* wb = WsB + (warp * KW / 2) * UL + lane;
#pragma unroll 2
        for (int k4 = 0; k4 < KW / 4; ++k4) {
            const float4 a0 = wa[(2 * k4) * UL], a1 = wa[(2 * k4 + 1) * UL];
            const float4 c0 = wb[(2 * k4) * UL], c1 = wb[(2 * k4 + 1) * UL];
#pragma unroll
            for (int b = 0; b < BT; ++b) {
                const float4 hv = *reinterpret_cast<const float4*>(hc + b * H + 4 * k4);      // warp-uniform broadcast
                const float2 h01 = make_float2(hv.x, hv.y), h23 = make_float2(hv.z, hv.w);
                acc[0][b] = lstm_ffma2(make_float2(a0.x, a0.y), h01, acc[0][b]);
                acc[1][b] = lstm_ffma2(make_float2(a0.z, a0.w), h01, acc[1][b]);
                acc[2][b] = lstm_ffma2(make_float2(c0.x, c0.y), h01, acc[2][b]);
                acc[3][b] = lstm_ffma2(make_float2(c0.z, c0.w), h01, acc[3][b]);
                acc[0][b] = lstm_ffma2(make_float2(a1.x, a1.y), h23, acc[0][b]);
                acc[1][b] = lstm_ffma2(make_float2(a1.z, a1.w), h23, acc[1][b]);
                acc[2][b] = lstm_ffma2(make_float2(c1.x, c1.y), h23, acc[2][b]);
                acc[3][b] = lstm_ffma2(make_float2(c1.z, c1.w), h23, acc[3][b]);
            }
        }
#pragma unroll
        for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int b = 0; b < BT; ++b) red[((warp * 4 + g) * BT + b) * UL + lane] = acc[g][b].x + acc[g][b].y;
        __syncthreads();
        if (cell) {
            float gate[4];
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float sacc = 0.f;
#pragma unroll
                for (int ks = 0; ks < KS; ++ks) sacc += red[((ks * 4 + g) * BT + cb) * UL + lane];
                gate[g] = gin[g] + (sacc + bias[g]);
            }
            if (act) {
                c_state = sigmoid_f(gate[1]) * c_state + sigmoid_f(gate[0]) * tanhf(gate[2]);
                h_last = sigmoid_f(gate[3]) * tanhf(c_state);
            }
            const float h = h_last;
            const uint32_t hoff = (uint32_t)((nxt * BT + cb) * H + rank * UL + lane) * 4u;
            const uint32_t boff = (uint32_t)nxt * 8u;
#pragma unroll
            for (int r = 0; r < kLstmCluster; ++r) lstm_st_async(r_h[r] + hoff, h, r_bar[r] + boff);
            if (act && b0 + cb < B) y[((size_t)(b0 + cb) * T + t) * 2 * H + dir * H + rank * UL + lane] = h;
        }
        __syncthreads();            // the partial-sum buffer is rewritten by the next step's gate phase
    }
    if (lengths != nullptr && cell && b0 + cb < B)          // pad_packed_sequence: zeros behind the utterance
        for (int t = len; t < T; ++t) y[((size_t)(b0 + cb) * T + t) * 2 * H + dir * H + rank * UL + lane] = 0.f;
    cluster.sync();                 // no CTA leaves while a peer may still be storing into its shared memory
}

template <int BT>
static int launch_lstm_v2(const float* G, const float* whh, const float* bhh, float* y, int B, int T, const int32_t* lengths,
                          cudaStream_t st) {
    constexpr int HH = 256;
    const size_t smem = ((size_t)HH * 4 * (HH / kLstmCluster) + 2 * BT * HH + (kLstmThreads / 32) * 4 * BT * (HH / kLstmCluster)) * sizeof(float) + 16;
    ST2_CUDA_CHECK(cudaFuncSetAttribute(lstm_bidir_v2_kernel<HH, BT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(kLstmCluster, 2, cdiv(B, BT));
    lstm_bidir_v2_kernel<HH, BT><<<grid, kLstmThreads, smem, st>>>(G, whh, bhh, y, B, T, lengths);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

int launch_lstm_bidir(const float* G, const float* whh, const float* bhh, float* y, int B, int T, int H, cudaStream_t st,
                      const int32_t* lengths) {
    ST2_REQUIRE(H == 256, "lstm: hidden size %d is not supported (d_hid must be 512)", H);
    ST2_REQUIRE(B > 0 && T > 0, "lstm: bad shape B=%d T=%d", B, T);
    // 4 utterances per cluster while all clusters are still co-resident (an 8-CTA cluster must sit inside one GPC, so
    // fewer fit than 148 / 8: the occupancy API says 15 on the B200; measured over 4 x 64 steps: B <= 24, 12 clusters of
    // BT = 4: 0.47 ms against 0.67 ms with BT = 8; B = 32, 16 clusters of BT = 4: two waves, 0.90 ms)
    static int max_clusters4[kMaxDevices] = {};          // per device: 0 = not asked yet
    int& mc4 = max_clusters4[current_device_slot()];
    if (mc4 == 0) {
        constexpr int HH4 = 256;
        const size_t smem4 = ((size_t)HH4 * 4 * (HH4 / kLstmCluster) + 2 * 4 * HH4 + (kLstmThreads / 32) * 4 * 4 * (HH4 / kLstmCluster)) * sizeof(float) + 16;
        cudaFuncSetAttribute(lstm_bidir_v2_kernel<HH4, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(kLstmCluster, 2, 64);
        cfg.blockDim = dim3(kLstmThreads);
        cfg.dynamicSmemBytes = smem4;
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeClusterDimension;
        attr.val.clusterDim.x = kLstmCluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
        cfg.attrs = &attr; cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, lstm_bidir_v2_kernel<HH4, 4>, &cfg) != cudaSuccess || n <= 0) { n = 8; cudaGetLastError(); }
        mc4 = n;
        if (tune().verbose) fprintf(stderr, "lstm: %d co-resident clusters of 8 CTAs (BT=4 configuration)\n", n);
    }
    const bool bt4 = cdiv(B, 4) * 2 <= mc4;
    return bt4 ? launch_lstm_v2<4>(G, whh, bhh, y, B, T, lengths, st) : launch_lstm_v2<8>(G, whh, bhh, y, B, T, lengths, st);
}

}  // namespace st2

// ------------------------------------------------------------------------------------------------------------------
// Duration half of the predictor (SURVEY.md 8(f) N2; reference models.py:372-392, :485-520, inference.py:242-245)
// ------------------------------------------------------------------------------------------------------------------
namespace st2 {

// x[b][l][C .. C+S) = s[b][0 .. S): the style columns DurationEncoder concatenates to every token (models.py:489-490, :499)
__global__ void concat_style_kernel(float* __restrict__ x, int ld, int C, const float* __restrict__ s, int S, int64_t rows, int L) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * S) return;
    const int64_t row = i / S;
    const int c = (int)(i - row * S);
    x[row * ld + C + c] = s[(row / L) * S + c];
}

// AdaLayerNorm (models.py:372-392) on channels-last x [B][L][C]: LayerNorm over C (biased variance, eps 1e-5), then
// (1 + gamma) * xhat + beta with gamma | beta = h[b][h_off .. h_off + 2C); writes y[row][0..C) with pitch ld_y.
// One warp per token; C = 512 -> 16 values per lane kept in registers, mean and variance by warp shuffles (two pass).
// PLAIN: the TextEncoder's LayerNorm (models.py:224-236) + LeakyReLU(slope): y = lrelu(gamma[c] * xhat + beta[c]) with
// h = gamma, h + ld_h = beta (per channel, shared by every row)
template <int C, bool PLAIN>
__global__ void ada_layer_norm_kernel(const float* __restrict__ x, const float* __restrict__ h, int ld_h, int h_off,
                                      float* __restrict__ y, int ld_y, int64_t rows, int L, float slope, float eps) {
    constexpr int PER = C / 32;
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const float* xr = x + row * C;
    float v[PER];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < PER / 4; ++i) {
        const float4 t = *reinterpret_cast<const float4*>(xr + (i * 32 + lane) * 4);
        v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
        sum += (t.x + t.y) + (t.z + t.w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum * (1.f / C);
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) { const float dlt = v[i] - mean; sq = fmaf(dlt, dlt, sq); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    const float rstd = rsqrtf(sq * (1.f / C) + eps);
    const float* hb = PLAIN ? h : h + (row / L) * ld_h + h_off;
    const float* bb = PLAIN ? h + ld_h : hb + C;
    const float one = PLAIN ? 0.f : 1.f;
    float* yr = y + row * ld_y;
#pragma unroll
    for (int i = 0; i < PER / 4; ++i) {
        const int c = (i * 32 + lane) * 4;
        const float4 g = *reinterpret_cast<const float4*>(hb + c), b = *reinterpret_cast<const float4*>(bb + c);
        float4 o;
        o.x = fmaf(one + g.x, (v[4 * i] - mean) * rstd, b.x);
        o.y = fmaf(one + g.y, (v[4 * i + 1] - mean) * rstd, b.y);
        o.z = fmaf(one + g.z, (v[4 * i + 2] - mean) * rstd, b.z);
        o.w = fmaf(one + g.w, (v[4 * i + 3] - mean) * rstd, b.w);
        if (PLAIN) {
            o.x = o.x > 0.f ? o.x : o.x * slope; o.y = o.y > 0.f ? o.y : o.y * slope;
            o.z = o.z > 0.f ? o.z : o.z * slope; o.w = o.w > 0.f ? o.w : o.w * slope;
        }
        *reinterpret_cast<float4*>(yr + c) = o;
    }
}

// x[b][l][0 .. ncols) = 0 for l >= lengths[b]: the masked_fill_(m, 0.0) calls of TextEncoder.forward (models.py:262, :266) and
// DurationEncoder.forward (models.py:491, :500) on channels-last rows of pitch ld.  One warp per row; rows inside the utterance
// are left alone.
__global__ void mask_rows_kernel(float* __restrict__ x, int ld, int ncols, const int32_t* __restrict__ lengths, int64_t rows, int L) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int b = (int)(row / L), l = (int)(row - (int64_t)b * L);
    if (l < __ldg(lengths + b)) return;
    float* xr = x + row * ld;
    for (int c = lane; c < ncols; c += 32) xr[c] = 0.f;
}

// nn.Embedding lookup into channels-last rows: y[row][0..C) = table[tok[row]][0..C)   (models.py:259)
__global__ void embedding_kernel(const int64_t* __restrict__ tok, const float* __restrict__ table, float* __restrict__ y, int C,
                                 int64_t rows, int n_symbols) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int c4 = C / 4;
    if (i >= rows * c4) return;
    const int64_t row = i / c4;
    const int c = (int)(i - row * c4) * 4;
    int64_t t = tok[row];
    t = t < 0 ? 0 : (t >= n_symbols ? n_symbols - 1 : t);          // the host wrapper rejects out-of-range ids; never read outside
    *reinterpret_cast<float4*>(y + row * C + c) = __ldg(reinterpret_cast<const float4*>(table + t * C + c));
}

// channels-last [B][L][C] -> the reference's [B][C][L] (32 x 32 tiles through shared memory)
__global__ void cl_to_cf_kernel(const float* __restrict__ x, float* __restrict__ y, int L, int C) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, l0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int l = l0 + i, c = c0 + threadIdx.x;
        if (l < L && c < C) tile[i][threadIdx.x] = x[((size_t)b * L + l) * C + c];
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int c = c0 + i, l = l0 + threadIdx.x;
        if (l < L && c < C) y[((size_t)b * C + c) * L + l] = tile[threadIdx.x][i];
    }
}

// duration[row] = sum_j sigmoid(x[row] . W[j] + bias[j])   (duration_proj + torch.sigmoid(...).sum(-1), inference.py:244-245)
// One warp per token: x row in registers, one warp-reduced dot product per output bin.
template <int C>
__global__ void duration_head_kernel(const float* __restrict__ x, const float* __restrict__ W, const float* __restrict__ bias,
                                     float* __restrict__ duration, int64_t rows, int nbins) {
    constexpr int PER = C / 32;
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    float v[PER];
#pragma unroll
    for (int i = 0; i < PER / 4; ++i) {
        const float4 t = *reinterpret_cast<const float4*>(x + row * C + (i * 32 + lane) * 4);
        v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
    }
    float total = 0.f;
    for (int j = 0; j < nbins; ++j) {
        const float* wj = W + (size_t)j * C;
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < PER / 4; ++i) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(wj + (i * 32 + lane) * 4));
            acc = fmaf(v[4 * i], w.x, acc); acc = fmaf(v[4 * i + 1], w.y, acc);
            acc = fmaf(v[4 * i + 2], w.z, acc); acc = fmaf(v[4 * i + 3], w.w, acc);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        total += sigmoid_f(acc + __ldg(bias + j));
    }
    if (lane == 0) duration[row] = total;
}

int launch_mask_rows(float* x, int ld, int ncols, const int32_t* lengths, int B, int L, cudaStream_t st) {
    const int64_t rows = (int64_t)B * L;
    mask_rows_kernel<<<(unsigned)cdiv(rows, 8), 256, 0, st>>>(x, ld, ncols, lengths, rows, L);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

int launch_concat_style(float* x, int ld, int C, const float* s, int S, int B, int L, cudaStream_t st) {
    const int64_t n = (int64_t)B * L * S;
    concat_style_kernel<<<cdiv(n, 256), 256, 0, st>>>(x, ld, C, s, S, (int64_t)B * L, L);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

int launch_ada_layer_norm(const float* x, const float* h, int ld_h, int h_off, float* y, int ld_y, int B, int L, int C,
                          cudaStream_t st) {
    ST2_REQUIRE(C == 512 && ld_y % 4 == 0 && ld_h % 4 == 0 && h_off % 4 == 0, "ada_layer_norm: needs 512 channels (got %d)", C);
    const int64_t rows = (int64_t)B * L;
    ada_layer_norm_kernel<512, false><<<cdiv(rows, 8), 256, 0, st>>>(x, h, ld_h, h_off, y, ld_y, rows, L, 0.f, 1e-5f);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

int launch_layer_norm_lrelu(const float* x, const float* gamma, const float* beta, float slope, float* y, int B, int L, int C,
                            cudaStream_t st, float eps) {
    ST2_REQUIRE(C == 512, "layer_norm: needs 512 channels (got %d)", C);
    const int64_t rows = (int64_t)B * L;
    ada_layer_norm_kernel<512, true><<<cdiv(rows, 8), 256, 0, st>>>(x, gamma, (int)(beta - gamma), 0, y, C, rows, L, slope, eps);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

int launch_embedding(const int64_t* tok, const float* table, float* y, int B, int L, int C, int n_symbols, cudaStream_t st) {
    ST2_REQUIRE(C % 4 == 0, "embedding: channels must be a multiple of 4");
    const int64_t n = (int64_t)B * L * (C / 4);
    embedding_kernel<<<cdiv(n, 256), 256, 0, st>>>(tok, table, y, C, (int64_t)B * L, n_symbols);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

int launch_cl_to_cf(const float* x, float* y, int B, int L, int C, cudaStream_t st) {
    dim3 grid(cdiv(L, 32), cdiv(C, 32), B), block(32, 8);
    cl_to_cf_kernel<<<grid, block, 0, st>>>(x, y, L, C);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

int launch_duration_head(const float* x, const float* W, const float* bias, float* duration, int B, int L, int C, int nbins,
                         cudaStream_t st) {
    ST2_REQUIRE(C == 512 && nbins > 0, "duration_head: needs 512 channels (got %d)", C);
    const int64_t rows = (int64_t)B * L;
    duration_head_kernel<512><<<cdiv(rows, 8), 256, 0, st>>>(x, W, bias, duration, rows, nbins);
    ST2_LAUNCH_CHECK();
    return ST2_OK;
}

}  // namespace st2
