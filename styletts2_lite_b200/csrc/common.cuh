// Shared declarations for the st2_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/st2_b200.h"

namespace st2 {

void set_error(const char* fmt, ...);
extern thread_local int64_t g_launch_count;

#define ST2_CUDA_CHECK(expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            ::st2::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                             __FILE__, __LINE__);                                         \
            return ST2_ERR_CUDA;                                                          \
        }                                                                                 \
    } while (0)

#define ST2_LAUNCH_CHECK()                                                                \
    do {                                                                                  \
        ::st2::g_launch_count++;                                                          \
        cudaError_t _e = cudaGetLastError();                                              \
        if (_e != cudaSuccess) {                                                          \
            ::st2::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e),  \
                             __FILE__, __LINE__);                                         \
            return ST2_ERR_CUDA;                                                          \
        }                                                                                 \
    } while (0)

#define ST2_REQUIRE(cond, ...)                                                            \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            ::st2::set_error(__VA_ARGS__);                                                \
            return ST2_ERR_INVALID;                                                       \
        }                                                                                 \
    } while (0)

static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// Process-wide test hooks: they let the tests reach or pin a kernel path at fixture sizes.  All default to 0 (the planners'
// choice) and are changed only through st2_set_tuning().  Not synchronised: set them while no forward is running.
struct Tune {
    int no_pipe = 0;                        // conv_pipe: decline every shape, so conv_fused runs the ones it would take
    int row_always = 0;                     // conv_row: take every geometry it can launch, small problems too (tests of its scheduling)
    int row_sub = 0;                        // conv_row: only this tile split (0 = planner's choice)
    int no_row_inline_coef = 0;             // conv_row: always launch the coefficient kernel (reference for the in-kernel coefficients)
    int verbose = 0;                        // print the conv_pipe / conv_row / lstm plans to stderr
};
const Tune& tune();
int tune_set(const char* name, int value);    // ST2_OK, or ST2_ERR_INVALID for an unknown name

// per-device cache of one-time function attributes / properties: a process may drive several GPUs, and
// cudaFuncAttributeMaxDynamicSharedMemorySize applies to the device that was current when it was set
static constexpr int kMaxDevices = 64;
static inline int current_device_slot() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
    return dev;
}
int device_num_sms();                          // SM count of the current device (cached per device)

enum Act { ACT_NONE = 0, ACT_LRELU = 1, ACT_SNAKE = 2, ACT_GELU = 3 };
enum OutDtype { DT_F32 = 0, DT_BF16 = 1, DT_F16 = 2 };
// kernel categories of the per-launch event profile (st2_decoder_get_profile)
enum ProfCat {
    PC_CONV_TC = 0,     // tcgen05 implicit-GEMM conv               (bound: tensor)
    PC_CONV_SIMT = 1,   // fp32 FFMA conv                            (bound: fp32 pipe / hbm)
    PC_NORM_STATS = 2,  // InstanceNorm statistics                   (bound: hbm, read only)
    PC_NORM_COEF = 3,   // per-(b,c) affine coefficients             (tiny)
    PC_AFFINE_ACT = 4,  // AdaIN affine + Snake / LeakyReLU          (bound: hbm)
    PC_SOURCE = 5,      // SineGen + harmonic source (+ STFT front)  (bound: hbm)
    PC_POST = 6,        // Snake + conv_post + tanh / iSTFT head     (bound: hbm)
    PC_MISC = 7,        // layout, style fc, pool, taps
    PC_CONV_FUSED = 8,  // conv_fused_kernel: fused AdaIN/act -> tcgen05 conv -> residual/stats, register-staged (256-ch: tensor)
    PC_CONV_PIPE = 9,   // conv_pipe_kernel: the same fusion fully TMA-fed (C <= 128, ups; bound: hbm / shared memory)
    PC_LSTM = 10,       // lstm_bidir_kernel: recurrence of the predictor's shared BiLSTM (bound: latency, T sequential steps)
    PC_CONV_ROW = 11,   // conv_row_kernel: the 32/64-channel resblock convs, row-per-thread epilogue (bound: hbm / shared memory)
    PC_COUNT = 12
};

// ---- HBM-bound kernels (kernels_norm.cu) ---------------------------------------------
// InstanceNorm statistics of channels-last x[B][T][ld] over T: partial (sum, sumsq) in
// double per time slab, then mean / rstd folded with the AdaIN affine into y = a*x + b.
int64_t adain_scratch_bytes(int B, int T, int C);
int launch_in_stats(const float* x, int ld, int B, int T, int C, void* scratch, cudaStream_t st);
// coef[b][0][c] = a, coef[b][1][c] = b  (c < Cpad; zero beyond C).  h: [B][ld_h] with
// gamma at h_off + c and beta at h_off + C + c; h == nullptr -> a = 1, b = 0 (no norm).
int launch_adain_coef(const void* scratch, const float* h, int ld_h, int h_off, float* coef, int B,
                      int T, int C, int Cpad, cudaStream_t st);
// y = act(a*x+b); snake uses alpha[c].  y pitch ld_y, dtype out_dtype; processes Cpad channels.
int launch_affine_act(const float* x, int ld_x, const float* coef, const float* alpha, int act,
                      float slope, void* y, int ld_y, int out_dtype, int B, int T, int Cpad,
                      cudaStream_t st);

// misc elementwise (kernels_misc.cu)
int launch_cf_to_cl(const float* src, float* dst, int ld_dst, int B, int C, int T, cudaStream_t st);
int launch_f0n_conv(const float* f0, const float* n, const float* wf, const float* bf, const float* wn,
                    const float* bn, float* dst0, int ld0, int c0, int pad0_from, float* dst1, int ld1,
                    int c1, int pad1_from, int B, int T, cudaStream_t st);
int launch_style_fc(const float* s, const float* W, const float* bias, float* h, int B, int R, int K,
                    cudaStream_t st);
int launch_pool_dw(const float* x, int ld_x, const float* w, const float* bias, float* y, int ld_y, int B,
                   int T, int C, int Cpad, cudaStream_t st);
int launch_pool_dw16(const float* x, int ld_x, const float* w, const float* bias, void* y, int ld_y, int out_dtype, int B,
                     int T, int Cpad, cudaStream_t st);
int noise_conv_parts(int Tout, int stride);
// stats: float2 (sum, sumsq) tile partials of y - bias (the coefficient kernel's stat_shift); y16: y stored as fp16 without the bias
int launch_noise_conv(const float* har, const float* w, const float* bias, float* y, void* stats, int B, int S, int Tout,
                      int C, int k, int stride, int pad, cudaStream_t st, int y16 = 0);
int launch_post_hifigan(const float* x, int ld_x, const float* alpha, const float* w, const float* bias,
                        float* out, int B, int S, int C, int fast, cudaStream_t st, int x16 = 0);
int launch_copy_dense(const float* src, int ld, float* dst, int64_t rows, int C, cudaStream_t st);
int launch_half_to_float(const void* src, float* dst, int64_t n, cudaStream_t st);
int launch_fold_pack(const float* g, const float* v, float* wp, int d0, int d1, int k, int transposed,
                     cudaStream_t st);
int launch_cast16(const float* src, void* dst, int64_t n, int out_dtype, cudaStream_t st);
int launch_pack_w16(const float* wp, void* w16, int k, int Cin, int Cout, int CinPad, int CoutPad, int out_dtype,
                    cudaStream_t st);

// source / stft (kernels_source.cu; compiled without fast-math)
int launch_sinegen_frames(const float* f0, float* frames, int B, int L2, int scale, cudaStream_t st);
int launch_sinegen_phase(const float* frames, float* phase, int B, int L2, int scale, cudaStream_t st);
int launch_har_source(const float* f0, const float* frames, const float* noise, uint64_t seed, const uint64_t* seed_dev,
                      const float* lin_w, const float* lin_b, float* har, int B, int L2, int scale,
                      cudaStream_t st);
int launch_stft_transform(const float* har, const float* wr, const float* wi, float* out, int ld_out, int B,
                          int S, int n_fft, int hop, cudaStream_t st);
int launch_istft_head(const float* x, int ld_x, const float* wr, const float* wi, float* out, int B,
                      int frames, int S, int n_fft, int hop, cudaStream_t st);

// BiLSTM recurrence (kernels_lstm.cu): G [B][T][2][4H] input half of the gates, whh [2][H][4H], bhh [2][4H] -> y [B][T][2H]
// lengths: per-utterance token counts on the device (pack_padded_sequence semantics), nullptr = every utterance has T steps
int launch_lstm_bidir(const float* G, const float* whh, const float* bhh, float* y, int B, int T, int H, cudaStream_t st,
                      const int32_t* lengths = nullptr);
int launch_mask_rows(float* x, int ld, int ncols, const int32_t* lengths, int B, int L, cudaStream_t st);

// duration half of the predictor (kernels_lstm.cu)
int launch_concat_style(float* x, int ld, int C, const float* s, int S, int B, int L, cudaStream_t st);
int launch_ada_layer_norm(const float* x, const float* h, int ld_h, int h_off, float* y, int ld_y, int B, int L, int C,
                          cudaStream_t st);
int launch_layer_norm_lrelu(const float* x, const float* gamma, const float* beta, float slope, float* y, int B, int L, int C,
                            cudaStream_t st, float eps = 1e-5f);
// Vocos generator pieces (vocos.cu; reference Modules/vocos.py)
int launch_dwconv7(const float* x, const float* w7, const float* bias, float* y, int B, int T, int C, cudaStream_t st);
int launch_scale_cols(float* w, float* bias, int rows, int ld, int cols, const float* scale, cudaStream_t st);
int launch_vocos_basis(const float* window, float* basis, int n_fft, int k_pad, cudaStream_t st);
int launch_vocos_spec(const float* o, int ld_o, void* a, int ld_a, int out_dtype, int64_t rows, int bins, cudaStream_t st);
int launch_vocos_ola(const float* frames, const float* window, float* out, int B, int T, int n_fft, int hop, cudaStream_t st);
int launch_embedding(const int64_t* tok, const float* table, float* y, int B, int L, int C, int n_symbols, cudaStream_t st);
int launch_cl_to_cf(const float* x, float* y, int B, int L, int C, cudaStream_t st);
int launch_duration_head(const float* x, const float* W, const float* bias, float* duration, int B, int L, int C, int nbins,
                         cudaStream_t st);

// length regulator (length_regulator.cu)
int launch_round_durations(const float* duration, const int32_t* n_tokens, int32_t* dur, int32_t* total,
                           int B, int L, cudaStream_t st);
int launch_smooth_durations(const float* duration, const int32_t* n_tokens, const float* z, const float* prev_mean, float t,
                            float speed, float* out, float* mean_out, int B, int L, cudaStream_t st, int chain = 0);
int launch_length_regulate(const float* src, const int32_t* dur, float* out, int B, int C, int L, int F,
                           int channels_last, cudaStream_t st);

// ---- convolutions ----------------------------------------------------------------------
// One description for Conv1d and (polyphase) ConvTranspose1d on channels-last tensors:
//   for output index m in [0,M) and phase p in [0,phases):
//     t_out = m*out_stride + p - out_pad        (store if 0 <= t_out < Tout)
//     acc[co] = sum_j sum_ci x[b][m*in_stride + j*tap_step + in_off][ci] * W[widx(p,j)][ci][co]
//     widx(p,j) = p + j*w_step            (Conv1d: phases=1, w_step=1; ConvT: w_step=stride)
//   y = (acc + bias + res[b][t_out >> res_shift][co] (+ y_old if accumulate)) * scale
//   mirror: the row written at t_out == 2 is also written at row 0 (ReflectionPad1d((1,0)))
struct ConvArgs {
    const float* x;  int ld_x;  int Tin;
    const void* x16; int ld_x16;            // 16-bit operand copy (tensor-core path)
    const float* w;                          // packed fp32 [k][Cin][Cout]
    const void* w16;                         // packed 16-bit [k][CoutPad][CinPad] (tensor-core path)
    int w16_cin_pad, w16_cout_pad;
    const float* bias;
    const float* res; int ld_res; int res_shift;
    float* y; int ld_y; int Tout;
    int B, Cin, Cout, M;
    int ntaps, tap_step, in_off, in_stride;
    int phases, w_step, out_stride, out_pad;
    float scale; int accumulate; int mirror;
    int fmt16;                               // DT_BF16 / DT_F16 for the tensor-core path
    int x16in;                               // fused path: the input tensor x is 16-bit (fmt16) with pitch ld_x elements
    int y16out;                              // fused path: write y as fp16; statistics still from the fp32 values
    int epi_gelu;                            // conv_tc only: y = GELU(conv + bias) stored in the 16-bit format fmt16 with pitch ld_y
                                             // elements (the operand of the next pointwise conv); no residual / accumulate / scale
    int res16;                               // fused path (conv_pipe only): the residual tensor is fp16 with pitch ld_res elements
    const void* acc_src; int acc16;          // fused path (conv_pipe only): with accumulate, read the old values from acc_src (pitch
                                             // ld_y; fp16 when acc16) instead of y -- partial sums of a stage kept in fp16
};
int launch_conv_simt(const ConvArgs& a, cudaStream_t st);
int launch_conv_tc(const ConvArgs& a, cudaStream_t st);   // tcgen05 + TMA
bool conv_tc_supported(const ConvArgs& a);
// fused [affine + act] -> tcgen05 conv -> [bias/res/scale/acc + per-tile (sum,sumsq)] (conv_fused.cu); x fp32
bool conv_fused_supported(const ConvArgs& a);
int fused_stats_parts(const ConvArgs& a);
int launch_conv_fused(const ConvArgs& a, const float* coef, int coef_ld, int act, float slope, const float* alpha,
                      void* stats_out, cudaStream_t st);
// stride-1 convs: fully TMA-fed pipeline (conv_pipe.cu); launch_conv_fused dispatches to it when supported
bool conv_pipe_supported(const ConvArgs& a);
int launch_conv_pipe(const ConvArgs& a, const float* coef, int coef_ld, int act, float slope, const float* alpha,
                     void* stats_out, cudaStream_t st);
int launch_add_vec(float* dst, const float* a, const float* b, int n, cudaStream_t st);
// x_offset (optional, [C]): the tensor the coefficients will be applied to is stored as x - x_offset[c];
// stat_shift (optional, [C]): the partials are of x - stat_shift[c] (noise_conv: of the conv without its bias)
int launch_adain_coef_f2(const void* partial, int nparts, const float* h, int ld_h, int h_off, float* coef, int B, int T,
                         int C, int Cpad, cudaStream_t st, const float* x_offset = nullptr, const float* stat_shift = nullptr);
// 32 / 64-channel stride-1 Snake convs on fp16 stage-private tensors: row-per-thread epilogue, residual through the tensor
// core, statistics per (CTA, utterance, epilogue warp) (conv_row.cu).  `desc` describes where the partials of an utterance
// live; launch_adain_coef_row turns them into AdaIN coefficients.
struct RowStatsDesc { int grid, J, nwarp, mmt, tq, tr, C; };
// where a conv_row launch finds what it needs to compute the AdaIN coefficients of its input itself: the partials of the
// conv_row launch that produced the input, the style rows (gamma | beta at h_off) and the row count the statistics are over
struct RowCoefSrc { const void* partial; RowStatsDesc desc; const float* h; int ld_h; int h_off; int T; };
bool conv_row_inline_coef_ok(const ConvArgs& a);
bool conv_row_supported(const ConvArgs& a);                 // geometry, shared-memory plan and enough tiles to fill the grid
bool conv_row_can_launch(const ConvArgs& a);                // geometry and plan only (unit tests force small problems through it)
int64_t conv_row_stats_bytes(int B, int T, int C);
int launch_conv_row(const ConvArgs& a, const float* coef, int coef_ld, int act, const float* alpha, void* stats_out,
                    RowStatsDesc* desc, cudaStream_t st, const RowCoefSrc* src = nullptr);
int launch_adain_coef_row(const void* partial, const RowStatsDesc& d, const float* h, int ld_h, int h_off, float* coef, int B,
                          int T, int C, int Cpad, cudaStream_t st);

}  // namespace st2
